"""CPU tests of the transcript state that crosses the C ABI (bpp_transcript_*: host only, no device) and of the
argument checks of the stand-alone inner-product batch that run before any device work."""
import random
import struct

import pytest

from oracle import merlin

STATE_BYTES = 208


def _export(t: merlin.Transcript) -> bytes:
    """the oracle's Strobe128 in the library's layout: 25 little-endian lanes, pos | pos_begin << 8 | cur_flags << 16"""
    s = t.strobe
    return bytes(s.state) + struct.pack("<Q", s.pos | s.pos_begin << 8 | s.cur_flags << 16)


def _import(state: bytes) -> merlin.Transcript:
    assert len(state) == STATE_BYTES
    s = object.__new__(merlin.Strobe128)
    s.state = bytearray(state[:200])
    w = struct.unpack("<Q", state[200:])[0]
    s.pos, s.pos_begin, s.cur_flags = w & 0xFF, (w >> 8) & 0xFF, (w >> 16) & 0xFF
    t = object.__new__(merlin.Transcript)
    t.strobe = s
    return t


def _lib():
    import bpperm_b200
    return bpperm_b200.load()


def test_merlin_kat_through_the_c_abi():
    from bpperm_b200.ipa import Transcript
    t = Transcript(b"test protocol")
    t.append_message(b"some label", b"some data")
    assert t.challenge_bytes(b"challenge", 32).hex() == "d5a21972d0d5fe320c0d263fac7fffb8145aa640af6e9bca177c03c7efcf0615"


def test_new_state_equals_the_oracle_export():
    from bpperm_b200.ipa import Transcript
    for label in (b"", b"test", b"x" * 300, bytes(range(256))):
        assert Transcript(label).state == _export(merlin.Transcript(label))


@pytest.mark.parametrize("seed", range(6))
def test_random_scripts_match_the_oracle_and_round_trip(seed):
    """appends and challenges of random lengths (across the 166-byte rate, labels with NUL bytes), the state compared
    after every step, and continued from states carried back and forth between the library and the oracle"""
    from bpperm_b200.ipa import Transcript
    rs = random.Random(seed)
    label = rs.randbytes(rs.randrange(0, 40))
    ours, ref = Transcript(label), merlin.Transcript(label)
    for step in range(40):
        lab = rs.randbytes(rs.randrange(0, 20))
        if rs.random() < 0.5:
            msg = rs.randbytes(rs.choice([0, 1, 31, 32, 64, 165, 166, 167, 400, rs.randrange(0, 1000)]))
            ours.append_message(lab, msg)
            ref.append_message(lab, msg)
        else:
            n = rs.choice([0, 1, 32, 64, 166, 200, rs.randrange(0, 500)])
            assert ours.challenge_bytes(lab, n) == ref.challenge_bytes(lab, n), step
        assert ours.state == _export(ref), step
        if step % 7 == 3:   # hand the transcript to the other side and back
            ref = _import(ours.state)
            ours = Transcript(state=_export(ref))
    assert ours.state == _export(ref)


def test_impossible_states_and_null_arguments_are_refused():
    import ctypes
    lib = _lib()
    st = ctypes.create_string_buffer(STATE_BYTES)
    assert lib.bpp_transcript_new(b"t", 1, st) == 0
    good = st.raw
    assert lib.bpp_transcript_new(None, 1, st) == -3
    assert lib.bpp_transcript_new(b"t", 1, None) == -3
    assert lib.bpp_transcript_append_message(None, b"l", 1, b"m", 1) == -3
    assert lib.bpp_transcript_append_message(st, b"l", 1, None, 1) == -3
    assert lib.bpp_transcript_challenge_bytes(st, b"l", 1, None, 4) == -3
    for bad_word in (166, 167 << 8, 1 << 24):   # pos beyond the rate, pos_begin beyond it, stray high bits
        ctypes.memmove(st, good[:200] + struct.pack("<Q", bad_word), STATE_BYTES)
        out = ctypes.create_string_buffer(8)
        assert lib.bpp_transcript_challenge_bytes(st, b"l", 1, out, 8) == -3
        assert lib.bpp_transcript_append_message(st, b"l", 1, b"m", 1) == -3
    # empty label and empty message are fine (NULL with length 0)
    ctypes.memmove(st, good, STATE_BYTES)
    assert lib.bpp_transcript_append_message(st, None, 0, None, 0) == 0


def test_ipa_entry_points_validate_without_a_device():
    import ctypes
    lib = _lib()
    assert lib.bpp_ipa_proof_len(1) == 64
    assert lib.bpp_ipa_proof_len(8) == 32 * 8
    assert lib.bpp_ipa_proof_len(8192) == 32 * 28
    assert lib.bpp_ipa_proof_len(0) == 0 and lib.bpp_ipa_proof_len(6) == 0
    out = ctypes.c_void_p()
    assert lib.bpp_ipa_batch_create(None, None, 0, 0, 0, 8, 1, ctypes.byref(out)) == -3
    assert lib.bpp_ipa_batch_prove(None, None, None, None, b"a", b"b", ctypes.create_string_buffer(208),
                                   ctypes.create_string_buffer(64)) == -3
    assert lib.bpp_ipa_batch_verify(None, None, None, None, b"P", b"p", ctypes.create_string_buffer(208),
                                    ctypes.create_string_buffer(1)) == -3
    lib.bpp_ipa_batch_free(None)
