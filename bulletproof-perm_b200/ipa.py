"""The stand-alone inner-product argument (bulletproofs 4.0.0 inner_product_proof.rs), batched, and the transcript
state it runs on (include/bpperm.h: bpp_transcript_*, bpp_ipa_batch_*).

A `Transcript` is merlin's Transcript held as its 208-byte state; it needs no device.  `InnerProductBatch` proves and
verifies `count` proofs of length n at once over one uploaded point set: G = gens[g_off:g_off+n], H = gens[h_off:h_off+n],
Q_p = q_p * gens[q_off].
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

from ._lib import BppError, load
from .backend import Backend, Points

TRANSCRIPT_BYTES = 208


def _status(lib, rc: int):
    if rc != 0:
        raise BppError(rc, lib.bpp_strerror(rc).decode())


class Transcript:
    """merlin::Transcript as a caller-held state (26 little-endian u64: the Keccak lanes, then pos | pos_begin << 8 |
    cur_flags << 16).  Host only."""

    def __init__(self, label: bytes = None, state: bytes = None):
        self._lib = load()
        self._st = ctypes.create_string_buffer(TRANSCRIPT_BYTES)
        if state is not None:
            if len(state) != TRANSCRIPT_BYTES:
                raise ValueError(f"state: {TRANSCRIPT_BYTES} bytes")
            ctypes.memmove(self._st, state, TRANSCRIPT_BYTES)
        else:
            if label is None:
                raise ValueError("Transcript(label) or Transcript(state=...)")
            _status(self._lib, self._lib.bpp_transcript_new(label, len(label), self._st))

    @property
    def state(self) -> bytes:
        return self._st.raw

    def clone(self) -> "Transcript":
        return Transcript(state=self.state)

    def append_message(self, label: bytes, message: bytes):
        _status(self._lib, self._lib.bpp_transcript_append_message(self._st, label, len(label), message, len(message)))

    def append_u64(self, label: bytes, x: int):
        self.append_message(label, int(x).to_bytes(8, "little"))

    def challenge_bytes(self, label: bytes, n: int) -> bytes:
        out = ctypes.create_string_buffer(n)
        _status(self._lib, self._lib.bpp_transcript_challenge_bytes(self._st, label, len(label), out, n))
        return out.raw


def proof_len(n: int) -> int:
    """32 (2 lg n + 2); 0 unless n is a power of two"""
    return load().bpp_ipa_proof_len(n)


def _states(transcripts: Sequence[Transcript], count: int) -> ctypes.Array:
    if len(transcripts) != count:
        raise ValueError(f"{count} transcripts expected")
    buf = ctypes.create_string_buffer(TRANSCRIPT_BYTES * count)
    ctypes.memmove(buf, b"".join(t.state for t in transcripts), TRANSCRIPT_BYTES * count)
    return buf


def _write_back(transcripts: Sequence[Transcript], buf, only: Optional[bytes] = None):
    raw = buf.raw
    for p, t in enumerate(transcripts):
        if only is None or only[p]:
            ctypes.memmove(t._st, raw[TRANSCRIPT_BYTES * p:TRANSCRIPT_BYTES * (p + 1)], TRANSCRIPT_BYTES)


class InnerProductBatch:
    """`count` inner-product proofs of length n (a power of two, <= 8192) over `gens`.  Scalars are 32-byte
    little-endian, concatenated per proof: a, b, G_factors, H_factors count x n x 32; q count x 32; None factors or q
    stand for ones."""

    def __init__(self, backend: Backend, gens: Points, g_off: int, h_off: int, q_off: int, n: int, count: int):
        self.be, self.n, self.count = backend, n, count
        self.proof_len = proof_len(n)
        hnd = ctypes.c_void_p()
        backend._check(backend._lib.bpp_ipa_batch_create(backend._ctx, gens._h, g_off, h_off, q_off, n, count,
                                                          ctypes.byref(hnd)))
        self._h = hnd
        backend._adopt(self)

    def prove(self, transcripts: Sequence[Transcript], a: bytes, b: bytes, q: bytes = None, G_factors: bytes = None,
              H_factors: bytes = None) -> bytes:
        """InnerProductProof::create for every proof; the transcripts advance as create advances them.  Returns
        count x proof_len bytes (L_0 R_0 .. a b each)."""
        st = _states(transcripts, self.count)
        out = ctypes.create_string_buffer(self.proof_len * self.count)
        self.be._check(self.be._lib.bpp_ipa_batch_prove(self._h, q, G_factors, H_factors, a, b, st, out))
        _write_back(transcripts, st)
        return out.raw

    def verify(self, transcripts: Sequence[Transcript], P: bytes, proofs: bytes, q: bytes = None, G_factors: bytes = None,
               H_factors: bytes = None) -> bytes:
        """InnerProductProof::verify for every proof (P: count x 32 compressed).  Returns count accept bytes; the
        transcripts of accepted proofs advance as verify advances them, the others stay as they were."""
        st = _states(transcripts, self.count)
        acc = ctypes.create_string_buffer(self.count)
        self.be._check(self.be._lib.bpp_ipa_batch_verify(self._h, q, G_factors, H_factors, P, proofs, st, acc))
        _write_back(transcripts, st, acc.raw)
        return acc.raw

    def verify_combined(self, transcripts: Sequence[Transcript], P: bytes, proofs: bytes, q: bytes = None,
                        G_factors: bytes = None, H_factors: bytes = None, verifier_seed: bytes = None) -> bytes:
        """The decisions and transcripts of `verify`, through one random-linear-combination MSM over the batch (every
        proof on its own only when that combination is not the identity, or for batches of fewer than 1024 proof
        points).  verifier_seed: 32 bytes of secret, fresh randomness; None = the library draws them from the OS."""
        if verifier_seed is not None and len(verifier_seed) != 32:
            raise ValueError("verifier_seed: 32 bytes or None")
        st = _states(transcripts, self.count)
        acc = ctypes.create_string_buffer(self.count)
        self.be._check(self.be._lib.bpp_ipa_batch_verify_combined(self._h, q, G_factors, H_factors, P, proofs, verifier_seed,
                                                                  st, acc))
        _write_back(transcripts, st, acc.raw)
        return acc.raw

    def gather_accept(self, per: int) -> bytes:
        """Sharded verification: all ranks' accept bytes of their last verify (nranks x per, rank r's at r * per),
        through the library's NCCL communicator (Backend.comm_init); this rank's own bytes without one."""
        nr, _ = self.be.comm_info()
        out = ctypes.create_string_buffer(per * nr)
        self.be._check(self.be._lib.bpp_ipa_batch_gather_accept(self._h, per, out))
        return out.raw

    def free(self):
        if self._h and self.be._ctx:
            self.be._lib.bpp_ipa_batch_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
