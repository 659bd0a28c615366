"""GPU parity of the Ristretto decode (RFC 9496 4.3.1, ge_decompress): the point ingestion kernel and the verifier's
decompression kernels against oracle/ristretto255.py, for valid encodings and for every class of invalid one."""
import random

import pytest

from oracle import acproof as A, cref, ipa, ristretto255 as R
from oracle.chacha import ChaChaRng

pytestmark = pytest.mark.gpu
P = R.P


def _classify(enc: bytes) -> str:
    """Why oracle decompress rejects enc ("valid" when it does not), following RFC 9496 4.3.1 step by step."""
    s = int.from_bytes(enc, "little")
    if s >= P:
        return "non-canonical"
    if s & 1:
        return "negative-s"
    ss = s * s % P
    u1, u2 = (1 - ss) % P, (1 + ss) % P
    u2s = u2 * u2 % P
    v = (-(R.D * u1 % P * u1) - u2s) % P
    ok, inv = R.sqrt_ratio_i(1, v * u2s % P)
    if not ok:
        return "non-square"
    dx = inv * u2 % P
    x = R._abs(2 * s * dx)
    y = u1 * (inv * dx % P * v % P) % P
    if R._is_neg(x * y % P):
        return "negative-t"
    if y == 0:
        return "y-zero"
    return "valid"


def _invalid_encodings():
    """Two encodings of every invalid class (y = 0 has one even canonical encoding, p - 1)."""
    rng = random.Random(9496)
    out = {"non-canonical": [P + 1, 2 ** 256 - 2], "negative-s": [1, R.compress(R.pt_mul(7, R.BASEPOINT))],
           "y-zero": [P - 1], "non-square": [], "negative-t": []}
    while len(out["non-square"]) < 2 or len(out["negative-t"]) < 2:
        s = rng.randrange(0, P) & ~1
        c = _classify(s.to_bytes(32, "little"))
        if c in ("non-square", "negative-t") and len(out[c]) < 2:
            out[c].append(s)
    for c, v in out.items():
        out[c] = [e if isinstance(e, bytes) else e.to_bytes(32, "little") for e in v]
        if c == "negative-s":
            out[c][1] = bytes([out[c][1][0] | 1]) + out[c][1][1:]
    for c, v in out.items():
        assert all(_classify(e) == c for e in v), c
    return out


def _valid_encodings():
    """The RFC 9496 A.1 multiples 0..15 of the generator and random points."""
    rng = ChaChaRng(b"\x31" * 32)
    encs = [R.compress(R.pt_mul(i, R.BASEPOINT)) for i in range(16)]
    encs += [R.compress(R.from_uniform_bytes(rng.fill_bytes(64))) for _ in range(200)]
    assert all(_classify(e) == "valid" for e in encs)
    return encs


def test_decode_round_trips_valid_encodings(backend):
    encs = _valid_encodings()
    assert encs[1].hex() == "e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76"   # RFC 9496 A.1
    pts = backend.upload_points(encs)
    assert backend.compress_points(pts) == b"".join(encs)
    # the decoded points also enter an MSM correctly: sum of (i + 1) * P_i
    sc = b"".join(R.sc_bytes(i + 1) for i in range(len(encs)))
    assert backend.vartime_multiscalar_mul(sc, pts) == cref.msm(sc, cref.decompress(b"".join(encs)))
    pts.free()


def test_decode_rejects_every_invalid_class(backend):
    from bpperm_b200._lib import BppError
    good = _valid_encodings()[:3]
    for cls, encs in _invalid_encodings().items():
        for e in encs:
            assert R.decompress(e) is None
            with pytest.raises(BppError):
                backend.upload_points(good + [e])


def _sb(v):
    return b"".join(R.sc_bytes(s) for s in v)


@pytest.mark.parametrize("mode", ["reference-fixed", "fixed"])
def test_verifier_rejects_invalid_commitment_and_proof_points(backend, mode):
    """Proof 0 intact; then one proof per invalid class with V_0 replaced, one per class with T_i replaced (i cycles
    over T1, T3, T4, T5, T6), and in `fixed` mode one per class with L_0 replaced; the last proof has a valid but wrong
    T1.  Accept bytes: 1 for proof 0 only."""
    from bpperm_b200 import acproof as G
    k = 4
    maker = ipa.make_instance if mode == "fixed" else A.make_instance
    core, prover, V = maker(k, ChaChaRng(b"\x44" * 32))
    WL, WR, WO, WV = core["sparse"]
    cir = G.Circuit(backend, core["n"], core["Q"], core["m"], WL, WR, WO, WV, core["c_vec"])
    gens = G.Generators(backend, R.compress(core["g_base"]), R.compress(core["h_base"]),
                        [R.compress(p) for p in core["G_vec"]], [R.compress(p) for p in core["H_vec"]])
    n, m = core["n"], core["m"]
    bad = [e for v in _invalid_encodings().values() for e in v]
    fields = [None] + [("V", e) for e in bad] + [("T", e) for e in bad]
    if mode == "fixed":
        fields += [("L", e) for e in bad]
    fields.append(("T", R.compress(R.pt_mul(3, R.BASEPOINT))))
    B = len(fields)
    Vc = bytearray(b"".join(R.compress(p) for p in V) * B)
    seeds = b"".join(bytes([i + 1]) * 32 for i in range(B))
    proofs = bytearray(G.prove_batch(backend, cir, gens, _sb(prover["a_L"]) * B, _sb(prover["a_R"]) * B,
                                     _sb(prover["a_O"]) * B, _sb(prover["gamma"]) * B, seeds, B, mode, V=bytes(Vc)))
    plen = G.proof_len(n, mode) if mode == "fixed" else G.proof_len(n)
    assert list(G.verify_batch(backend, cir, gens, bytes(proofs), bytes(Vc), B, mode)) == [1] * B
    t_words = [3, 4, 5, 6, 7]
    for i, f in enumerate(fields):
        if f is None:
            continue
        kind, e = f
        if kind == "V":
            Vc[i * 32 * m: i * 32 * m + 32] = e
        else:
            w = t_words[i % 5] if kind == "T" else 11
            proofs[i * plen + 32 * w: i * plen + 32 * w + 32] = e
    acc = list(G.verify_batch(backend, cir, gens, bytes(proofs), bytes(Vc), B, mode))
    assert acc == [1] + [0] * (B - 1)
