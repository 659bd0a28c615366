"""GPU parity of the stand-alone inner-product batch (bpp_ipa_batch_*) against oracle/ipa.py
(InnerProductProof.create) and a restatement of bulletproofs 4.0.0 InnerProductProof::verify, per proof: proof bytes,
the transcript state left behind, and accept decisions under tampering; plus every launch form of the rounds and a
cross-check against the `fixed` mode prover, which runs the same rounds with Q = w g and H_factors = y^-n."""
import random

import pytest

from oracle import cref, ipa, ristretto255 as R
from oracle.chacha import ChaChaRng
from oracle.merlin import Transcript as OTranscript

pytestmark = pytest.mark.gpu
L = R.L


def _sb(v):
    return b"".join(R.sc_bytes(s) for s in v)


class _Set:
    """nG + nH + 1 random generators, uploaded as one point set: Q base at 0, G from 1, H after G"""

    def __init__(self, backend, n, seed, window_bits=0):
        rng = ChaChaRng(bytes([seed]) * 32)
        self.Q = rng.point()
        self.G = [rng.point() for _ in range(n)]
        self.H = [rng.point() for _ in range(n)]
        self.enc = [R.compress(p) for p in [self.Q] + self.G + self.H]
        self.pts = backend.upload_points(self.enc)
        if window_bits:
            backend.precompute(self.pts, window_bits)
        self.n = n


def _oracle_verify(trans, q, gf, hf, P_enc, proof, G, H, Qbase):
    """bulletproofs 4.0.0 InnerProductProof::from_bytes + verify"""
    n = len(G)
    lg = n.bit_length() - 1
    if len(proof) != 32 * (2 * lg + 2):
        return False
    w = [proof[32 * i:32 * i + 32] for i in range(2 * lg + 2)]
    a, b = int.from_bytes(w[-2], "little"), int.from_bytes(w[-1], "little")
    if a >= L or b >= L:
        return False
    pr = ipa.InnerProductProof(w[0:2 * lg:2], w[1:2 * lg:2], a, b)
    vs = pr.verification_scalars(n, trans)
    if vs is None:
        return False
    u_sq, u_inv_sq, s = vs
    Ls = [R.decompress(x) for x in pr.L_vec]
    Rs = [R.decompress(x) for x in pr.R_vec]
    P = R.decompress(P_enc)
    if P is None or any(x is None for x in Ls + Rs):
        return False
    gs = [a * s[i] % L * gf[i] % L for i in range(n)]
    hs = [b * s[n - 1 - i] % L * hf[i] % L for i in range(n)]
    rhs = R.vartime_multiscalar_mul(gs + hs + [a * b % L * q % L] + [(L - x) % L for x in u_sq] + [(L - x) % L for x in u_inv_sq],
                                    G + H + [Qbase] + Ls + Rs)
    return R.pt_eq(P, rhs)


def _fast_create(trans, q, gf, hf, Graw, Hraw, Qraw, a, b):
    """InnerProductProof::create with the generators never folded (the scalar-fold form of ipa_kernels.cuh) and the
    MSMs in C: the same bytes as oracle/ipa.py (checked in test_fast_restatement_matches_the_oracle) at sizes where the
    Python oracle takes minutes"""
    n = len(a)
    lg = n.bit_length() - 1
    ipa.innerproduct_domain_sep(trans, n)
    a, b = list(a), list(b)
    s, si = [1], [1]
    out = b""
    for j in range(lg):
        nj = n >> j
        h = nj // 2
        sc_L, sc_R, pts_L, pts_R = [], [], [], []
        for g in range(n):
            i, t = g % nj, g // nj
            if i >= h:
                sc_L.append(a[i - h] * s[t] % L * gf[g] % L); pts_L.append(Graw[g])
                sc_R.append(b[i - h] * si[t] % L * hf[g] % L); pts_R.append(Hraw[g])
            else:
                sc_R.append(a[i + h] * s[t] % L * gf[g] % L); pts_R.append(Graw[g])
                sc_L.append(b[i + h] * si[t] % L * hf[g] % L); pts_L.append(Hraw[g])
        c_L = sum(x * y for x, y in zip(a[:h], b[h:nj])) % L
        c_R = sum(x * y for x, y in zip(a[h:nj], b[:h])) % L
        Lc = cref.msm(_sb(sc_L + [c_L * q % L]), b"".join(pts_L + [Qraw]))
        Rc = cref.msm(_sb(sc_R + [c_R * q % L]), b"".join(pts_R + [Qraw]))
        trans.append_point(b"L", Lc)
        trans.append_point(b"R", Rc)
        out += Lc + Rc
        u = trans.challenge_scalar(b"u")
        ui = R.sc_inv(u)
        a = [(x * u + ui * y) % L for x, y in zip(a[:h], a[h:nj])]
        b = [(x * ui + u * y) % L for x, y in zip(b[:h], b[h:nj])]
        s = [v for x in s for v in (x * ui % L, x * u % L)]
        si = [v for x in si for v in (x * u % L, x * ui % L)]
    return out + R.sc_bytes(a[0]) + R.sc_bytes(b[0])


def _inputs(rs, count, n, factors):
    a = [[rs.randrange(L) for _ in range(n)] for _ in range(count)]
    b = [[rs.randrange(L) for _ in range(n)] for _ in range(count)]
    q = [rs.randrange(L) for _ in range(count)]
    gf = [[rs.randrange(L) for _ in range(n)] if factors else [1] * n for _ in range(count)]
    hf = [[rs.randrange(L) for _ in range(n)] if factors else [1] * n for _ in range(count)]
    return a, b, q, gf, hf


def _transcripts(rs, count):
    """random prefixes, built on both sides with the same calls"""
    from bpperm_b200.ipa import Transcript
    ours, ref = [], []
    for _ in range(count):
        lab = rs.randbytes(rs.randrange(1, 12))
        t, o = Transcript(lab), OTranscript(lab)
        for _ in range(rs.randrange(0, 4)):
            l, m = rs.randbytes(rs.randrange(0, 9)), rs.randbytes(rs.randrange(0, 200))
            t.append_message(l, m)
            o.append_message(l, m)
        ours.append(t)
        ref.append(o)
    return ours, ref


def _batch(backend, S, n, count):
    from bpperm_b200.ipa import InnerProductBatch
    return InnerProductBatch(backend, S.pts, 1, 1 + S.n, 0, n, count)


def _prove(backend, S, n, count, seed, factors):
    rs = random.Random(seed)
    a, b, q, gf, hf = _inputs(rs, count, n, factors)
    ours, ref = _transcripts(rs, count)
    init = [t.state for t in ours]
    bt = _batch(backend, S, n, count)
    proofs = bt.prove(ours, b"".join(_sb(x) for x in a), b"".join(_sb(x) for x in b), _sb(q),
                      b"".join(_sb(x) for x in gf) if factors else None, b"".join(_sb(x) for x in hf) if factors else None)
    bt.free()
    return proofs, (a, b, q, gf, hf), ours, ref, init


@pytest.mark.parametrize("n,count", [(1, 3), (2, 4), (4, 5), (8, 3), (64, 3), (128, 4)])
@pytest.mark.parametrize("factors", [False, True])
def test_prove_matches_the_oracle_bytes_and_transcript(backend, n, count, factors):
    S = _Set(backend, n, 11)
    proofs, (a, b, q, gf, hf), ours, ref, init = _prove(backend, S, n, count, 1000 * n + count + factors, factors)
    plen = 32 * (2 * (n.bit_length() - 1) + 2)
    assert len(proofs) == count * plen
    for p in range(count):
        want = ipa.InnerProductProof.create(ref[p], R.pt_mul(q[p], S.Q), gf[p], hf[p], S.G, S.H, a[p], b[p]).to_bytes()
        assert proofs[p * plen:(p + 1) * plen] == want, p
        assert ours[p].challenge_bytes(b"next", 32) == ref[p].challenge_bytes(b"next", 32), p


def test_fast_restatement_matches_the_oracle():
    rs = random.Random(5)
    rng = ChaChaRng(b"\x05" * 32)
    n = 32
    Q, G, H = rng.point(), [rng.point() for _ in range(n)], [rng.point() for _ in range(n)]
    raw = lambda p: cref.decompress(R.compress(p))  # noqa: E731
    a, b, q, gf, hf = _inputs(rs, 1, n, True)
    want = ipa.InnerProductProof.create(OTranscript(b"t"), R.pt_mul(q[0], Q), gf[0], hf[0], G, H, a[0], b[0]).to_bytes()
    got = _fast_create(OTranscript(b"t"), q[0], gf[0], hf[0], [raw(p) for p in G], [raw(p) for p in H], raw(Q), a[0], b[0])
    assert got == want


def test_large_deck_shape_n8192_matches_the_restatement_and_verifies(backend):
    n = 8192
    S = _Set(backend, n, 12)
    proofs, (a, b, q, gf, hf), ours, ref, init = _prove(backend, S, n, 1, 77, True)
    raw = cref.decompress(b"".join(S.enc))
    PT = cref.PT
    Graw = [raw[PT * (1 + i):PT * (2 + i)] for i in range(n)]
    Hraw = [raw[PT * (1 + n + i):PT * (2 + n + i)] for i in range(n)]
    want = _fast_create(ref[0], q[0], gf[0], hf[0], Graw, Hraw, raw[:PT], a[0], b[0])
    assert proofs == want
    assert ours[0].challenge_bytes(b"next", 16) == ref[0].challenge_bytes(b"next", 16)
    # P = <a, G'> + <b, H'> + <a, b> Q with the factors applied
    P = cref.msm(_sb([x * f % L for x, f in zip(a[0], gf[0])] + [x * f % L for x, f in zip(b[0], hf[0])] +
                     [sum(x * y for x, y in zip(a[0], b[0])) * q[0] % L]), b"".join(Graw + Hraw + [raw[:PT]]))
    from bpperm_b200.ipa import Transcript
    bt = _batch(backend, S, n, 2)
    bad = bytearray(proofs)
    bad[-1] ^= 1   # b + 2^248: still canonical, wrong
    acc = bt.verify([Transcript(state=init[0]), Transcript(state=init[0])], P * 2, proofs + bytes(bad), _sb(q * 2),
                    _sb(gf[0]) * 2, _sb(hf[0]) * 2)
    assert acc == b"\x01\x00"


@pytest.mark.parametrize("n,count", [(8, 1), (8, 3), (8, 1100), (8, 1300), (64, 1100)])
def test_every_launch_form_matches_the_oracle_on_a_sample(backend, n, count):
    """count <= 1023: the fused tail (k_ipa_lr_tail); above: split + compress + k_ipa_challenge; 1300 proofs of n = 8:
    2600 outputs per round, the warp-per-output form on 148 SMs"""
    S = _Set(backend, n, 13)
    proofs, (a, b, q, gf, hf), ours, ref, init = _prove(backend, S, n, count, count * 7 + n, True)
    plen = 32 * (2 * (n.bit_length() - 1) + 2)
    for p in sorted(random.Random(count).sample(range(count), min(16, count))):
        want = ipa.InnerProductProof.create(ref[p], R.pt_mul(q[p], S.Q), gf[p], hf[p], S.G, S.H, a[p], b[p]).to_bytes()
        assert proofs[p * plen:(p + 1) * plen] == want, p
        assert ours[p].challenge_bytes(b"c", 8) == ref[p].challenge_bytes(b"c", 8), p


def test_reproduces_the_inner_product_words_of_a_fixed_mode_proof(backend):
    """52 cards, `fixed` mode: the oracle's prover state gives l, r, w, y and the transcript before the inner-product
    argument; the stand-alone prover with q = w, H_factors = y^-n over g, h, G, H (gens order of bpp_gens_create:
    g_off 2, h_off 2 + n', q_off 0) must give the last 2 lg n' + 2 words of the GPU `fixed` proof."""
    from bpperm_b200 import acproof as G
    from bpperm_b200.ipa import InnerProductBatch, Transcript
    rng = ChaChaRng(b"\x34" * 32)
    core, prover, V = ipa.make_instance(52, rng, dense_weights=True)
    n = core["n"]
    npad = ipa.next_pow2(n)
    lg = npad.bit_length() - 1
    seed = b"\x09" * 32
    # the oracle prover, its transcript captured where create() starts
    captured = {}
    orig = ipa.InnerProductProof.create.__func__

    def spy(cls, trans, Q, Gf, Hf, Gv, Hv, av, bv, msm=None):
        captured["tr"] = trans.clone()
        return orig(cls, trans, Q, Gf, Hf, Gv, Hv, av, bv, msm)
    ipa.InnerProductProof.create = classmethod(spy)
    try:
        ref_proof, st = ipa.prove(core, prover, V, ChaChaRng(seed))
    finally:
        ipa.InnerProductProof.create = classmethod(orig)
    WL, WR, WO, WV = core["sparse"]
    cir = G.Circuit(backend, core["n"], core["Q"], core["m"], WL, WR, WO, WV, core["c_vec"])
    gens = G.Generators(backend, R.compress(core["g_base"]), R.compress(core["h_base"]),
                        [R.compress(p) for p in core["G_vec"]], [R.compress(p) for p in core["H_vec"]])
    Vc = b"".join(R.compress(p) for p in V)
    gpu = G.prove_batch(backend, cir, gens, _sb(prover["a_L"]), _sb(prover["a_R"]), _sb(prover["a_O"]), _sb(prover["gamma"]),
                        seed, 1, "fixed", V=Vc)
    assert gpu == ref_proof
    # the transcript before the IPA, rebuilt through the ABI state (the oracle's Strobe state, byte for byte)
    s = captured["tr"].strobe
    state = bytes(s.state) + (s.pos | s.pos_begin << 8 | s.cur_flags << 16).to_bytes(8, "little")
    enc = [R.compress(core["g_base"]), R.compress(core["h_base"])] + [R.compress(p) for p in core["G_vec"][:npad]] + \
          [R.compress(p) for p in core["H_vec"][:npad]]
    pts = backend.upload_points(enc)
    bt = InnerProductBatch(backend, pts, 2, 2 + npad, 0, npad, 1)
    y_inv = R.sc_inv(st["y"])
    out = bt.prove([Transcript(state=state)], _sb(st["l"]), _sb(st["r"]), _sb([st["w"]]), None, _sb(ipa.std_powers(y_inv, npad)))
    assert out == gpu[-32 * (2 * lg + 2):]


def test_verify_accepts_valid_batches_and_follows_the_oracle_under_tampering(backend):
    from bpperm_b200.ipa import InnerProductBatch, Transcript
    n, count, lg = 8, 4, 3
    plen = 32 * (2 * lg + 2)
    S = _Set(backend, n, 14)
    a, b, q, gf, hf = _inputs(random.Random(21), count, n, True)
    labels = [b"ipa-test-%d" % p for p in range(count)]
    pbt = InnerProductBatch(backend, S.pts, 1, 1 + n, 0, n, count)
    proofs = pbt.prove([Transcript(x) for x in labels], b"".join(_sb(x) for x in a), b"".join(_sb(x) for x in b), _sb(q),
                       b"".join(_sb(x) for x in gf), b"".join(_sb(x) for x in hf))
    P = [R.compress(R.vartime_multiscalar_mul(
        [x * f % L for x, f in zip(a[p], gf[p])] + [x * f % L for x, f in zip(b[p], hf[p])] +
        [sum(x * y for x, y in zip(a[p], b[p])) * q[p] % L], S.G + S.H + [S.Q])) for p in range(count)]
    cases = [(labels[p], proofs[p * plen:(p + 1) * plen], P[p], q[p], gf[p], hf[p]) for p in range(count)]
    base = proofs[:plen]
    flip = lambda bts, i: bts[:i] + bytes([bts[i] ^ 1]) + bts[i + 1:]  # noqa: E731
    t0 = lambda pr, P0=P[0], q0=q[0], g0=gf[0], h0=hf[0]: (labels[0], pr, P0, q0, g0, h0)  # noqa: E731
    for j in range(lg):
        cases.append(t0(flip(base, 32 * 2 * j + 3)))
        cases.append(t0(flip(base, 32 * (2 * j + 1) + 5)))
    cases.append(t0(flip(base, 32 * 2 * lg)))                          # a
    cases.append(t0(flip(base, 32 * (2 * lg + 1) + 7)))                # b
    cases.append(t0(base, P0=P[1]))                                    # P
    cases.append(t0(base, q0=(q[0] + 1) % L))                          # q
    cases.append(t0(base, g0=[(gf[0][0] + 1) % L] + gf[0][1:]))        # a G factor
    cases.append(t0(base, h0=hf[0][:-1] + [(hf[0][-1] + 2) % L]))      # an H factor
    cases.append(t0(bytes(32) + base[32:]))                            # all-zero L_0
    cases.append(t0(base[:32] + b"\xff" * 32 + base[64:]))            # invalid R_0 encoding
    a_plus_l = (int.from_bytes(base[32 * 2 * lg:32 * 2 * lg + 32], "little") + L).to_bytes(32, "little")
    cases.append(t0(base[:32 * 2 * lg] + a_plus_l + base[-32:]))       # a + l
    cases.append(t0(base, P0=b"\xff" * 32))                           # invalid P
    cases.append((b"ipa-test-other",) + t0(base)[1:])                  # another transcript prefix
    bt = InnerProductBatch(backend, S.pts, 1, 1 + n, 0, n, len(cases))
    trs = [Transcript(c[0]) for c in cases]
    acc = bt.verify(trs, b"".join(c[2] for c in cases), b"".join(c[1] for c in cases), _sb([c[3] for c in cases]),
                    b"".join(_sb(c[4]) for c in cases), b"".join(_sb(c[5]) for c in cases))
    for i, (lab, pr, Pp, qq, g, h) in enumerate(cases):
        o = OTranscript(lab)
        want = _oracle_verify(o, qq, g, h, Pp, pr, S.G, S.H, S.Q)
        assert acc[i] == int(want), (i, acc[i], want)
        if want:   # the transcript left behind is dalek's
            assert trs[i].challenge_bytes(b"after", 16) == o.challenge_bytes(b"after", 16), i
    assert acc[:count] == b"\x01" * count and sum(acc[count:]) == 0


def test_argument_errors(backend):
    import ctypes
    from bpperm_b200 import BppError
    from bpperm_b200.ipa import InnerProductBatch, Transcript
    S = _Set(backend, 8, 15)
    for n in (3, 6, 16384, 0):
        with pytest.raises(BppError) as ei:
            InnerProductBatch(backend, S.pts, 1, 9, 0, n, 1)
        assert ei.value.status == -3, n
    with pytest.raises(BppError) as ei:
        InnerProductBatch(backend, S.pts, 1, 9, 0, 8, 0)
    assert ei.value.status == -3
    for g_off, h_off, q_off in ((10, 1, 0), (1, 10, 0), (1, 9, 17), (2 ** 63, 1, 0)):
        with pytest.raises(BppError) as ei:
            InnerProductBatch(backend, S.pts, g_off, h_off, q_off, 8, 1)
        assert ei.value.status == -4, (g_off, h_off, q_off)
    bt = InnerProductBatch(backend, S.pts, 1, 9, 0, 8, 2)
    ok = _sb([1] * 16)
    big = _sb([1] * 15) + L.to_bytes(32, "little")
    for kw in ({"a": big, "b": ok}, {"a": ok, "b": big}, {"a": ok, "b": ok, "q": _sb([1]) + (L + 5).to_bytes(32, "little")},
               {"a": ok, "b": ok, "G_factors": big}, {"a": ok, "b": ok, "H_factors": big}):
        with pytest.raises(BppError) as ei:
            bt.prove([Transcript(b"t"), Transcript(b"t")], **kw)
        assert ei.value.status == -6, kw.keys()
    lib = backend._lib
    st = ctypes.create_string_buffer(Transcript(b"t").state * 2)
    out = ctypes.create_string_buffer(2 * 256)
    assert lib.bpp_ipa_batch_prove(bt._h, None, None, None, None, ok, st, out) == -3
    assert lib.bpp_ipa_batch_verify(bt._h, None, None, None, None, out, st, out) == -3
    bad_state = ctypes.create_string_buffer(Transcript(b"t").state[:200] + (200).to_bytes(8, "little") + Transcript(b"t").state)
    assert lib.bpp_ipa_batch_prove(bt._h, None, None, None, ok, ok, bad_state, out) == -3
