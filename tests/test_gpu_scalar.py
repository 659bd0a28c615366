"""Scalar arithmetic mod l against Python integers, bit-exact, through bpp_test_op's scalar op codes: the primitives of
sc25519.cuh at limb and range edges, the unreduced sums of up to SC_MAC_MAX products that the dot kernels reduce once,
and the warp's nine-limb sum.  Then the dot kernels' chunk branch at proof level (batches of the warp form with lanes of
15 and 16 products), the reduction of caller scalars mod l at the shuffle prover's entry points, and the table MSM at
the edge of its digit range, every window width."""
import random

import numpy as np
import pytest

from oracle import acproof as A, cref, ristretto255 as R

L = R.L
RR = 2 ** 256
RINV = pow(RR, -1, L)
(SC_ADD, SC_SUB, SC_NEG, SC_MONT, SC_MUL, SC_INVERT, SC_REDUCE256, SC_FROM_WIDE, SC_MONT_REDUCE, SC_WARP_SUM,
 SC_MAC) = range(11, 22)
SC_MAC_MAX = 15
LIMBS = [0, 1, 2 ** 31, 2 ** 32 - 2, 2 ** 32 - 1]
# not canonical: each must give the bytes of its value mod l (or, for the _dev table MSM, of its low 255 bits)
RAW = [L, L + 1, 2 ** 255 - 1, 2 ** 255, 2 ** 255 + 2 ** 254, 2 ** 256 - 1]
INVALID_ARG = -3


def _le(x, w=32):
    return x.to_bytes(w, "little")


def _edges_raw():
    """Edge values as 256-bit integers, some >= l: limb patterns from LIMBS (every limb equal, alternating, seeded mixes)."""
    xs = [0, 1, 2, L - 2, L - 1, 2 ** 252 - 1, 2 ** 252, 2 ** 252 + 1, (L - 1) // 2, RR % L, RR * RR % L, 2 ** 128,
          2 ** 224 % L]
    xs += [sum(v << (32 * i) for i in range(8)) for v in LIMBS]
    xs += [sum((v if i % 2 else w) << (32 * i) for i in range(8)) for v in LIMBS for w in LIMBS if v != w]
    rnd = random.Random(5)
    xs += [sum(rnd.choice(LIMBS) << (32 * i) for i in range(8)) for _ in range(20)]
    return xs


def _edges():
    return sorted(set(x % L for x in _edges_raw()))


def _run(backend, op, pairs, w=32):
    a = b"".join(_le(x, w) for x, _ in pairs)
    b = b"".join(_le(y, w) for _, y in pairs)
    out = backend.test_op(op, a, b)
    return [int.from_bytes(out[32 * i:32 * i + 32], "little") for i in range(len(pairs))]


def _check(backend, op, pairs, fn):
    got = _run(backend, op, pairs)
    bad = [(hex(x), hex(y)) for (x, y), g in zip(pairs, got) if g != fn(x, y)]
    assert not bad, (op, len(bad), bad[:4])


def test_chunk_bound():
    """Why SC_MAC_MAX is 15: 15 products of canonical scalars stay below sc_mont_reduce's bound l * 2^256, 16 need not."""
    assert 15 * (L - 1) ** 2 < L * RR <= 16 * (L - 1) ** 2
    assert SC_MAC_MAX == 15


@pytest.mark.gpu
@pytest.mark.parametrize("op,fn", [(SC_ADD, lambda a, b: (a + b) % L), (SC_SUB, lambda a, b: (a - b) % L),
                                   (SC_MUL, lambda a, b: a * b % L), (SC_MONT, lambda a, b: a * b * RINV % L),
                                   (SC_NEG, lambda a, b: -a % L), (SC_INVERT, lambda a, b: pow(a, L - 2, L))],
                         ids=["add", "sub", "mul", "mont", "neg", "invert"])
def test_canonical_ops(backend, op, fn):
    """Every pair of canonical edge values, then 20 000 random pairs."""
    rnd = random.Random(op)
    e = _edges()
    pairs = [(a, b) for a in e for b in e] + [(rnd.randrange(L), rnd.randrange(L)) for _ in range(20000)]
    _check(backend, op, pairs, fn)


@pytest.mark.gpu
def test_mont_with_one_raw_operand(backend):
    """sc_mont needs a * b < l * 2^256 only: any 256-bit a against a canonical b."""
    rnd = random.Random(3)
    raw = _edges_raw() + RAW
    pairs = [(a, b) for a in raw for b in _edges()] + [(rnd.getrandbits(256), rnd.randrange(L)) for _ in range(20000)]
    _check(backend, SC_MONT, pairs, lambda a, b: a * b * RINV % L)


@pytest.mark.gpu
def test_reduce256_and_from_wide(backend):
    rnd = random.Random(4)
    raw = _edges_raw() + RAW
    _check(backend, SC_REDUCE256, [(a, 0) for a in raw] + [(rnd.getrandbits(256), 0) for _ in range(20000)],
           lambda a, b: a % L)
    pairs = [(a, b) for a in raw for b in raw] + [(rnd.getrandbits(256), rnd.getrandbits(256)) for _ in range(20000)]
    _check(backend, SC_FROM_WIDE, pairs, lambda lo, hi: (lo + (hi << 256)) % L)


@pytest.mark.gpu
def test_mont_reduce_at_its_bound(backend):
    """t = t_lo + 2^256 t_hi for t < l * 2^256: the largest t, t_lo = 0 (the carry sc_mont_reduce derives from t_lo != 0),
    t_hi = 0, multiples of l, products of edge values, random t."""
    rnd = random.Random(6)
    ts = [L * RR - 1, RR, (L - 1) * RR, L * RR - RR, L * RR - RR + 1]
    ts += [x for x in _edges_raw() + RAW]                                 # t_hi = 0
    ts += [h * RR for h in _edges()]                                       # t_lo = 0
    ts += [q * L for q in [1, 2, 2 ** 128, 2 ** 255, RR - 1] + [rnd.getrandbits(256) for _ in range(100)]]
    e = _edges()
    ts += [a * b for a in e for b in e]
    ts += [rnd.randrange(L * RR) for _ in range(20000)]
    assert all(0 <= t < L * RR for t in ts)
    got = _run(backend, SC_MONT_REDUCE, [(t % RR, t >> 256) for t in ts])
    bad = [hex(t) for t, g in zip(ts, got) if g != t * RINV % L]
    assert not bad, (len(bad), bad[:4])


def _mac_want(a, b, K):
    n = len(a)
    return [sum(a[(i + j) % n] * b[(i + j) % n] for j in range(K)) * RINV % L for i in range(n)]


@pytest.mark.gpu
def test_mac_sums_up_to_the_chunk(backend):
    """sc_mac sums of K = 1..SC_MAC_MAX products, reduced once: every operand l - 1 (the largest sum), the Montgomery
    forms of the edge values, random operands.  K = SC_MAC_MAX + 1 is refused: a 16th product of l - 1 passes the bound."""
    import bpperm_b200
    n = 64
    top = [L - 1] * n
    e = _edges()
    mont = [x * RR % L for x in e] + [L - 1, L - 2]
    ma = [mont[i % len(mont)] for i in range(2 * n)]
    mb = [mont[(7 * i + 3) % len(mont)] for i in range(2 * n)]
    rnd = random.Random(9)
    ra = [rnd.randrange(L) for _ in range(2000)]
    rb = [rnd.randrange(L) for _ in range(2000)]
    for K in range(1, SC_MAC_MAX + 2):
        for a, b in ((top, top), (ma, mb), (ra, rb)):
            if K > SC_MAC_MAX:
                with pytest.raises(bpperm_b200.BppError) as ei:
                    _run(backend, SC_MAC + K - 1, list(zip(a, b)))
                assert ei.value.status == INVALID_ARG
                continue
            assert _run(backend, SC_MAC + K - 1, list(zip(a, b))) == _mac_want(a, b, K), (K, len(a))
    # the largest sum the dot kernels reduce: 15 (l - 1)^2, and 15 Montgomery products of the edges' largest forms
    assert _run(backend, SC_MAC + SC_MAC_MAX - 1, [(L - 1, L - 1)] * 32) == [SC_MAC_MAX * (L - 1) ** 2 * RINV % L] * 32


@pytest.mark.gpu
def test_warp_sum(backend):
    """warp_sum9 + sc_from9 over groups of 32 lanes: all l - 1, all 0, all 2^256 - 1 (any 256-bit lane value fits the
    nine limbs), mixed and random groups.  n % 32 != 0 is refused."""
    import bpperm_b200
    rnd = random.Random(11)
    groups = [[L - 1] * 32, [0] * 32, [2 ** 256 - 1] * 32, [L - 1 if i % 2 else 0 for i in range(32)],
              [rnd.choice(_edges()) for _ in range(32)]] + [[rnd.randrange(L) for _ in range(32)] for _ in range(600)]
    vals = [v for g in groups for v in g]
    got = _run(backend, SC_WARP_SUM, [(v, 0) for v in vals])
    for gi, g in enumerate(groups):
        assert got[32 * gi:32 * gi + 32] == [sum(g) % L] * 32, gi
    with pytest.raises(bpperm_b200.BppError) as ei:
        _run(backend, SC_WARP_SUM, [(1, 0)] * 48)
    assert ei.value.status == INVALID_ARG


# ------------------------------------------------------------------------------ the dot kernels' chunk at proof level
def _sb(v):
    return b"".join(_le(s) for s in v)


def _witness(k, v):
    """a_L, a_R, a_O of the shuffle circuit for v = input deck | output deck | x (tests/test_gpu_acproof_decisions.py)."""
    n, x = 2 * k, v[-1]
    aL, aR, aO = [0] * n, [0] * n, [0] * n
    for gb, vb in ((0, 0), (k - 1, k)):
        for i in range(k - 1):
            aL[gb + i] = (v[vb] - x) % L if i == 0 else aO[gb + i - 1]
            aR[gb + i] = (v[vb + i + 1] - x) % L
            aO[gb + i] = aL[gb + i] * aR[gb + i] % L
    return aL, aR, aO


class _Setup:
    """The library's k-card shuffle circuit and generators, and the C restatement over the same points: the dense
    instance (cref.AcpInstance) for "reference-fixed", the sparse one with next_pow2(n) generators for "fixed"."""

    def __init__(self, backend, k, mode, seed):
        from bpperm_b200 import acproof as G
        n, Q, m, WL, WR, WO, WV, cv = A.shuffle_circuit(k)
        self.k, self.n, self.m, self.mode = k, n, m, mode
        ng = G.next_pow2(n) if mode == "fixed" else n
        rs = np.random.RandomState(seed)
        enc = cref.compress(cref.from_uniform(rs.randint(0, 256, size=(2 * ng + 2, 64), dtype=np.uint8).tobytes()))
        p = [enc[32 * i:32 * i + 32] for i in range(2 * ng + 2)]
        if mode == "fixed":
            self.inst = cref.AcpFixedInstance(n, Q, m, WL, WR, WO, WV, _sb(cv), p[0], p[1], b"".join(p[2:2 + ng]),
                                              b"".join(p[2 + ng:]))
        else:
            def dense(M, rows):
                return b"".join(_sb(r) for r in A.dense(M, rows, Q))
            self.inst = cref.AcpInstance(n, Q, m, dense(WL, n), dense(WR, n), dense(WO, n), dense(WV, m), _sb(cv), p[0],
                                         p[1], b"".join(p[2:2 + n]), b"".join(p[2 + n:]))
        self.cir = G.Circuit.shuffle(backend, k)
        self.gens = G.Generators(backend, p[0], p[1], p[2:2 + ng], p[2 + ng:], 8)

    def prove(self, aL, aR, aO, gamma, Ve, seed):
        V = cref.decompress(Ve)
        if self.mode == "fixed":
            return self.inst.prove(_sb(aL), _sb(aR), _sb(aO), _sb(gamma), V, seed, V_enc=Ve)
        return self.inst.prove_verify(_sb(aL), _sb(aR), _sb(aO), _sb(gamma), V, seed, 1, do_verify=False, V_enc=Ve)[0]

    def verify(self, proof, Ve):
        if self.mode == "fixed":
            return self.inst.verify(proof, cref.decompress(Ve), V_enc=Ve)
        return self.inst.verify(proof, None, 1, V_enc=Ve)

    def free(self):
        self.gens.free()
        self.cir.free()


def _deck(k):
    return [L - 1, L - 2, 2 ** 252, 2 ** 255 % L] + list(range(1, k - 3))


def _inputs(k, B, seed):
    rs = np.random.RandomState(seed)
    m = 2 * k + 1
    perm = np.stack([rs.permutation(k) for _ in range(B)]).astype(np.uint32)
    x = [int.from_bytes(rs.bytes(32), "little") % L for _ in range(B)]
    gamma = [[int.from_bytes(rs.bytes(32), "little") % L for _ in range(m)] for _ in range(B)]
    seeds = [rs.bytes(32) for _ in range(B)]
    return perm, x, gamma, seeds


def _prove_gen(backend, s, deck, perm, x, gamma, seeds):
    from bpperm_b200 import acproof as G
    B = len(x)
    b = G.Batch(backend, s.cir, s.gens, B, s.mode)
    b.gen_shuffle_witness(_sb(deck), perm.tobytes(), _sb(x), b"".join(_sb(g) for g in gamma), b"".join(seeds))
    V = b.commit(None)
    b.prove()
    P = b.download_proofs()
    return b, V, P


@pytest.mark.gpu
@pytest.mark.parametrize("k,mode", [(240, "reference-fixed"), (241, "reference-fixed"), (240, "fixed"), (256, "fixed")])
def test_dot_chunks_in_the_warp_form(backend, k, mode):
    """B = 256 takes k_acp_dots_warp.  k = 240 (n = 480): 15 products per lane in the first stage, so the chunk reduce
    fires on the last element and the final reduce sees t = 0; m = 481 gives lane 0 a 16th product.  k = 241: lanes 0
    and 1 get 16.  `fixed` at k = 256: n' = 512 for t_hat.  Proofs equal the C prover's, the GPU verifier accepts all,
    and a B = 255 batch (the block form, k_acp_dots) of the same inputs gives the same proofs."""
    s = _Setup(backend, k, mode, 7000 + k)
    B, m = 256, s.m
    deck = _deck(k)
    perm, x, gamma, seeds = _inputs(k, B, 100 + k)
    b, V, P = _prove_gen(backend, s, deck, perm, x, gamma, seeds)
    plen, vlen = b.proof_len, 32 * m
    for p in (0, 1, 31, 32, 255):
        v = deck + [deck[j] for j in perm[p]] + [x[p]]
        aL, aR, aO = _witness(k, v)
        Ve = V[p * vlen:(p + 1) * vlen]
        assert Ve == cref.compress(s.inst.commit(_sb(v), _sb(gamma[p]))), p
        assert P[p * plen:(p + 1) * plen] == s.prove(aL, aR, aO, gamma[p], Ve, seeds[p]), (k, mode, p)
    b.upload_proofs(P, V)
    b.verify(b"\x05" * 32)
    assert b.download_accept() == b"\x01" * B
    b.free()
    b2, V2, P2 = _prove_gen(backend, s, deck, perm[:255], x[:255], gamma[:255], seeds[:255])
    assert V2 == V[:255 * vlen]
    for p in (0, 1, 31, 32, 254):
        assert P2[p * plen:(p + 1) * plen] == P[p * plen:(p + 1) * plen], (k, mode, p)
    b2.free()
    s.free()


@pytest.mark.gpu
def test_unsatisfied_witness_of_largest_operands_in_the_warp_form(backend):
    """Every a_L, a_R, a_O = l - 1 (the constraints do not hold): the largest products the dot kernels sum.  A sample of
    the proofs equals the C prover's; GPU and C verifier both reject."""
    from bpperm_b200 import acproof as G
    k, B = 240, 256
    s = _Setup(backend, k, "reference-fixed", 7300)
    n, m = s.n, s.m
    rs = np.random.RandomState(17)
    vs = [[int.from_bytes(rs.bytes(32), "little") % L for _ in range(m)] for _ in range(B)]
    gamma = [[int.from_bytes(rs.bytes(32), "little") % L for _ in range(m)] for _ in range(B)]
    seeds = [rs.bytes(32) for _ in range(B)]
    top = _sb([L - 1] * n) * B
    b = G.Batch(backend, s.cir, s.gens, B, "reference-fixed")
    b.upload_witness(top, top, top, b"".join(_sb(g) for g in gamma), b"".join(seeds))
    V = b.commit(b"".join(_sb(v) for v in vs))
    b.prove()
    P = b.download_proofs()
    plen, vlen = b.proof_len, 32 * m
    for p in (0, 31, 255):
        Ve = V[p * vlen:(p + 1) * vlen]
        pb = P[p * plen:(p + 1) * plen]
        assert pb == s.prove([L - 1] * n, [L - 1] * n, [L - 1] * n, gamma[p], Ve, seeds[p]), p
        assert not s.verify(pb, Ve)
    b.upload_proofs(P, V)
    b.verify(b"\x05" * 32)
    assert b.download_accept() == bytes(B)
    b.free()
    s.free()


# ------------------------------------------------------------------------ caller scalars at the prover's entry points
def _raw_spread(vals, rs, frac=0.25):
    """(raw, reduced): vals with each value of RAW in the first slots and a share of the others replaced by their
    largest representative below a value of RAW (>= l, up to 2^256 - 1); reduced = raw mod l."""
    out = list(vals)
    for i in range(len(out)):
        if rs.rand() < frac:
            v = out[i] % L
            out[i] = v + (RAW[rs.randint(len(RAW))] - v) // L * L
    for i, r in enumerate(RAW):
        out[i % len(out)] = r
    return out, [v % L for v in out]


def _to_dev(buf):
    import torch
    return torch.frombuffer(bytearray(buf), dtype=torch.uint8).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["host", "device"])
def test_uploaded_witness_and_v_are_taken_mod_l(backend, where):
    """bpp_acp_batch_upload_witness and bpp_acp_batch_commit(v): a_L, a_R, a_O, gamma and v holding values >= l (up to
    2^256 - 1) give the commitments and proofs of the same values reduced on the host."""
    import torch
    from bpperm_b200 import acproof as G
    k, B = 5, 40
    s = _Setup(backend, k, "reference-fixed", 7400)
    n, m = s.n, s.m
    rs = np.random.RandomState(23)
    deck = _deck(k)
    perm, x, gamma, seeds = _inputs(k, B, 24)
    wit = [_witness(k, deck + [deck[j] for j in perm[p]] + [x[p]]) for p in range(B)]
    vs = [deck + [deck[j] for j in perm[p]] + [x[p]] for p in range(B)]
    flat = {"aL": [a for w in wit for a in w[0]], "aR": [a for w in wit for a in w[1]], "aO": [a for w in wit for a in w[2]],
            "gamma": [g for gg in gamma for g in gg], "v": [v for vv in vs for v in vv]}
    spread = {key: _raw_spread(val, rs) for key, val in flat.items()}
    raw = {key: val[0] for key, val in spread.items()}
    red = {key: val[1] for key, val in spread.items()}
    assert all(any(v >= L for v in val) for val in raw.values())
    seeds_b = b"".join(seeds)
    out = []
    for vals in (red, raw):
        bufs = {key: _sb(val) for key, val in vals.items()}
        b = G.Batch(backend, s.cir, s.gens, B, "reference-fixed")
        if where == "host":
            b.upload_witness(bufs["aL"], bufs["aR"], bufs["aO"], bufs["gamma"], seeds_b)
            V = b.commit(bufs["v"])
        else:
            d = {key: _to_dev(buf) for key, buf in bufs.items()}
            d_seeds = _to_dev(seeds_b)
            torch.cuda.synchronize()
            b.upload_witness_ptr(d["aL"].data_ptr(), d["aR"].data_ptr(), d["aO"].data_ptr(), d["gamma"].data_ptr(),
                                 d_seeds.data_ptr())
            V = b.commit(d["v"].data_ptr())
        b.prove()
        out.append((V, b.download_proofs()))
        b.free()
    assert out[1][0] == out[0][0]
    assert out[1][1] == out[0][1]
    plen = G.proof_len(n)
    assert out[0][1][:plen] == s.prove(red["aL"][:n], red["aR"][:n], red["aO"][:n], red["gamma"][:m], out[0][0][:32 * m],
                                       seeds[0])
    s.free()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["host", "device"])
def test_generated_witness_inputs_are_taken_mod_l(backend, where):
    """bpp_acp_batch_gen_shuffle_witness: deck, x and gamma holding values >= l give the commitments and proofs of the
    same values reduced on the host."""
    import torch
    from bpperm_b200 import acproof as G
    k, B = 6, 40
    s = _Setup(backend, k, "reference-fixed", 7500)
    rs = np.random.RandomState(29)
    deck = _deck(k)
    perm, x, gamma, seeds = _inputs(k, B, 30)
    (deck_raw, deck_red), (x_raw, x_red), (g_raw, g_red) = (_raw_spread(deck, rs, 0.5), _raw_spread(x, rs),
                                                            _raw_spread([g for gg in gamma for g in gg], rs))
    out = []
    for d_, x_, g_ in ((deck_red, x_red, g_red), (deck_raw, x_raw, g_raw)):
        bufs = [_sb(d_), perm.tobytes(), _sb(x_), _sb(g_), b"".join(seeds)]
        b = G.Batch(backend, s.cir, s.gens, B, "reference-fixed")
        if where == "host":
            b.gen_shuffle_witness(*bufs)
        else:
            d = [_to_dev(buf) for buf in bufs]
            torch.cuda.synchronize()
            b.gen_shuffle_witness(*[t.data_ptr() for t in d])
        V = b.commit(None)
        b.prove()
        out.append((V, b.download_proofs()))
        b.free()
    assert out[1][0] == out[0][0]
    assert out[1][1] == out[0][1]
    s.free()


@pytest.mark.gpu
def test_dev_table_msm_ignores_bit_255(backend):
    """bpp_msm_vartime_batch_dev clears bit 255 of every scalar, as bpp_msm_mixed_dev does: scalars with it set give
    the host form's bytes for the same scalars with it cleared (which the host form alone would refuse)."""
    import torch
    rs = np.random.RandomState(31)
    n, c = 9, 8
    pts = backend.upload_points(cref.compress(cref.from_uniform(rs.randint(0, 256, size=(n, 64), dtype=np.uint8).tobytes())))
    backend.precompute(pts, c)
    for count in (3, 2400):               # the block and the warp form
        vals = [RAW[i % len(RAW)] if i % 3 == 0 else int.from_bytes(rs.bytes(32), "little") for i in range(count * n)]
        want = backend.msm_batch(_sb([v & (2 ** 255 - 1) for v in vals]), pts, n, count)
        d_sc = _to_dev(_sb(vals))
        d_out = torch.zeros(32 * count, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        backend._check(backend._lib.bpp_msm_vartime_batch_dev(backend._ctx, d_sc.data_ptr(), count, pts._h, 0, n,
                                                               d_out.data_ptr()))
        backend.synchronize()
        assert bytes(d_out.cpu().numpy().tobytes()) == want, count
    pts.free()


# ---------------------------------------------------------------------------------- the table MSM at its digit edge
def _top_digit(s, c):
    """Top digit of s + K for the fixed-base tables of width c (bpp_points_precompute's K)."""
    Wn = (256 + c - 1) // c
    K = sum(1 << (c * w + c - 1) for w in range(Wn - 1))
    return (s + K) >> (c * (Wn - 1)), K, Wn


def _edge_scalars(c):
    """2^255 - 1, which gives the largest top digit of any scalar below 2^255, the smallest scalar with that top digit,
    and 0, 1, l - 1."""
    top, K, Wn = _top_digit(2 ** 255 - 1, c)
    s = (top << (c * (Wn - 1))) - K
    assert 0 <= s < 2 ** 255 and _top_digit(s, c)[0] == top and _top_digit(s - 1, c)[0] == top - 1
    return [2 ** 255 - 1, s, 0, 1, L - 1]


def test_edge_scalars_reach_the_top_digit_bound():
    """The reference computation behind test_table_msm_at_the_digit_edge: below 2^255 the top digit of s + K never passes
    the table's 2^(c-1) rows and reaches them exactly where the top window is c bits wide (c = 4, 8, 16); elsewhere the
    top window is narrower and 2^255 - 1 gives its largest digit."""
    for c in range(4, 21):
        top = _top_digit(2 ** 255 - 1, c)[0]
        assert top <= 1 << (c - 1)
        assert (top == 1 << (c - 1)) == (256 % c == 0), c
        assert _top_digit(2 ** 255 + 2 ** 254, c)[0] > top     # bit 255 set: past what the table holds for c = 4, 8, 16


@pytest.mark.gpu
@pytest.mark.parametrize("c", list(range(4, 21)))
def test_table_msm_at_the_digit_edge(backend, c):
    """bpp_msm_vartime_batch over scalars with the largest top digit of s + K below 2^255 (_edge_scalars; exactly the
    table's 2^(c-1) rows at c = 4, 8, 16), at every table width, in the block form (3 MSMs) and the warp form (2400 MSMs), against the C oracle.
    Two points from c = 16 on: a table of c = 20 is 650 MB per point."""
    n = 2 if c >= 16 else 6
    rs = np.random.RandomState(40 + c)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8).tobytes()
    raw = cref.from_uniform(blobs)
    pts = backend.points_from_uniform(blobs)
    backend.precompute(pts, c)
    edge = _edge_scalars(c)
    for count in (3, 2400):
        vals = [edge[(i * 5 + i // n) % len(edge)] for i in range(count * n)]
        sc = _sb(vals)
        out = backend.msm_batch(sc, pts, n, count)
        for j in sorted({0, 1, 2, count // 2, count - 1}):
            assert out[32 * j:32 * j + 32] == cref.msm(sc[32 * n * j:32 * n * (j + 1)], raw), (c, count, j)
    pts.free()
