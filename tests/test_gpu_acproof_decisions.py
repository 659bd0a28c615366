"""Accept bytes of the mode 0 / mode 1 batch verifier against a verifier that reads nothing but the proof bytes and the
commitments (cref.AcpInstance.verify: orc_acp_verify of oracle/c/acproof_ref.c, pinned to oracle.acproof's
verify_proof_bytes on the CPU).  Every expected decision below comes from that oracle.

- a tamper matrix over every field of a 5-card proof, RLC on and off, device and host transcripts, modes 1 and 0;
- the bench's shape: 52 cards, 4096 proofs, corruptions on warp, block and form boundaries; a second round whose only
  corruptions sit at 2048 or above, where the combined check alone decides; honest proofs byte-identical to the oracle;
- proofs of non-shuffles in a batch of the warp form;
- four lanes run as the bench runs them (own backend, urgent stream and host thread, shared generators and circuit,
  priority split, device-buffer witness, pinned staging), batches created from the lanes' threads;
- the witness kernels' clamp of out-of-range permutation indices.
Generators are tabled at c = 8: the same warp form of the table-gather MSM as the bench's c = 16, in 80 MB."""
import threading

import numpy as np
import pytest

from oracle import acproof as A, cref, ristretto255 as R

pytestmark = pytest.mark.gpu
L = R.L
OTHER_PT = R.compress(R.pt_mul(11, R.BASEPOINT))
INVALID_PT = b"\x01" + bytes(31)      # s odd: not a canonical non-negative field element
CORRUPT_AT = [0, 31, 32, 147, 148, 2047, 2048, 2367, 2368, 4095]   # warp, block (148 SMs) and form boundaries


def _sb(v):
    return b"".join(R.sc_bytes(s) for s in v)


def _field(pb, f):
    return int.from_bytes(pb[32 * f:32 * f + 32], "little")


def _put(pb, f, value):
    if isinstance(value, int):
        value = value.to_bytes(32, "little")
    return pb[:32 * f] + value + pb[32 * f + 32:]


def _flip(pb, f, bit):
    b = bytearray(pb)
    b[32 * f + bit // 8] ^= 1 << (bit % 8)
    return bytes(b)


class _Shuffle:
    """The k-card shuffle circuit over seeded generators: the library's (Circuit.shuffle, Generators) and the C
    oracle's dense instance over the same points."""

    def __init__(self, backend, k, c, seed):
        from bpperm_b200 import acproof as G
        n, Q, m, WL, WR, WO, WV, cv = A.shuffle_circuit(k)
        self.k, self.n, self.Q, self.m = k, n, Q, m
        rs = np.random.RandomState(seed)
        enc = cref.compress(cref.from_uniform(rs.randint(0, 256, size=(2 * n + 2, 64), dtype=np.uint8).tobytes()))
        self.pts = [enc[32 * i:32 * i + 32] for i in range(2 * n + 2)]

        def dense(M, rows):
            return b"".join(_sb(r) for r in A.dense(M, rows, Q))
        p = self.pts
        self.inst = cref.AcpInstance(n, Q, m, dense(WL, n), dense(WR, n), dense(WO, n), dense(WV, m), _sb(cv), p[0], p[1],
                                     b"".join(p[2:2 + n]), b"".join(p[2 + n:]))
        self.cir = G.Circuit.shuffle(backend, k)
        self.gens = self.new_gens(backend, c)

    def new_gens(self, backend, c):
        from bpperm_b200 import acproof as G
        p, n = self.pts, self.n
        return G.Generators(backend, p[0], p[1], p[2:2 + n], p[2 + n:], c)

    def verify(self, proof, V_enc, mode=1):
        """The oracle's decision: 1 accept, 0 reject."""
        return int(self.inst.verify(bytes(proof), None, mode, V_enc=bytes(V_enc)))

    def free(self):
        self.gens.free()
        self.cir.free()


_SHUFFLES = {}


def _shuffle(backend, k, c):
    if (k, c) not in _SHUFFLES:
        _SHUFFLES[(k, c)] = _Shuffle(backend, k, c, 5200 + k)
    return _SHUFFLES[(k, c)]


@pytest.fixture(scope="module", autouse=True)
def _free_shuffles():
    yield
    for s in _SHUFFLES.values():
        s.free()
    _SHUFFLES.clear()


def _inputs(k, B, seed):
    """What gen_shuffle_witness takes, as numpy arrays (bench.py synth_shuffle_inputs' shapes): deck 1..k."""
    rs = np.random.RandomState(seed)
    m = 2 * k + 1
    deck = list(range(1, k + 1))
    perm = np.stack([rs.permutation(k) for _ in range(B)]).astype(np.uint32)
    x = rs.randint(0, 256, size=(B, 32), dtype=np.uint8)
    x[:, 31] = 0
    gamma = rs.randint(0, 256, size=(B * m, 32), dtype=np.uint8)
    gamma[:, 31] &= 0x0F
    seeds = rs.randint(0, 256, size=(B, 32), dtype=np.uint8)
    return {"deck": deck, "perm": perm, "x": x, "gamma": gamma, "seeds": seeds}


def _witness(k, v):
    """a_L, a_R, a_O of the shuffle circuit for the values v = input deck | output deck | x (multiplication gates
    satisfied whatever v is; the linear constraints hold iff the output deck is a permutation of the input deck)."""
    n, x = 2 * k, v[-1]
    aL, aR, aO = [0] * n, [0] * n, [0] * n
    for gb, vb in ((0, 0), (k - 1, k)):
        for i in range(k - 1):
            aL[gb + i] = (v[vb] - x) % L if i == 0 else aO[gb + i - 1]
            aR[gb + i] = (v[vb + i + 1] - x) % L
            aO[gb + i] = aL[gb + i] * aR[gb + i] % L
    return aL, aR, aO


def _values(inp, p):
    deck = inp["deck"]
    return deck + [deck[j] for j in inp["perm"][p]] + [int.from_bytes(inp["x"][p].tobytes(), "little")]


def _prove(sh, backend, inp, B, mode=1):
    """gen_shuffle_witness -> commit(None) -> prove: (batch, V, proofs) as lists per proof."""
    from bpperm_b200 import acproof as G
    b = G.Batch(backend, sh.cir, sh.gens, B, mode)
    b.gen_shuffle_witness(_sb(inp["deck"]), inp["perm"].tobytes(), inp["x"].tobytes(), inp["gamma"].tobytes(),
                          inp["seeds"].tobytes())
    V = b.commit(None)
    b.prove()
    P = b.download_proofs()
    plen, vlen = b.proof_len, 32 * sh.m
    return b, [V[p * vlen:(p + 1) * vlen] for p in range(B)], [P[p * plen:(p + 1) * plen] for p in range(B)]


def _verify(b, proofs, Vs, seed=b"\x07" * 32, rlc=True, host=False):
    b.set_batch_rlc(rlc)
    b.set_host_transcripts(host)
    b.upload_proofs(b"".join(proofs), b"".join(Vs))
    b.verify(seed)
    return b.download_accept()


def _mismatch(got, want, idx, names=None):
    return [(p, names[p] if names else None, got[p], want[p]) for p in idx if got[p] != want[p]]


# ---------------------------------------------------------------------------------------------- tamper matrix
def _tamper_kinds(n):
    """(name, f(proof, V) -> (proof, V)): one corruption each, over every 32-byte field of the proof."""
    kinds = []
    for f in range(11 + 2 * n):
        kinds.append((f"flip{f}", lambda pb, V, f=f: (_flip(pb, f, (37 * f) % 255), V)))
        kinds.append((f"bit255_{f}", lambda pb, V, f=f: (_put(pb, f, _field(pb, f) | 1 << 255), V)))
        if f < 8:
            kinds.append((f"other{f}", lambda pb, V, f=f: (_put(pb, f, OTHER_PT), V)))
            kinds.append((f"identity{f}", lambda pb, V, f=f: (_put(pb, f, bytes(32)), V)))
            kinds.append((f"invalid{f}", lambda pb, V, f=f: (_put(pb, f, INVALID_PT), V)))
        else:
            kinds.append((f"plus1_{f}", lambda pb, V, f=f: (_put(pb, f, (_field(pb, f) + 1) % L), V)))
            kinds.append((f"plusl_{f}", lambda pb, V, f=f: (_put(pb, f, _field(pb, f) + L), V)))
    kinds.append(("swap_AI_AO", lambda pb, V: (pb[32:64] + pb[:32] + pb[64:], V)))
    kinds.append(("V0_other", lambda pb, V: (pb, OTHER_PT + V[32:])))
    kinds.append(("Vlast_other", lambda pb, V: (pb, V[:-32] + OTHER_PT)))
    kinds.append(("Vmid_invalid", lambda pb, V: (pb, V[:96] + INVALID_PT + V[128:])))
    return kinds


@pytest.mark.parametrize("mode", [1, 0], ids=["reference-fixed", "reference"])
def test_tamper_matrix_decisions_equal_the_oracle(backend, mode):
    k = 5
    sh = _shuffle(backend, k, 0)
    n = sh.n
    kinds = _tamper_kinds(n)
    K = len(kinds)
    B = K + 8          # + a V swap (2 proofs), one invalid proof twice (2), 4 honest proofs
    assert B >= 2 * (11 + 2 * n)
    inp = _inputs(k, B, 500 + mode)
    b, Vs, proofs = _prove(sh, backend, inp, B, mode)
    names = ["honest"] * B
    for i, (name, fn) in enumerate(kinds):
        proofs[i], Vs[i] = fn(proofs[i], Vs[i])
        names[i] = name
    Vs[K], Vs[K + 1] = Vs[K + 1], Vs[K]
    names[K] = names[K + 1] = "V_swapped"
    proofs[K + 2] = proofs[K + 3] = _put(proofs[K + 2], 9, (_field(proofs[K + 2], 9) + 1) % L)
    Vs[K + 3] = Vs[K + 2]
    names[K + 2] = names[K + 3] = "same_invalid_twice"
    want = bytes(sh.verify(proofs[p], Vs[p], mode) for p in range(B))
    accepted = {names[p] for p in range(B) if want[p]}
    if mode == 1:   # the oracle itself: s + l is s, everything else is a different proof
        assert accepted == {"honest"} | {f"plusl_{f}" for f in range(8, 11 + 2 * n)}
    else:           # the reference's verifier never accepts (circuit_lib.rs:541-544)
        assert accepted == set()
    for host in (False, True):
        for rlc in (True, False):
            got = _verify(b, proofs, Vs, rlc=rlc, host=host)
            assert got == want, (host, rlc, _mismatch(got, want, range(B), names))
    b.free()


# ---------------------------------------------------------------------------------------------- production shape
# corruptions that pass the verifier's cheap checks (decoding, t == <l, r>): only the MSM can reject them
_MSM_ONLY = [
    ("tau_x+1", lambda pb, V, n: (_put(pb, 8, (_field(pb, 8) + 1) % L), V)),
    ("mu+1", lambda pb, V, n: (_put(pb, 9, (_field(pb, 9) + 1) % L), V)),
    ("A_I_other", lambda pb, V, n: (_put(pb, 0, OTHER_PT), V)),
    ("S_other", lambda pb, V, n: (_put(pb, 2, OTHER_PT), V)),
    ("T4_other", lambda pb, V, n: (_put(pb, 5, OTHER_PT), V)),
    ("A_O_identity", lambda pb, V, n: (_put(pb, 1, bytes(32)), V)),
    ("V7_other", lambda pb, V, n: (pb, V[:224] + OTHER_PT + V[256:])),
    ("swap_AI_AO", lambda pb, V, n: (pb[32:64] + pb[:32] + pb[64:], V)),
]
_OTHERS = [
    ("T6_invalid", lambda pb, V, n: (_put(pb, 7, INVALID_PT), V)),
    ("t+1", lambda pb, V, n: (_put(pb, 10, (_field(pb, 10) + 1) % L), V)),
    ("r_last+1", lambda pb, V, n: (_put(pb, 10 + 2 * n, (_field(pb, 10 + 2 * n) + 1) % L), V)),
    ("mu+l", lambda pb, V, n: (_put(pb, 9, _field(pb, 9) + L), V)),          # accepted
    ("l0_bit255", lambda pb, V, n: (_put(pb, 11, _field(pb, 11) | 1 << 255), V)),
    ("V_last_invalid", lambda pb, V, n: (pb, V[:-32] + INVALID_PT)),
    ("flip_A_O", lambda pb, V, n: (_flip(pb, 1, 77), V)),
]


def _corrupt(proofs, Vs, where, kinds, n):
    names = {}
    for i, p in enumerate(where):
        name, fn = kinds[i % len(kinds)]
        proofs[p], Vs[p] = fn(proofs[p], Vs[p], n)
        names[p] = name
    return names


def test_production_shape_decisions_and_proof_bytes(backend):
    k, B = 52, 4096
    sh = _shuffle(backend, k, 8)
    n = sh.n
    inp = _inputs(k, B, 600)
    b, Vs, proofs = _prove(sh, backend, inp, B)
    rs = np.random.RandomState(601)
    extra = sorted(set(int(p) for p in rs.choice(B, 40, replace=False)) - set(CORRUPT_AT))[:31]
    where1 = CORRUPT_AT + extra                                         # 41 proofs, 1 %
    sample = sorted(set(int(p) for p in rs.choice(B, 60, replace=False)) - set(where1))[:24]
    # honest proofs of the device-generated witness: byte-identical to the oracle's prover on the same inputs
    for p in sample:
        v = _values(inp, p)
        aL, aR, aO = _witness(k, v)
        gam = inp["gamma"][p * sh.m:(p + 1) * sh.m].tobytes()
        pb, ok = sh.inst.prove_verify(_sb(aL), _sb(aR), _sb(aO), gam, cref.decompress(Vs[p]), inp["seeds"][p].tobytes(), 1,
                                      V_enc=Vs[p])
        assert ok == 1 and proofs[p] == pb, p
    honest = (list(proofs), list(Vs))
    # round 1: corruptions of every kind, on the boundaries
    names = _corrupt(proofs, Vs, where1, _MSM_ONLY + _OTHERS, n)
    want = {p: sh.verify(proofs[p], Vs[p]) for p in where1 + sample}
    assert all(want[p] == 1 for p in sample)
    assert {names[p] for p in where1 if want[p]} == {"mu+l"}
    for seed, rlc in ((b"\x11" * 32, True), (b"\x11" * 32, False), (None, True)):
        got = _verify(b, proofs, Vs, seed, rlc)
        assert _mismatch(got, want, sorted(want), names) == [], (seed, rlc)
        assert all(got[p] == 1 for p in range(B) if p not in want), (seed, rlc)
    # round 2: every corruption at 2048 or above and rejected only by the MSM, so that an all-accepting combined check
    # decides the batch on its own if it wrongly weighs them out
    proofs, Vs = list(honest[0]), list(honest[1])
    where2 = [2048, 2367, 2368, 4095] + sorted(set(int(p) for p in rs.choice(np.arange(2049, 4095), 30, replace=False))
                                             - {2367, 2368} - set(sample))[:12]
    names = _corrupt(proofs, Vs, where2, _MSM_ONLY, n)
    want = {p: sh.verify(proofs[p], Vs[p]) for p in where2}
    assert not any(want.values())
    want.update({p: 1 for p in sample})
    for seed, rlc in ((b"\x12" * 32, True), (b"\x12" * 32, False), (None, True)):
        got = _verify(b, proofs, Vs, seed, rlc)
        assert _mismatch(got, want, sorted(want), names) == [], (seed, rlc)
        assert all(got[p] == 1 for p in range(B) if p not in want), (seed, rlc)
    b.free()


# ---------------------------------------------------------------------------------------------- non-shuffles
def test_non_shuffles_are_rejected_beside_accepted_neighbours(backend):
    from bpperm_b200 import acproof as G
    k, B = 52, 2400
    sh = _shuffle(backend, k, 8)
    m = sh.m
    inp = _inputs(k, B, 700)
    DUP, WRONG_V, NOT_PERM = 5, 9, 2368
    honest_row = inp["perm"][DUP].copy()
    inp["perm"][DUP][1] = inp["perm"][DUP][0]               # a card twice, another missing
    b = G.Batch(backend, sh.cir, sh.gens, B)
    b.gen_shuffle_witness(_sb(inp["deck"]), inp["perm"].tobytes(), inp["x"].tobytes(), inp["gamma"].tobytes(),
                          inp["seeds"].tobytes())
    V = bytearray(b.commit(None))
    # WRONG_V: the witness is an honest shuffle, the commitments bound and checked are those of another deck
    v = _values(inp, WRONG_V)
    v[k + 3] = 1000
    gam = inp["gamma"][WRONG_V * m:(WRONG_V + 1) * m].tobytes()
    V[WRONG_V * 32 * m:(WRONG_V + 1) * 32 * m] = cref.compress(sh.inst.commit(_sb(v), gam))
    V = bytes(V)
    b.upload_commitments(V)
    b.prove()
    P = b.download_proofs()
    b.upload_proofs(P, V)
    b.verify(b"\x21" * 32)
    got = b.download_accept()
    plen, vlen = b.proof_len, 32 * m
    for p in (DUP - 1, DUP, DUP + 1, WRONG_V - 1, WRONG_V, WRONG_V + 1):
        assert got[p] == sh.verify(P[p * plen:(p + 1) * plen], V[p * vlen:(p + 1) * vlen]) == (p not in (DUP, WRONG_V)), p
    assert got == bytes(0 if p in (DUP, WRONG_V) else 1 for p in range(B))
    # NOT_PERM: an uploaded witness whose multiplication gates all hold but whose output deck is not a permutation
    vals = [_values(inp, p) for p in range(B)]
    vals[DUP] = _values(dict(inp, perm={DUP: honest_row}), DUP)   # the honest permutation of the round above
    vals[NOT_PERM][k] = (vals[NOT_PERM][k] + 1) % L
    wit = [_witness(k, v) for v in vals]
    aO = wit[NOT_PERM][2]
    assert all(a * r % L == o for a, r, o in zip(*wit[NOT_PERM]))
    assert aO[k - 2] != aO[2 * k - 3]                         # the two running products differ
    b.upload_witness(b"".join(_sb(w[0]) for w in wit), b"".join(_sb(w[1]) for w in wit), b"".join(_sb(w[2]) for w in wit),
                     inp["gamma"].tobytes(), inp["seeds"].tobytes())
    V2 = b.commit(b"".join(_sb(v) for v in vals))
    b.prove()
    P2 = b.download_proofs()
    b.upload_proofs(P2, V2)
    b.verify(b"\x22" * 32)
    got = b.download_accept()
    for p in (NOT_PERM - 1, NOT_PERM, NOT_PERM + 1):
        assert got[p] == sh.verify(P2[p * plen:(p + 1) * plen], V2[p * vlen:(p + 1) * vlen]) == (p != NOT_PERM), p
    assert got == bytes(0 if p == NOT_PERM else 1 for p in range(B))
    b.free()


# ---------------------------------------------------------------------------------------------- lanes
_LANE_KINDS = _MSM_ONLY[:5] + [_OTHERS[1]]


@pytest.mark.parametrize("late", [False, True], ids=["decompress-forked-early", "decompress-late"])
def test_lanes_as_the_bench_runs_them(backend, monkeypatch, late):
    """4 lanes x 2400 proofs (warp form and H_sum: >= 16 proofs per SM), 3 rounds.  Proof bytes must equal the same
    inputs proved alone on the session backend without the priority split; accept bytes must equal the oracle's
    decisions (the corrupted proof and its neighbours against the oracle, every other proof's bytes equal to the lone
    run's, which the production-shape test pins to the oracle's prover)."""
    import torch
    import bpperm_b200
    from bpperm_b200 import acproof as G
    if late:
        monkeypatch.setenv("BPP_DECOMPRESS_LATE", "1")
    else:
        monkeypatch.delenv("BPP_DECOMPRESS_LATE", raising=False)
    k, B, NL, ROUNDS = 52, 2400, 4, 3
    sh = _shuffle(backend, k, 8)
    n, m = sh.n, sh.m
    plen, vlen = G.proof_len(n), 32 * m
    sets = [[_inputs(k, B, 800 + 10 * ln + r + 100 * late) for r in range(ROUNDS)] for ln in range(NL)]
    # the same inputs alone on the session backend (its generators are another set over the same points)
    ref = G.Batch(backend, sh.cir, sh.gens, B)
    refP, refV = {}, {}
    for ln in range(NL):
        for r in range(ROUNDS):
            inp = sets[ln][r]
            ref.gen_shuffle_witness(_sb(inp["deck"]), inp["perm"].tobytes(), inp["x"].tobytes(), inp["gamma"].tobytes(),
                                    inp["seeds"].tobytes())
            refV[ln, r] = ref.commit(None)
            ref.prove()
            refP[ln, r] = ref.download_proofs()
    ref.free()
    dev = torch.device("cuda", 0)

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).pin_memory()
    d_deck = pin(np.frombuffer(_sb(sets[0][0]["deck"]), dtype=np.uint8)).to(dev)
    dsets = {}
    for ln in range(NL):
        for r in range(ROUNDS):
            inp = sets[ln][r]
            dsets[ln, r] = {kk: pin(inp[kk]).to(dev) for kk in ("perm", "x", "gamma", "seeds")}
            dsets[ln, r]["V"] = pin(np.frombuffer(refV[ln, r], dtype=np.uint8)).to(dev)
            dsets[ln, r]["hV"] = pin(np.frombuffer(refV[ln, r], dtype=np.uint8))
    torch.cuda.synchronize(dev)
    gens = sh.new_gens(backend, 8)    # fresh: its H_sum table is built by whichever lane's batch comes first
    lanes = []
    for ln in range(NL):
        st = torch.cuda.Stream(dev, priority=-1)
        be_l = bpperm_b200.Backend(0)
        be_l.set_stream(st.cuda_stream)
        lanes.append({"be": be_l, "stream": st, "proofs": torch.empty(B * plen, dtype=torch.uint8).pin_memory(),
                      "accept": torch.empty(B, dtype=torch.uint8).pin_memory(), "batch": None})
    where = {(ln, r): (997 * ln + 389 * r + 31) % B for ln in range(NL) for r in range(ROUNDS)}
    got_P, got_acc, sent, errors = {}, {}, {}, []
    barrier = threading.Barrier(NL)

    def lane(ln):
        try:
            L_ = lanes[ln]
            barrier.wait()
            bt = G.Batch(L_["be"], sh.cir, gens, B)
            L_["batch"] = bt
            bt.set_priority_split(True)
            hp, hp_np, ha = L_["proofs"], L_["proofs"].numpy(), L_["accept"]
            for r in range(ROUNDS):
                d = dsets[ln, r]
                bt.gen_shuffle_witness(d_deck.data_ptr(), d["perm"].data_ptr(), d["x"].data_ptr(), d["gamma"].data_ptr(),
                                       d["seeds"].data_ptr())
                bt.upload_commitments(d["V"].data_ptr())
                bt.prove()
                bt.download_proofs_ptr(hp.data_ptr())
                got_P[ln, r] = hp_np.tobytes()
                p = where[ln, r]
                pb, _ = _LANE_KINDS[(ln * ROUNDS + r) % len(_LANE_KINDS)][1](got_P[ln, r][p * plen:(p + 1) * plen], None, n)
                hp_np[p * plen:(p + 1) * plen] = np.frombuffer(pb, dtype=np.uint8)
                sent[ln, r] = pb
                bt.upload_proofs_ptr(hp.data_ptr(), d["hV"].data_ptr())
                bt.verify(None)
                bt.download_accept_ptr(ha.data_ptr())
                L_["be"].synchronize()
                got_acc[ln, r] = ha.numpy().tobytes()
        except BaseException as e:   # reported from the main thread
            errors.append((ln, repr(e)))
            barrier.abort()

    threads = [threading.Thread(target=lane, args=(ln,)) for ln in range(NL)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for L_ in lanes:
        if L_["batch"] is not None:
            L_["batch"].free()
        L_["be"].close()
    gens.free()
    assert not errors, errors
    for ln in range(NL):
        for r in range(ROUNDS):
            assert got_P[ln, r] == refP[ln, r], (ln, r)
            p = where[ln, r]
            V = refV[ln, r]
            want = {p: sh.verify(sent[ln, r], V[p * vlen:(p + 1) * vlen])}
            for q in ((p - 1) % B, (p + 1) % B):
                want[q] = sh.verify(refP[ln, r][q * plen:(q + 1) * plen], V[q * vlen:(q + 1) * vlen])
            assert want[p] == 0 and want[(p + 1) % B] == 1
            acc = got_acc[ln, r]
            assert {q: acc[q] for q in want} == want, (ln, r)
            assert acc == bytes(0 if q == p else 1 for q in range(B)), (ln, r)


# ---------------------------------------------------------------------------------------------- the witness clamp
@pytest.mark.parametrize("k", [5, 70], ids=["thread-per-chain", "block-scan"])
def test_witness_clamps_out_of_range_indices(backend, k):
    """perm indices k, k + 1 and k + B - 1: still inside the batch's own staging buffer (gamma | deck | x | perm), read
    as the deck's last card.  The proofs of such witnesses are not shuffles and are rejected."""
    from bpperm_b200 import acproof as G
    B = 4
    sh = _shuffle(backend, k, 0)
    m = sh.m
    inp = _inputs(k, B, 900 + k)
    for p, j, idx in ((1, 0, k), (2, 3, k + 1), (3, k - 1, k + B - 1)):
        if inp["perm"][p][j] == k - 1:     # clamped onto the card it replaces, it would still be a permutation
            j = (j + 1) % k
        inp["perm"][p][j] = idx
    b = G.Batch(backend, sh.cir, sh.gens, B)
    b.gen_shuffle_witness(_sb(inp["deck"]), inp["perm"].tobytes(), inp["x"].tobytes(), inp["gamma"].tobytes(),
                          inp["seeds"].tobytes())
    V = b.commit(None)
    clamped = dict(inp, perm=np.minimum(inp["perm"], k - 1))
    want_V = b"".join(cref.compress(sh.inst.commit(_sb(_values(clamped, p)), inp["gamma"][p * m:(p + 1) * m].tobytes()))
                      for p in range(B))
    assert V == want_V
    b.prove()
    P = b.download_proofs()
    b.upload_proofs(P, V)
    b.verify(b"\x31" * 32)
    got = b.download_accept()
    plen, vlen = b.proof_len, 32 * m
    want = bytes(sh.verify(P[p * plen:(p + 1) * plen], V[p * vlen:(p + 1) * vlen]) for p in range(B))
    assert want == b"\x01\x00\x00\x00" and got == want
    b.free()
