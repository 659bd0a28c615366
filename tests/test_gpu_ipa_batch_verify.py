"""Combined batch verification of the stand-alone inner-product argument (bpp_ipa_batch_verify_combined): proof for proof
the decisions of bpp_ipa_batch_verify and of a restatement of bulletproofs 4.0.0 InnerProductProof::verify, and
byte-identical transcripts, on all-valid batches and on batches with tampered proofs of every kind; on both sides of
the rule that sends small batches straight to the per-proof path (which side ran is read from the BPP_ACP_TRACE=1
stage line); decisions independent of the verifier seed; the weights bound to P and the proof index (two proofs that
differ only by P + D and P - D must not cancel); argument errors; and the batch sharded over two GPUs."""
import ctypes
import os
import random
import re
import socket

import numpy as np
import pytest

from oracle import cref, ipa
from oracle.merlin import Transcript as OTranscript

pytestmark = pytest.mark.gpu
L = 2 ** 252 + 27742317777372353535851937790883648493
TB = 208


def _sb(v):
    return b"".join(int(x % L).to_bytes(32, "little") for x in v)


def _ints(arr):
    return [int.from_bytes(r.tobytes(), "little") for r in arr]


class _Case:
    """count proofs of length n over G | H | Q (g_off 0, h_off n, q_off 2n) with random factors and q; proofs from the
    GPU prover, P = <a gf, G> + <b hf, H> + <a, b> q Q through the library's batched table MSM (the oracle re-checks a
    sample and every tampered proof)."""

    def __init__(self, be, count, n, seed):
        from bpperm_b200.ipa import InnerProductBatch, Transcript
        rs = np.random.RandomState(seed)
        self.be, self.count, self.n, self.lg = be, count, n, n.bit_length() - 1
        self.plen = 32 * (2 * self.lg + 2)
        blobs = rs.randint(0, 256, size=(2 * n + 1, 64), dtype=np.uint8).tobytes()
        self.pts = be.points_from_uniform(blobs)
        raw = cref.from_uniform(blobs)
        self.raw = [raw[cref.PT * i:cref.PT * (i + 1)] for i in range(2 * n + 1)]

        def sc(cnt):
            s = rs.randint(0, 256, size=(cnt, 32), dtype=np.uint8)
            s[:, 31] &= 0x0F
            return s
        a, b, gf, hf, q = sc(count * n), sc(count * n), sc(count * n), sc(count * n), sc(count)
        self.labels = [b"ipa-bv-%d" % (p % 13) for p in range(count)]
        bt = InnerProductBatch(be, self.pts, 0, n, 2 * n, n, count)
        self.proofs = bt.prove([Transcript(x) for x in self.labels], a.tobytes(), b.tobytes(), q.tobytes(), gf.tobytes(),
                               hf.tobytes())
        bt.free()
        ai, bi, gi, hi, self.q = _ints(a), _ints(b), _ints(gf), _ints(hf), _ints(q)
        self.gf = [gi[p * n:(p + 1) * n] for p in range(count)]
        self.hf = [hi[p * n:(p + 1) * n] for p in range(count)]
        msm = b""
        for p in range(count):
            av, bv = ai[p * n:(p + 1) * n], bi[p * n:(p + 1) * n]
            msm += _sb([x * f for x, f in zip(av, self.gf[p])] + [x * f for x, f in zip(bv, self.hf[p])] +
                       [sum(x * y for x, y in zip(av, bv)) % L * self.q[p]])
        Pb = be.msm_batch(msm, self.pts, 2 * n + 1, count)
        self.P = [Pb[32 * p:32 * p + 32] for p in range(count)]
        self.victims = {}

    def tamper(self, every=50, first=7, kinds=tuple(range(10))):
        """>= 1 % of the proofs, every kind of `kinds` in turn: 0-4 a, b, L_j, R_j, P flipped; 5 a + l; 6 all-zero L_j;
        7 undecodable R_j; 8 a wrong G factor; 9 a wrong H factor; 10 undecodable P.  5, 6, 7 and 10 are refused before
        any MSM."""
        pr = bytearray(self.proofs)
        lg, plen = self.lg, self.plen
        for k, p in enumerate(range(first, self.count, every)):
            kind, j, o = kinds[k % len(kinds)], k % lg, p * plen
            if kind == 0:
                pr[o + 32 * 2 * lg] ^= 1
            elif kind == 1:
                pr[o + 32 * (2 * lg + 1) + 3] ^= 1
            elif kind == 2:
                pr[o + 64 * j + 3] ^= 1
            elif kind == 3:
                pr[o + 64 * j + 32 + 5] ^= 1
            elif kind == 4:
                self.P[p] = bytes([self.P[p][0] ^ 2]) + self.P[p][1:]
            elif kind == 5:
                a = int.from_bytes(pr[o + 64 * lg:o + 64 * lg + 32], "little") + L
                pr[o + 64 * lg:o + 64 * lg + 32] = a.to_bytes(32, "little")
            elif kind == 6:
                pr[o + 64 * j:o + 64 * j + 32] = bytes(32)
            elif kind == 7:
                pr[o + 64 * j + 32:o + 64 * j + 64] = b"\xff" * 32
            elif kind == 8:
                self.gf[p] = [(self.gf[p][0] + 1) % L] + self.gf[p][1:]
            elif kind == 10:
                self.P[p] = b"\xff" * 32
            else:
                self.hf[p] = self.hf[p][:-1] + [(self.hf[p][-1] + 3) % L]
            self.victims[p] = kind
        self.proofs = bytes(pr)
        return self

    def args(self):
        return (b"".join(self.P), self.proofs, _sb(self.q), b"".join(_sb(g) for g in self.gf),
                b"".join(_sb(h) for h in self.hf))

    def states(self):
        from bpperm_b200.ipa import Transcript
        return b"".join(Transcript(x).state for x in self.labels)

    def oracle(self, p):
        """bulletproofs 4.0.0 InnerProductProof::from_bytes + verify on proof p (MSM in C); (decision, transcript)"""
        n, lg = self.n, self.lg
        pr = self.proofs[p * self.plen:(p + 1) * self.plen]
        w = [pr[32 * i:32 * i + 32] for i in range(2 * lg + 2)]
        a, b = int.from_bytes(w[-2], "little"), int.from_bytes(w[-1], "little")
        tr = OTranscript(self.labels[p])
        if a >= L or b >= L:
            return False, tr
        vs = ipa.InnerProductProof(w[0:2 * lg:2], w[1:2 * lg:2], a, b).verification_scalars(n, tr)
        if vs is None:
            return False, tr
        u_sq, u_inv_sq, s = vs
        try:
            pts = b"".join(self.raw) + cref.decompress(b"".join(w[:2 * lg:2]) + b"".join(w[1:2 * lg:2]))
            cref.decompress(self.P[p])
        except ValueError:
            return False, tr
        gf, hf = self.gf[p], self.hf[p]
        scal = _sb([a * s[i] * gf[i] for i in range(n)] + [b * s[n - 1 - i] * hf[i] for i in range(n)] +
                   [a * b * self.q[p]] + [-x for x in u_sq] + [-x for x in u_inv_sq])
        return cref.msm(scal, pts) == self.P[p], tr


def _both(be, case, seed=b"\x5a" * 32, traced=False, capfd=None):
    """bpp_ipa_batch_verify and bpp_ipa_batch_verify_combined on the same inputs through the C ABI: (accept, states) of
    each, and the stage names of the combined call's BPP_ACP_TRACE=1 line ("rlc-msm": the batch MSM ran; "check": the
    per-proof tail ran)"""
    from bpperm_b200.ipa import InnerProductBatch
    if traced:
        os.environ["BPP_ACP_TRACE"] = "1"
    try:
        bt = InnerProductBatch(be, case.pts, 0, case.n, 2 * case.n, case.n, case.count)
    finally:
        os.environ.pop("BPP_ACP_TRACE", None)
    P, proofs, q, gf, hf = case.args()
    lib = be._lib
    out = []
    for combined in (False, True):
        st = ctypes.create_string_buffer(case.states(), TB * case.count)
        acc = ctypes.create_string_buffer(case.count)
        if combined:
            be._check(lib.bpp_ipa_batch_verify_combined(bt._h, q, gf, hf, P, proofs, seed, st, acc))
        else:
            be._check(lib.bpp_ipa_batch_verify(bt._h, q, gf, hf, P, proofs, st, acc))
        out.append((acc.raw, st.raw))
    bt.free()
    stages = None
    if traced:
        err = capfd.readouterr().err
        line = [ln for ln in err.splitlines() if ln.startswith("[ipa trace] verify_combined:")][-1]
        stages = [name.strip() for name, _ in re.findall(r" ([^|:]+?) (\d+) us \|", line)]
    return out[0], out[1], stages


def _check_parity(case, v, c, sample=24):
    (acc_v, st_v), (acc_c, st_c) = v, c
    assert acc_c == acc_v
    assert st_c == st_v
    rs = random.Random(case.count * 31 + case.n)
    valid = [p for p in range(case.count) if p not in case.victims]
    for p in sorted(case.victims) + rs.sample(valid, min(sample, len(valid))):
        want, tr = case.oracle(p)
        assert acc_c[p] == int(want), (p, case.victims.get(p), acc_c[p])
        if want:   # the state left behind is dalek's
            from bpperm_b200.ipa import Transcript
            assert Transcript(state=st_c[TB * p:TB * (p + 1)]).challenge_bytes(b"after", 16) == tr.challenge_bytes(b"after", 16)
    for p in case.victims:
        assert acc_c[p] == 0, (p, case.victims[p])


@pytest.mark.parametrize("count,n,rlc", [(4096, 128, True), (4096, 8, True), (1, 8192, False), (68, 128, False), (69, 128, True)])
def test_decisions_and_transcripts_match_verify_and_the_oracle(backend, capfd, count, n, rlc):
    """(68, 128): 1020 proof points, below the 1024 of the per-proof rule; (69, 128): 1035, the batch MSM"""
    case = _Case(backend, count, n, 1000 + count + n)
    v, c, stages = _both(backend, case, traced=True, capfd=capfd)
    assert ("rlc-msm" in stages) == rlc and ("check" in stages) == (not rlc)
    assert c[0] == b"\x01" * count
    _check_parity(case, v, c)
    if count == 1:   # a batch of one: the proof itself tampered (b flipped)
        pr = bytearray(case.proofs)
        pr[32 * (2 * case.lg + 1) + 3] ^= 1
        case.proofs = bytes(pr)
        case.victims = {0: 1}
    else:
        case.tamper()
        assert len(case.victims) >= max(1, count // 100)
    v, c, stages = _both(backend, case, traced=True, capfd=capfd)
    assert ("rlc-msm" in stages) == rlc and "check" in stages
    _check_parity(case, v, c)


def test_decisions_do_not_depend_on_the_seed(backend):
    from bpperm_b200.ipa import InnerProductBatch, Transcript
    case = _Case(backend, 300, 8, 77).tamper(every=20, first=3)
    bt = InnerProductBatch(backend, case.pts, 0, 8, 16, 8, case.count)
    P, proofs, q, gf, hf = case.args()
    want = None
    for seed in (b"\x01" * 32, bytes(range(32)), None):
        trs = [Transcript(x) for x in case.labels]
        acc = bt.verify_combined(trs, P, proofs, q, gf, hf, verifier_seed=seed)
        if want is None:
            trv = [Transcript(x) for x in case.labels]
            want = bt.verify(trv, P, proofs, q, gf, hf)
            assert [t.state for t in trv] == [t.state for t in trs]
        assert acc == want, seed
    assert want.count(0) == len(case.victims) and all(want[p] == 0 for p in case.victims)
    with pytest.raises(ValueError):
        bt.verify_combined([Transcript(x) for x in case.labels], P, proofs, q, gf, hf, verifier_seed=b"short")


def test_two_copies_with_P_plus_and_minus_D_do_not_cancel(backend, capfd):
    """Proofs 10 and 11 are the bytes of proof 0 under its transcript, with P_0 + D and P_0 - D: both false, and with
    equal weights their errors +D and -D would cancel in the combination (a build with rho_p = 1 accepts both).  The
    weights bind P and the proof index, so the combination fails and the per-proof tail rejects exactly these two."""
    case = _Case(backend, 80, 128, 5)   # 80 x 15 proof points: the batch MSM runs
    plen = case.plen
    D = case.raw[3]   # G_3: not the identity
    P0 = cref.decompress(case.P[0])
    plus = cref.msm(_sb([1, 1]), P0 + D)
    minus = cref.msm(_sb([1, L - 1]), P0 + D)
    pr = bytearray(case.proofs)
    for p, Pp in ((10, plus), (11, minus)):
        pr[p * plen:(p + 1) * plen] = case.proofs[:plen]
        case.labels[p], case.q[p], case.gf[p], case.hf[p], case.P[p] = case.labels[0], case.q[0], case.gf[0], case.hf[0], Pp
        case.victims[p] = "P +- D"
    case.proofs = bytes(pr)
    v, c, stages = _both(backend, case, traced=True, capfd=capfd)
    assert "rlc-msm" in stages and "check" in stages
    assert c[0] == b"\x01" * 10 + b"\x00\x00" + b"\x01" * 68
    _check_parity(case, v, c, sample=4)


def test_refused_proofs_alone_leave_the_combination_at_the_identity(backend, capfd):
    """Bad proofs of the kinds refused before the MSM only (a + l, all-zero L_j, undecodable R_j, undecodable P): their
    weights are 0, the combination of the rest is the identity, and k_rlc_accept's bytes are final - the per-proof tail
    does not run - and equal verify's"""
    case = _Case(backend, 160, 8, 31).tamper(every=11, first=4, kinds=(5, 6, 7, 10))   # 160 x 7 proof points
    v, c, stages = _both(backend, case, traced=True, capfd=capfd)
    assert "rlc-msm" in stages and "check" not in stages
    assert c[0].count(0) == len(case.victims) >= 8
    _check_parity(case, v, c)


def test_weights_are_the_documented_construction(backend):
    """rho_p read back from the device equals a CPU restatement: proof p's transcript after verify, continued with
    "proof-tail" a || b, "P" P_p, "verifier-seed" seed, u64 "proof-index" p, then challenge scalar "rho".  Pins every
    input - P included, which no in-batch cancellation can (the index already separates two proofs of one batch)."""
    from bpperm_b200.ipa import InnerProductBatch, Transcript
    case = _Case(backend, 150, 8, 41)   # 150 x 7 proof points: the combined check runs
    bt = InnerProductBatch(backend, case.pts, 0, 8, 16, 8, case.count)
    seed = bytes(range(100, 132))
    assert bt.verify_combined([Transcript(x) for x in case.labels], *case.args(), verifier_seed=seed) == b"\x01" * case.count
    rho = ctypes.create_string_buffer(32 * case.count)
    backend._check(backend._lib.bpp_ipa_batch_download_weights(bt._h, rho))
    lg, plen = case.lg, case.plen
    for p in range(case.count):
        pr = case.proofs[p * plen:(p + 1) * plen]
        w = [pr[32 * i:32 * i + 32] for i in range(2 * lg + 2)]
        tr = OTranscript(case.labels[p])
        assert ipa.InnerProductProof(w[0:2 * lg:2], w[1:2 * lg:2], 0, 0).verification_scalars(case.n, tr) is not None
        tr.append_message(b"proof-tail", w[-2] + w[-1])
        tr.append_message(b"P", case.P[p])
        tr.append_message(b"verifier-seed", seed)
        tr.append_u64(b"proof-index", p)
        assert int.from_bytes(rho.raw[32 * p:32 * p + 32], "little") == tr.challenge_scalar(b"rho"), p
    bt2 = InnerProductBatch(backend, case.pts, 0, 8, 16, 8, case.count)
    assert backend._lib.bpp_ipa_batch_download_weights(bt2._h, rho) == -3   # no combined check yet


def test_argument_errors_match_verify_before_any_device_work(backend):
    from bpperm_b200.ipa import InnerProductBatch, Transcript
    case = _Case(backend, 2, 8, 9)
    bt = InnerProductBatch(backend, case.pts, 0, 8, 16, 8, 2)
    lib = backend._lib
    P, proofs, q, gf, hf = case.args()
    good = Transcript(b"t").state
    bad_state = good[:200] + (200).to_bytes(8, "little")
    big = _sb([1] * 15) + L.to_bytes(32, "little")
    calls = [
        dict(P=None), dict(proofs=None), dict(st=None), dict(acc=None), dict(st=bad_state + good),
        dict(q=_sb([1]) + (L + 5).to_bytes(32, "little")), dict(gf=big), dict(hf=big),
    ]
    for kw in calls:
        res = []
        for combined in (False, True):
            a = dict(P=P, proofs=proofs, q=q, gf=gf, hf=hf, st=good * 2, acc=b"")
            a.update(kw)
            st = None if a["st"] is None else ctypes.create_string_buffer(a["st"], TB * 2)
            acc = None if a["acc"] is None else ctypes.create_string_buffer(b"\x77\x77", 2)
            if combined:
                rc = lib.bpp_ipa_batch_verify_combined(bt._h, a["q"], a["gf"], a["hf"], a["P"], a["proofs"], None, st, acc)
            else:
                rc = lib.bpp_ipa_batch_verify(bt._h, a["q"], a["gf"], a["hf"], a["P"], a["proofs"], st, acc)
            if acc is not None:
                assert acc.raw == b"\x77\x77", kw.keys()    # nothing was written: no device work ran
            if st is not None:
                assert st.raw == a["st"], kw.keys()
            res.append(rc)
        assert res[0] == res[1] and res[0] in (-3, -6), (kw.keys(), res)
    assert lib.bpp_ipa_batch_verify_combined(None, None, None, None, P, proofs, None, None, None) == -3
    assert lib.bpp_ipa_batch_gather_accept(None, 4, ctypes.create_string_buffer(4)) == -3
    assert lib.bpp_ipa_batch_gather_accept(bt._h, 1, ctypes.create_string_buffer(4)) == -3   # per < count


def test_gather_accept_without_a_communicator_returns_this_ranks_bytes(backend):
    from bpperm_b200.ipa import InnerProductBatch, Transcript
    case = _Case(backend, 40, 8, 13).tamper(every=9, first=2)
    bt = InnerProductBatch(backend, case.pts, 0, 8, 16, 8, case.count)
    acc = bt.verify_combined([Transcript(x) for x in case.labels], *case.args())
    assert bt.gather_accept(48) == acc + bytes(8)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = {"rank": rank}
    try:
        import bpperm_b200
        from bpperm_b200.ipa import InnerProductBatch, Transcript
        par = bpperm_b200.parallel
        be = bpperm_b200.Backend(rank)
        par.init_comm(be, world, rank, torch.device("cuda", rank))
        total, n = 4096, 8
        case = _Case(be, total, n, 2024).tamper(every=37, first=5)   # the same global batch on every rank
        P, proofs, qq, gf, hf = case.args()
        whole = InnerProductBatch(be, case.pts, 0, n, 2 * n, n, total)
        want = whole.verify([Transcript(x) for x in case.labels], P, proofs, qq, gf, hf)
        whole.free()
        off, cnt = par.shard_bounds(total, world, rank)
        per = (total + world - 1) // world
        sl = lambda buf, w: buf[w * off:w * (off + cnt)]  # noqa: E731
        bt = InnerProductBatch(be, case.pts, 0, n, 2 * n, n, cnt)
        bt.verify_combined([Transcript(x) for x in case.labels[off:off + cnt]], sl(P, 32), sl(proofs, case.plen), sl(qq, 32),
                           sl(gf, 32 * n), sl(hf, 32 * n))
        allacc = bt.gather_accept(per)
        rebuilt = b"".join(allacc[per * r:per * r + par.shard_bounds(total, world, r)[1]] for r in range(world))
        res["ok"] = rebuilt == want and want.count(0) == len(case.victims)
        bt.free()
        be.close()
    except Exception:  # pragma: no cover
        import traceback
        res["error"] = traceback.format_exc()
    finally:
        q.put(res)
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_sharded_over_two_gpus_gathers_the_single_gpu_decisions():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=500) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for r in res:
        assert "error" not in r, r.get("error")
        assert r["ok"], r
