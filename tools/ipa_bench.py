"""Stand-alone inner-product batch (bpp_ipa_batch_*): prove and verify times at (count, n) = (4096, 128), (4096, 8) and
(1, 8192), beside the inner-product rounds of the `fixed` mode prover on the same padded shape (52, 4 and 4096 cards),
taken from its BPP_ACP_TRACE=1 stage timeline.  prove / verify: host clock around the C calls, which end in a device
synchronisation (host input checks, pageable uploads and downloads included), after a warm-up; stage_median_ms: the
batch's own BPP_ACP_TRACE=1 timeline (device events) in separate runs; verify_vs_combined: verify and verify_combined
alternating, host clock, on the all-valid batch and on one with ~1 % corrupted proofs.  Inputs seeded.  Writes one JSON
file (argv[1]) with the card name and power limit beside the numbers.
--scaling OUT.json: verify_combined of 4096 proofs of n = 128 in total, sharded over the ranks of
`python -m torch.distributed.run --nproc-per-node N` (strong scaling; see strong_scaling)."""
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, ".")
import bpperm_b200  # noqa: E402

L = 2 ** 252 + 27742317777372353535851937790883648493
SHAPES = [(4096, 128), (4096, 8), (1, 8192)]
REPS = int(os.environ.get("IPA_BENCH_REPS", "10"))


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      text=True).strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": "unknown", "error": str(e)}


def scalars(rs, cnt):
    s = rs.randint(0, 256, size=(cnt, 32), dtype=np.uint8)
    s[:, 31] &= 0x0F   # < 2^252 < l
    return s


def stderr_of(fn) -> str:
    """what the library prints to file descriptor 2 while fn runs (its BPP_ACP_TRACE=1 stage lines)"""
    with tempfile.TemporaryFile(mode="w+b") as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        return f.read().decode(errors="replace")


def timed(fn, reps):
    fn()   # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return {"median_ms": 1e3 * float(np.median(ts)), "min_ms": 1e3 * min(ts), "max_ms": 1e3 * max(ts), "reps": reps}


def ipa_shape(be, count, n, rs):
    Ipa = bpperm_b200.ipa
    pts = be.points_from_uniform(rs.randint(0, 256, size=(2 * n + 1, 64), dtype=np.uint8).tobytes())   # G | H | Q
    a, b = scalars(rs, count * n), scalars(rs, count * n)
    A = a.reshape(count, n, 32)
    Bv = b.reshape(count, n, 32)
    # P = <a, G> + <b, H> + <a, b> Q through the library's batched table MSM
    c = []
    for p in range(count):
        av = [int.from_bytes(A[p, i].tobytes(), "little") for i in range(n)]
        bv = [int.from_bytes(Bv[p, i].tobytes(), "little") for i in range(n)]
        c.append((sum(x * y for x, y in zip(av, bv)) % L).to_bytes(32, "little"))
    msm_sc = b"".join(A[p].tobytes() + Bv[p].tobytes() + c[p] for p in range(count))
    P = be.msm_batch(msm_sc, pts, 2 * n + 1, count)
    bt = Ipa.InnerProductBatch(be, pts, 0, n, 2 * n, n, count)
    states = Ipa.Transcript(b"ipa-bench").state * count
    st = ctypes.create_string_buffer(len(states))
    proofs = ctypes.create_string_buffer(bt.proof_len * count)
    acc = ctypes.create_string_buffer(count)
    ab, bb = a.tobytes(), b.tobytes()
    lib = be._lib

    def prove():   # the C call alone: the states are reset in place, nothing else is converted
        ctypes.memmove(st, states, len(states))
        be._check(lib.bpp_ipa_batch_prove(bt._h, None, None, None, ab, bb, st, proofs))

    def verify():
        ctypes.memmove(st, states, len(states))
        be._check(lib.bpp_ipa_batch_verify(bt._h, None, None, None, P, proofs.raw, st, acc))

    tp = timed(prove, REPS)
    tv = timed(verify, REPS)
    combined = verify_pair(be, bt, count, n, P, proofs.raw, states)
    # stage timeline (device events) in a run of its own: the rounds alone, comparable with the `fixed` prover's stage
    os.environ["BPP_ACP_TRACE"] = "1"
    bt2 = Ipa.InnerProductBatch(be, pts, 0, n, 2 * n, n, count)
    del os.environ["BPP_ACP_TRACE"]
    bt2_h = bt2._h

    def traced():
        for _ in range(REPS + 1):
            ctypes.memmove(st, states, len(states))
            be._check(lib.bpp_ipa_batch_prove(bt2_h, None, None, None, ab, bb, st, proofs))
            ctypes.memmove(st, states, len(states))
            be._check(lib.bpp_ipa_batch_verify(bt2_h, None, None, None, P, proofs.raw, st, acc))
    log = stderr_of(traced)
    bt2.free()
    stages = {}
    for what in ("prove", "verify"):
        lines = [ln for ln in log.splitlines() if ln.startswith(f"[ipa trace] {what}:")][1:]   # the first is the warm-up
        for ln in lines:
            for name, us in re.findall(r" ([^|:]+?) (\d+) us \|", ln):
                stages.setdefault(f"{what}: {name}", []).append(float(us))
    stage_ms = {k: float(np.median(v)) / 1e3 for k, v in stages.items()}
    row = {"count": count, "n": n, "proof_bytes": bt.proof_len, "prove": tp, "verify": tv,
           "all_accepted": acc.raw == b"\x01" * count, "stage_median_ms": stage_ms, "verify_vs_combined": combined}
    bt.free()
    pts.free()
    return row


def corrupt(proofs: bytes, count: int, plen: int, every: int = 97) -> (bytes, bytes):
    """about 1 % of the proofs (every 97th, and the only one of a batch of one) with one bit of b flipped; the expected
    accept bytes"""
    bad, expect = bytearray(proofs), bytearray(b"\x01" * count)
    for p in range(min(3, count - 1), count, every):
        bad[(p + 1) * plen - 29] ^= 0x04
        expect[p] = 0
    return bytes(bad), bytes(expect)


def verify_pair(be, bt, count, n, P, good, states):
    """verify and verify_combined side by side, alternating, on the all-valid batch and on the batch with ~1 %
    corrupted proofs (verifier seed from the OS, as a caller would run it)"""
    lib = be._lib
    st = ctypes.create_string_buffer(len(states))
    acc = ctypes.create_string_buffer(count)
    bad, expect = corrupt(good, count, bt.proof_len)
    out = {"corrupted": expect.count(0)}
    for key, proofs, want in (("all_valid", good, b"\x01" * count), ("corrupted_1pct", bad, expect)):
        def one(fn):
            def run():
                ctypes.memmove(st, states, len(states))
                if fn == "verify":
                    be._check(lib.bpp_ipa_batch_verify(bt._h, None, None, None, P, proofs, st, acc))
                else:
                    be._check(lib.bpp_ipa_batch_verify_combined(bt._h, None, None, None, P, proofs, None, st, acc))
                return acc.raw
            return run
        ts = {"verify": [], "verify_combined": []}
        ok = True
        for fn in ts:
            ok = ok and one(fn)() == want   # warm-up and decisions
        for _ in range(REPS):
            for fn in ts:
                run = one(fn)
                t0 = time.perf_counter()
                run()
                ts[fn].append(time.perf_counter() - t0)
        out[key] = {fn: {"median_ms": 1e3 * float(np.median(v)), "min_ms": 1e3 * min(v), "max_ms": 1e3 * max(v)}
                    for fn, v in ts.items()}
        out[key]["decisions_match_expected"] = ok
        out[key]["combined_over_verify"] = out[key]["verify_combined"]["median_ms"] / out[key]["verify"]["median_ms"]
    return out


def strong_scaling(total=4096, n=128, reps=REPS):
    """4096 proofs of n = 128 IN TOTAL sharded over the ranks (torch.distributed.run, one process per GPU; a plain run
    is one rank), as bench.py's batch_verify: every rank proves and verifies its slice (verify_combined, seed from the
    OS), the accept bytes are gathered over the library's NCCL communicator (InnerProductBatch.gather_accept).  Time
    per step: host clock from a barrier to the gathered bytes on every rank, median over reps; rank 0 returns it."""
    import torch
    import torch.distributed as dist
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    Ipa, par = bpperm_b200.ipa, bpperm_b200.parallel
    if world > 1:
        torch.cuda.set_device(rank)
        dist.init_process_group("gloo")
    be = bpperm_b200.Backend(rank)
    par.init_comm(be, world, rank, torch.device("cuda", rank))
    rs = np.random.RandomState(7)
    pts = be.points_from_uniform(rs.randint(0, 256, size=(2 * n + 1, 64), dtype=np.uint8).tobytes())
    a, b = scalars(rs, total * n), scalars(rs, total * n)   # the same global set on every rank
    off, cnt = par.shard_bounds(total, world, rank)
    per = (total + world - 1) // world
    A, Bv = a.reshape(total, n, 32)[off:off + cnt], b.reshape(total, n, 32)[off:off + cnt]
    c = []
    for p in range(cnt):
        av = [int.from_bytes(A[p, i].tobytes(), "little") for i in range(n)]
        bv = [int.from_bytes(Bv[p, i].tobytes(), "little") for i in range(n)]
        c.append((sum(x * y for x, y in zip(av, bv)) % L).to_bytes(32, "little"))
    P = be.msm_batch(b"".join(A[p].tobytes() + Bv[p].tobytes() + c[p] for p in range(cnt)), pts, 2 * n + 1, cnt)
    bt = Ipa.InnerProductBatch(be, pts, 0, n, 2 * n, n, cnt)
    states = Ipa.Transcript(b"ipa-bench").state * cnt
    st = ctypes.create_string_buffer(len(states))
    good = ctypes.create_string_buffer(bt.proof_len * cnt)
    be._check(be._lib.bpp_ipa_batch_prove(bt._h, None, None, None, A.tobytes(), Bv.tobytes(), st, good))
    # the corrupted proofs by global index: every 97th from 3
    bad, expect = bytearray(good.raw), bytearray(b"\x01" * cnt)
    for g in range(3, total, 97):
        if off <= g < off + cnt:
            bad[(g - off + 1) * bt.proof_len - 29] ^= 0x04
            expect[g - off] = 0
    acc = ctypes.create_string_buffer(cnt)
    res = {}
    for key, proofs in (("all_valid", good.raw), ("corrupted_1pct", bytes(bad))):
        ts, gathered = [], b""
        for i in range(reps + 1):
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            ctypes.memmove(st, states, len(states))
            be._check(be._lib.bpp_ipa_batch_verify_combined(bt._h, None, None, None, P, proofs, None, st, acc))
            gathered = bt.gather_accept(per)
            if i:
                ts.append(time.perf_counter() - t0)
        mine = gathered[per * rank:per * rank + cnt]
        res[key] = {"median_ms": 1e3 * float(np.median(ts)), "min_ms": 1e3 * min(ts), "max_ms": 1e3 * max(ts),
                    "proofs_per_s": total / float(np.median(ts)),
                    "decisions_match_expected": mine == (b"\x01" * cnt if key == "all_valid" else bytes(expect))}
    bt.free()
    pts.free()
    be.close()
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return None
    return {"n_gpus": world, "total": total, "n": n, "on_rank0": cnt, "reps": reps, "card": card(), **res}


def fixed_rounds(be, count, npad, rs):
    """median time of the `fixed` prover's "inner-product rounds" stage (BPP_ACP_TRACE=1) on count proofs of the
    shuffle whose n pads to npad"""
    G, W = bpperm_b200.acproof, bpperm_b200.weights
    k = {128: 52, 8: 4, 8192: 4096}[npad]
    n, Q, m, WL, WR, WO, WV, cv = W.shuffle_circuit(k)
    ng = G.next_pow2(n)
    pts = be.points_from_uniform(rs.randint(0, 256, size=(2 * ng + 2, 64), dtype=np.uint8).tobytes())
    enc = be.compress_points(pts)
    cir = G.Circuit(be, n, Q, m, WL, WR, WO, WV, cv)
    gens = G.Generators(be, enc[:32], enc[32:64], [enc[64 + 32 * i: 96 + 32 * i] for i in range(ng)],
                        [enc[64 + 32 * (ng + i): 96 + 32 * (ng + i)] for i in range(ng)])
    sb = lambda vals: b"".join(int(x).to_bytes(32, "little") for x in vals)  # noqa: E731
    v, a_L, a_R, a_O = W.shuffle_witness(k, rs.permutation(k), int.from_bytes(rs.bytes(31), "little"))
    os.environ["BPP_ACP_TRACE"] = "1"
    batch = G.Batch(be, cir, gens, count, "fixed", b"test")
    del os.environ["BPP_ACP_TRACE"]
    batch.upload_witness(sb(a_L) * count, sb(a_R) * count, sb(a_O) * count, scalars(rs, count * m).tobytes(),
                         rs.randint(0, 256, size=(count, 32), dtype=np.uint8).tobytes())
    batch.commit(sb(v) * count, want=False)
    def run():
        for _ in range(REPS + 1):
            batch.prove()
            be.synchronize()
    log = stderr_of(run)
    us = [float(x) for x in re.findall(r"inner-product rounds (\d+) us", log)][1:]   # the first prove is the warm-up
    batch.free()
    gens.free()
    cir.free()
    return {"cards": k, "padded_n": ng, "count": count, "rounds_median_ms": float(np.median(us)) / 1e3 if us else None,
            "samples": len(us)}


def main():
    if len(sys.argv) > 2 and sys.argv[1] == "--scaling":
        # python -m torch.distributed.run --nproc-per-node N tools/ipa_bench.py --scaling OUT.json
        row = strong_scaling()
        if row is not None:
            print(json.dumps(row), flush=True)
            os.makedirs(os.path.dirname(sys.argv[2]) or ".", exist_ok=True)
            json.dump(row, open(sys.argv[2], "w"), indent=1)
        return
    be = bpperm_b200.Backend(0)
    rs = np.random.RandomState(2026)
    res = {"card": card(), "reps": REPS, "rows": []}
    for count, n in SHAPES:
        row = ipa_shape(be, count, n, rs)
        row["fixed_mode_rounds"] = fixed_rounds(be, count, n, rs)
        fr = row["fixed_mode_rounds"]["rounds_median_ms"]
        own = row["stage_median_ms"].get("prove: inner-product rounds")
        row["rounds_over_fixed_rounds"] = own / fr if fr and own else None
        print(json.dumps(row), flush=True)
        res["rows"].append(row)
    out = sys.argv[1] if len(sys.argv) > 1 else "ipa_bench.json"
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    json.dump(res, open(out, "w"), indent=1)


if __name__ == "__main__":
    main()
