"""Batched variable-base MSM (bpp_msm_multi*) on one GPU: µs per MSM, device-resident and host forms, beside the looped
trait call (bpp_msm_vartime_host) and the table path over a shared set (bpp_msm_vartime_batch), for
count in {64, 4096, 16384} x n in {2, 105, 209, 1024} and the ragged 52-card verifier mix, both point forms.

Every timed window is a host clock around calls that end in a device synchronise, after one warm-up call of the same shape,
and holds at least --min-seconds of work.  Outputs are checked against bpp_msm_vartime on a sample of each batch.  The card
name, power limit and max SM clock are read with nvidia-smi in the same run and written beside the numbers.

    python tools/msm_multi_bench.py [--out profiles/r5_msm_multi.json] [--min-seconds 1.0]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# IMAD.WIDE-equivalents per operation (SURVEY.md 8(d)): mixed add 7M, full add 9M, doubling 4S + 4M; a decode or a
# compress is dominated by one inverse square root (x^((p-5)/8): 250 S + 11 M) plus ~15 M around it
M, S = 72, 44
W_MADD, W_ADD, W_DBL, W_SQRT = 7 * M, 9 * M, 4 * S + 4 * M, 250 * S + 26 * M


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def timed(fn, sync, min_s):
    fn()
    sync()
    reps, t0 = 0, time.perf_counter()
    while True:
        fn()
        reps += 1
        if reps >= 3 and time.perf_counter() - t0 >= min_s:
            sync()
            el = time.perf_counter() - t0
            if el >= min_s:
                return el / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_msm_multi.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--pool", type=int, default=1 << 16, help="distinct random points the MSMs draw from")
    args = ap.parse_args()
    import torch
    import bpperm_b200

    info = gpu_info()
    be = bpperm_b200.Backend(0)
    stream = torch.cuda.Stream()
    be.set_stream(stream.cuda_stream)
    sync = stream.synchronize
    limit = be.imad_pipe_limit()
    rs = np.random.RandomState(2025)
    pool = be.points_from_uniform(rs.randint(0, 256, size=(args.pool, 64), dtype=np.uint8).tobytes())
    pool_enc = np.frombuffer(be.compress_points(pool), dtype=np.uint8).reshape(-1, 32)
    dev = torch.device("cuda")

    def inputs(sizes):
        T = int(sum(sizes))
        sc = rs.randint(0, 256, size=(T, 32), dtype=np.uint8)
        sc[:, 31] &= 0x0F   # below l's top byte: uniform-looking canonical scalars
        ix = rs.randint(0, args.pool, size=T).astype(np.uint32)
        return sc, ix, pool_enc[ix]

    results = []

    def run(label, sizes, check=4):
        sizes = [int(x) for x in sizes]
        count, T = len(sizes), int(sum(sizes))
        sc, ix, enc = inputs(sizes)
        with torch.cuda.stream(stream):
            d_sc = torch.from_numpy(sc).to(dev)
            d_enc = torch.from_numpy(np.ascontiguousarray(enc)).to(dev)
            d_ix = torch.from_numpy(ix.view(np.int32)).to(dev)
            d_out = torch.empty(32 * count, dtype=torch.uint8, device=dev)
            d_ok = torch.empty(count, dtype=torch.uint8, device=dev)
        sync()
        row = {"case": label, "count": count, "terms": T}
        for form in ("encoded", "indexed"):
            if form == "encoded":
                f = lambda: be.msm_multi_dev(sizes, d_sc.data_ptr(), d_enc.data_ptr(), d_out.data_ptr(), d_ok.data_ptr())
            else:
                f = lambda: be.msm_multi_indexed_dev(sizes, d_sc.data_ptr(), pool, d_ix.data_ptr(), d_out.data_ptr())
            per_call, reps = timed(f, sync, args.min_seconds)
            ops = be.last_op_counts()
            decodes = T if form == "encoded" else 0
            imad = (W_MADD * ops["mixed_adds"] + W_ADD * ops["full_adds"] + W_DBL * ops["doublings"] +
                    W_SQRT * (decodes + count))
            got = bytes(d_out.cpu().numpy())
            if form == "encoded":
                assert bytes(d_ok.cpu().numpy()) == b"\x01" * count
            # a sample against the single-MSM path
            starts = np.concatenate([[0], np.cumsum(sizes)])
            for j in sorted(set(np.linspace(0, count - 1, min(check, count)).astype(int).tolist())):
                a, b = int(starts[j]), int(starts[j + 1])
                want = be.vartime_multiscalar_mul(sc[a:b].tobytes(), enc[a:b].tobytes()) if b > a else bytes(32)
                assert got[32 * j:32 * j + 32] == want, (label, form, j)
            sb, eb = sc.tobytes(), enc.tobytes()
            if form == "encoded":
                h = lambda: be.msm_multi(sb, eb, sizes)
            else:
                h = lambda: be.msm_multi_indexed(sb, pool, ix, sizes)
            host_call, _ = timed(h, lambda: None, min(args.min_seconds, 0.5))
            row[form] = {"dev_us_per_msm": per_call / count * 1e6, "dev_ms_per_call": per_call * 1e3, "reps": reps,
                         "host_us_per_msm": host_call / count * 1e6,
                         "imad_per_msm": imad / count, "imad_fraction_of_limit": imad / per_call / limit,
                         "op_counts": dict(ops, decodes=decodes, compresses=count)}
        results.append(row)
        print(json.dumps(row), flush=True)

    for count in (64, 4096, 16384):
        for n in (2, 105, 209, 1024):
            run(f"uniform n={n}", [n] * count)
    # one proof's dynamic-point verifier sites at 52 cards (circuit_lib.rs:525-533, :552-565, :498, :509), 4096 proofs
    run("52-card verifier mix", [111, 110, 104, 104] * 4096)
    # both sides of each size-class boundary (msm_multi_kernels.cuh), 4096 MSMs
    for n in (32, 33, 1024, 1025):
        run(f"boundary n={n}", [n] * 4096)

    # the looped trait call and the table path, same run
    refs = {}
    for n in (2, 105, 209, 1024):
        sc, ix, enc = inputs([n])
        sb, eb = sc.tobytes(), enc.tobytes()
        be.msm_host(sb, eb)
        t0 = time.perf_counter()
        for _ in range(5):
            be.msm_host(sb, eb)
        host_call = (time.perf_counter() - t0) / 5
        tab = be.upload_points(eb)
        be.precompute(tab)
        count = 4096
        sc4 = rs.randint(0, 256, size=(count * n, 32), dtype=np.uint8)
        sc4[:, 31] &= 0x0F
        d_sc4 = torch.from_numpy(sc4).to(dev)
        d_o = torch.empty(32 * count, dtype=torch.uint8, device=dev)
        sync()
        per_call, _ = timed(lambda: be._check(be._lib.bpp_msm_vartime_batch_dev(be._ctx, d_sc4.data_ptr(), count, tab._h, 0, n,
                                                                               d_o.data_ptr())), sync, args.min_seconds)
        refs[str(n)] = {"vartime_host_us_per_call": host_call * 1e6, "table_batch_us_per_msm_4096": per_call / count * 1e6}
        print(json.dumps({"n": n, **refs[str(n)]}), flush=True)
        tab.free()

    out = {"gpu": info, "imad_pipe_limit_per_s": limit, "timing": "host clock around calls ending in a stream synchronise, "
           "after one warm-up call, >= %.1f s per window" % args.min_seconds, "results": results, "references": refs}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    be.close()


if __name__ == "__main__":
    main()
