"""Mixed MSMs (bpp_msm_mixed*) on one GPU: µs per MSM for `count` MSMs of n_static generators (a tabled set, c = 8) plus
n_dyn caller points each, three ways, device-resident and host forms:
  mixed     one bpp_msm_mixed call
  multi     bpp_msm_multi over the same terms, the generators included as encodings (all variable-base)
  separate  bpp_msm_vartime_batch + bpp_msm_multi over the two parts, which give no combined result
Shapes: the verifier's 4096 x (209 + 8), the reference's sites :552-565 (210 + 3) and :525-533 (2 + 110) at 52 cards, a
stand-alone inner-product verify at n = 128 (257 + 15), and 16384 / 64 x (209 + 8), 4096 x (2 + 2).

Every timed window is a host clock around calls that end in a device synchronise, after one warm-up call of the same shape,
and holds at least --min-seconds of work.  The mixed results are checked against the all-variable-base call on every MSM.
The IMAD.WIDE-equivalents of each call come from bpp_last_op_counts, as tools/msm_multi_bench.py counts them.  The card
name, power limit and max SM clock are read with nvidia-smi in the same run and written beside the numbers.  --profile
adds per-kernel device times of the mixed call (torch.profiler, after the timed windows).

    python tools/msm_mixed_bench.py [--out profiles/r8_msm_mixed.json] [--min-seconds 1.0] [--profile]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from msm_multi_bench import W_ADD, W_DBL, W_MADD, W_SQRT, gpu_info, timed   # noqa: E402

SHAPES = [   # (label, count, n_static, n_dyn)
    ("verifier 209 + 8", 4096, 209, 8),
    ("circuit_lib.rs:552-565, 52 cards", 4096, 210, 3),
    ("circuit_lib.rs:525-533, 52 cards", 4096, 2, 110),
    ("inner-product verify n = 128", 4096, 257, 15),
    ("verifier 209 + 8", 16384, 209, 8),
    ("verifier 209 + 8", 64, 209, 8),
    ("tiny 2 + 2", 4096, 2, 2),
]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_msm_mixed.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--pool", type=int, default=1 << 16, help="distinct random points the dynamic terms draw from")
    ap.add_argument("--profile", action="store_true", help="per-kernel device times of the mixed call (torch.profiler)")
    args = ap.parse_args()
    import torch
    import bpperm_b200

    info = gpu_info()
    be = bpperm_b200.Backend(0)
    stream = torch.cuda.Stream()
    be.set_stream(stream.cuda_stream)
    sync = stream.synchronize
    limit = be.imad_pipe_limit()
    rs = np.random.RandomState(2026)
    n_gens = max(s[2] for s in SHAPES)
    gens = be.points_from_uniform(rs.randint(0, 256, size=(n_gens, 64), dtype=np.uint8).tobytes())
    be.precompute(gens, 8)
    gens_enc = np.frombuffer(be.compress_points(gens), dtype=np.uint8).reshape(-1, 32)
    pool = be.points_from_uniform(rs.randint(0, 256, size=(args.pool, 64), dtype=np.uint8).tobytes())
    pool_enc = np.frombuffer(be.compress_points(pool), dtype=np.uint8).reshape(-1, 32)
    dev = torch.device("cuda")

    def scalars(n):
        sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
        sc[:, 31] &= 0x0F   # below l's top byte: uniform-looking canonical scalars
        return sc

    def imad(ops, decodes, compresses):
        return (W_MADD * ops["mixed_adds"] + W_ADD * ops["full_adds"] + W_DBL * ops["doublings"] +
                W_SQRT * (decodes + compresses))

    results, prof_rows = [], []
    for label, count, n_s, n_d in SHAPES:
        st = scalars(count * n_s)
        dy = scalars(count * n_d)
        dy_enc = np.ascontiguousarray(pool_enc[rs.randint(0, args.pool, size=count * n_d)])
        # the all-variable-base form: per MSM its static terms (generators as encodings) then its dynamic terms
        all_sc = np.concatenate([st.reshape(count, n_s, 32), dy.reshape(count, n_d, 32)], axis=1).reshape(-1, 32)
        all_enc = np.concatenate([np.broadcast_to(gens_enc[:n_s], (count, n_s, 32)), dy_enc.reshape(count, n_d, 32)],
                                 axis=1).reshape(-1, 32)
        sizes, all_sizes = [n_d] * count, [n_s + n_d] * count
        with torch.cuda.stream(stream):
            d_st, d_dy, d_enc = (torch.from_numpy(x).to(dev) for x in (st, dy, dy_enc))
            d_all_sc, d_all_enc = torch.from_numpy(all_sc).to(dev), torch.from_numpy(np.ascontiguousarray(all_enc)).to(dev)
            d_out, d_out2, d_out3 = (torch.empty(32 * count, dtype=torch.uint8, device=dev) for _ in range(3))
            d_ok, d_ok2 = (torch.empty(count, dtype=torch.uint8, device=dev) for _ in range(2))
        sync()
        f_mixed = lambda: be.msm_mixed_dev(gens, n_s, d_st.data_ptr(), sizes, d_dy.data_ptr(), d_enc.data_ptr(), d_out.data_ptr(),
                                           d_ok.data_ptr())
        f_multi = lambda: be.msm_multi_dev(all_sizes, d_all_sc.data_ptr(), d_all_enc.data_ptr(), d_out2.data_ptr(), d_ok2.data_ptr())
        f_table = lambda: be._check(be._lib.bpp_msm_vartime_batch_dev(be._ctx, d_st.data_ptr(), count, gens._h, 0, n_s,
                                                                       d_out3.data_ptr()))
        f_dyn = lambda: be.msm_multi_dev(sizes, d_dy.data_ptr(), d_enc.data_ptr(), d_out2.data_ptr(), d_ok2.data_ptr())

        def f_separate():
            f_table()
            f_dyn()

        row = {"case": label, "count": count, "n_static": n_s, "n_dyn": n_d}
        dev_t = {}
        for name, f in (("mixed", f_mixed), ("multi", f_multi), ("separate", f_separate), ("separate_table", f_table),
                        ("separate_dynamic", f_dyn)):
            per_call, reps = timed(f, sync, args.min_seconds)
            dev_t[name] = per_call
            row[name] = {"dev_us_per_msm": per_call / count * 1e6, "dev_ms_per_call": per_call * 1e3, "reps": reps}
        # operation counts and the check, one call each
        f_multi()
        ops = be.last_op_counts()
        row["multi"].update(imad_fraction_of_limit=imad(ops, count * (n_s + n_d), count) / dev_t["multi"] / limit, op_counts=ops)
        f_mixed()
        ops = be.last_op_counts()
        row["mixed"].update(imad_fraction_of_limit=imad(ops, count * n_d, count) / dev_t["mixed"] / limit, op_counts=ops)
        sync()
        assert bytes(d_ok.cpu().numpy()) == b"\x01" * count and bytes(d_ok2.cpu().numpy()) == b"\x01" * count
        f_multi()
        sync()
        assert bytes(d_out.cpu().numpy()) == bytes(d_out2.cpu().numpy()), label
        # host forms
        stb, dyb, encb = st.tobytes(), dy.tobytes(), dy_enc.tobytes()
        allb, alle = all_sc.tobytes(), np.ascontiguousarray(all_enc).tobytes()
        hmin = min(args.min_seconds, 0.5)
        row["mixed"]["host_us_per_msm"] = timed(lambda: be.msm_mixed(stb, gens, n_s, dyb, encb, sizes), lambda: None, hmin)[0] / count * 1e6
        row["multi"]["host_us_per_msm"] = timed(lambda: be.msm_multi(allb, alle, all_sizes), lambda: None, hmin)[0] / count * 1e6
        row["separate"]["host_us_per_msm"] = timed(lambda: (be.msm_batch(stb, gens, n_s, count), be.msm_multi(dyb, encb, sizes)),
                                                   lambda: None, hmin)[0] / count * 1e6
        row["mixed_over_multi"] = dev_t["mixed"] / dev_t["multi"]
        row["mixed_minus_separate_us_per_call"] = (dev_t["mixed"] - dev_t["separate"]) * 1e6
        results.append(row)
        print(json.dumps(row), flush=True)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            f_mixed()
            sync()
            reps = 5
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    f_mixed()
                sync()
            kern = {}
            for e in prof.key_averages():
                if e.device_type is not None and "CUDA" in str(e.device_type) and e.count:
                    t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                    kern[e.key] = {"us_per_call": t / reps, "launches_per_call": e.count / reps}
            prof_rows.append({"case": label, "count": count, "n_static": n_s, "n_dyn": n_d, "kernels": kern})
            print(json.dumps(prof_rows[-1]), flush=True)
        del d_st, d_dy, d_enc, d_all_sc, d_all_enc

    out = {"gpu": info, "imad_pipe_limit_per_s": limit, "timing": "host clock around calls ending in a stream synchronise, "
           "after one warm-up call, >= %.1f s per device window (host forms: >= %.1f s)" % (args.min_seconds, min(args.min_seconds, 0.5)),
           "table_window_bits": 8, "results": results}
    if prof_rows:
        out["profile"] = {"how": "torch.profiler, CUDA activities, 5 mixed calls per shape after the timed windows",
                          "rows": prof_rows}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    be.close()


if __name__ == "__main__":
    main()
