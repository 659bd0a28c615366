"""Per-kernel profile of bench.py's flagship step: the 52-card shuffle prove + verify, B = 4096 proofs per step, c = 16
tables, mode reference-fixed, the same seeded inputs as bench_shuffle (four rotating input sets, witness generated on the
device, verifier weights from the OS RNG).

Two runs of their own under torch.profiler (CUDA activities): one batch at a time on one stream, where a kernel's time is
its time alone, and `--lanes` batches in flight on as many streams (bench.py's headline shape), where kernels of
different lanes share the SMs.  For each kernel: device time per step, launches per step and, for the scalar kernels,
the bytes each reads and writes and the scalar products mod l the formula needs (both per proof, from the code: MODEL
below), set against the time as GB/s and as a share of the multiplier ceiling (0.71 of the IMAD.WIDE issue limit,
136 IMAD.WIDE per product; DESIGN.md section 1).  The card's name, power limit and clocks are read in the same call.

    python tools/scalar_profile.py --out /tmp/scalar_profile.json [--steps 12] [--lanes 6] [--form parent]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402

SC = 32                     # bytes per scalar
SC_MUL_IMAD = bench.SC_MUL_IMAD
CEILING = 0.71              # measured IMAD.WIDE share of the point kernels (DESIGN.md sections 1, 3.2)


def model(n, Q, m, form):
    """Per proof and step (one prove + one verify): kernel -> (scalars read, scalars written, products needed).
    Products: scalar multiplications mod l the formulas need (a dot of length n needs n, a Horner step one); format
    conversions and reductions are the kernels' own cost and are not counted.  Scalars: 32-byte fields of the proof
    block touched per proof (per-proof constants read by every thread count once).  form: 'change' = this tree's
    kernels, 'parent' = the kernels before the r7 scalar rewrite."""
    per = m + 8
    mdl = {
        # three Fibonacci power chains (y, z, y^-1) per proof, prover and verifier
        "k_acp_pow": (2 * 2, 2 * (2 * n + Q), 2 * (2 * n + Q)),
        # z*W rows: O(nnz) additions of z_q entries
        "k_acp_csr": (2 * 4 * n, 2 * (3 * n + m + 1), 0),
        # prover: 10 dots of length n, then <l, r> (n) and <zWV, gamma> (m); verifier: sigma and <l, r>
        "k_acp_dots_warp": (20 * n + 2 * n + 2 * m + 4 * n, 12 + 2, 10 * n + n + m + 2 * n),
        "k_acp_tcoef": (10, 12, 0),
        # l(x), r(x): three products each by Horner
        "k_acp_final": (6 * n + 1, 2 * n, 6 * n),
        "k_acp_final2": (17, 3, 15),
        # G: w (x lin - l), H: w y^-i (x zWL + zWO - y^i - r), V: -x^2 zWV, the few per-proof scalars
        "k_acp_vscal": (7 * n + m + 10, 2 * n + m + 10, 5 * n + m + 14),
        "k_rlc_weights": (3, 1, 0),
        "k_rlc_dyn_scalars": (per + 1, per, per),
        "k_rlc_stat_scalars": (2 * (2 * n + 2), 0, 2 * n + 2),
    }
    if form == "parent":
        mdl["k_acp_pow_unmont"] = (2 * (2 * n + Q), 2 * (2 * n + Q), 0)
        # prover and verifier alike: lin, l1, r0, r1, r3 from 8 inputs (the verifier uses lin only)
        mdl["k_acp_vec1"] = (2 * 8 * n, 2 * 5 * n, 4 * n)
    else:
        mdl["k_acp_pow_unmont"] = (2 * Q, 2 * Q, 0)                        # z_q only
        mdl["k_acp_vec1<true, true>"] = (8 * n, 7 * n, 3 * n)                   # prover: + y^i, y^-i out of Montgomery form
        mdl["k_acp_vec1<false, true>"] = (3 * n, 3 * n, n)                      # verifier: lin, y^i, y^-i
    return mdl


def gpu_info():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm"
        return subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], text=True).strip().splitlines()[0]
    except Exception as e:   # the numbers below still stand; the record says why the card is not named
        return f"nvidia-smi failed: {e}"


def short_name(key):
    name = key.split("(")[0].strip()
    if name.startswith("void "):
        name = name[5:]
    return name


def kernel_table(prof, steps):
    rows = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", None)
        if t is None:
            t = e.self_cuda_time_total
        if t <= 0:
            continue
        k = short_name(e.key)
        r = rows.setdefault(k, {"us_per_step": 0.0, "launches_per_step": 0.0})
        r["us_per_step"] += t / steps
        r["launches_per_step"] += e.count / steps
    return dict(sorted(rows.items(), key=lambda kv: -kv[1]["us_per_step"]))


def annotate(rows, mdl, B, products_per_us_ceiling):
    for k, r in rows.items():
        base = re.sub(r"<.*", "", k)
        key = k if k in mdl else (base if base in mdl else None)
        if key is None:
            continue
        rd, wr, prod = mdl[key]
        us = r["us_per_step"]
        r["bytes_per_step"] = B * (rd + wr) * SC
        r["gb_per_s"] = r["bytes_per_step"] / (us * 1e3)
        r["products_per_step"] = B * prod
        r["products_per_us"] = B * prod / us
        r["frac_of_ceiling"] = (B * prod / us) / products_per_us_ceiling if prod else 0.0
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--lanes", type=int, default=6)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--form", choices=("change", "parent"), default="change", help="which kernels' byte model applies")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bpperm_b200
    G = bpperm_b200.acproof
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    be = bpperm_b200.Backend(0)
    stream = torch.cuda.current_stream(dev)
    be.set_stream(stream.cuda_stream)
    k, B, mode = bench.K_CARDS, args.batch, "reference-fixed"
    cir, gens, enc, (n, Q, m, ng), _ = bench.shuffle_setup_mode(be, k, mode, 16)
    N_SETS = 4
    sets = [bench.synth_shuffle_inputs(k, B, 0, s) for s in range(N_SETS)]
    d_deck = torch.from_numpy(np.ascontiguousarray(sets[0][0])).to(dev)
    ds = [{kk: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for kk, v in zip(("perm", "x", "gamma", "seeds"), s[1:])}
          for s in sets]
    batch = G.Batch(be, cir, gens, B, mode, b"test")
    for s_i in range(N_SETS):
        d = ds[s_i]
        batch.gen_shuffle_witness(d_deck.data_ptr(), d["perm"].data_ptr(), d["x"].data_ptr(), d["gamma"].data_ptr(), d["seeds"].data_ptr())
        d["V"] = torch.from_numpy(np.frombuffer(batch.commit(None), dtype=np.uint8).copy()).to(dev)

    def step(bt, i):
        d = ds[i % N_SETS]
        bt.gen_shuffle_witness(d_deck.data_ptr(), d["perm"].data_ptr(), d["x"].data_ptr(), d["gamma"].data_ptr(), d["seeds"].data_ptr())
        bt.upload_commitments(d["V"].data_ptr())
        bt.prove()
        bt.verify(None)

    lanes = []
    for _ in range(args.lanes):
        st = torch.cuda.Stream(dev, priority=-1)
        be_l = bpperm_b200.Backend(0)
        be_l.set_stream(st.cuda_stream)
        b_l = G.Batch(be_l, cir, gens, B, mode, b"test")
        b_l.set_priority_split(True)
        lanes.append({"stream": st, "be": be_l, "batch": b_l})

    def run_lanes(cnt, first):
        def body(ln, idx):
            for i in idx:
                step(ln["batch"], i)
        th = [threading.Thread(target=body, args=(lanes[j], [first + t for t in range(cnt) if t % args.lanes == j]))
              for j in range(args.lanes)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        torch.cuda.synchronize()

    def run_single(cnt, first):
        for i in range(cnt):
            step(batch, first + i)
        torch.cuda.synchronize()

    peak = be.imad_pipe_limit()
    ceiling_per_us = CEILING * peak / SC_MUL_IMAD / 1e6
    mdl = model(n, Q, m, args.form)
    out = {"gpu": gpu_info(), "form": args.form, "batch": B, "k": k, "n": n, "Q": Q, "m": m, "steps": args.steps,
           "imad_peak_per_s": peak, "ceiling": {"share_of_imad_issue_limit": CEILING, "imad_per_product": SC_MUL_IMAD,
                                                "products_per_us": ceiling_per_us}}
    for name, run in (("single_stream", run_single), ("lanes", run_lanes)):
        run(args.warmup, 0)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        run(args.steps, args.warmup)                 # unprofiled: the step time the profile is set against
        ev1.record(stream)
        torch.cuda.synchronize()
        wall = ev0.elapsed_time(ev1) / args.steps
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(args.steps, args.warmup)
        rows = annotate(kernel_table(prof, args.steps), mdl, B, ceiling_per_us)
        scalar = {kk: r for kk, r in rows.items() if "products_per_step" in r}
        out[name] = {"ms_per_step_unprofiled": wall,
                     "scalar_kernels_us_per_step": sum(r["us_per_step"] for r in scalar.values()),
                     "all_kernels_us_per_step": sum(r["us_per_step"] for r in rows.values()),
                     "kernels": rows}
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for name in ("single_stream", "lanes"):
        print(f"{name}: {out[name]['ms_per_step_unprofiled']:.3f} ms/step, scalar kernels {out[name]['scalar_kernels_us_per_step']:.0f} us/step")
        for kk, r in list(out[name]["kernels"].items())[:40]:
            extra = f" {r['gb_per_s']:7.0f} GB/s {r['frac_of_ceiling']:.3f} of ceiling" if "gb_per_s" in r else ""
            print(f"  {kk:40s} {r['us_per_step']:9.1f} us x{r['launches_per_step']:.0f}{extra}")
    for ln in lanes:
        ln["batch"].free()
        ln["be"].close()
    batch.free()
    gens.free()
    cir.free()


if __name__ == "__main__":
    main()
