#!/usr/bin/env python
"""bench.py - headline benchmark of the B200 backend.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload shuffle|msm|both]
                    [--dump-outputs DIR]

BASELINE.json metric: "shuffle proofs/sec prove+verify (52-card); MSM points/sec at 2^20".
One "step" = one pass of the hot path over one batch of synthetic input.  Every leg's rate is timed over K steps (the
roofline's kernel timings and the pipe probes keep their own repetition counts).

--dump-outputs DIR: after the timed steps, the outputs of the last step of each leg (proofs, accept bytes, MSM results)
are written as DIR/<name>.npy, bytes as float32.  The inputs are seeded, so two builds run with the same arguments
can be compared output for output.

workload `shuffle` (headline; BASELINE configs[1], and configs[3] when --gpus > 1):
    one step = prove + verify a batch of `--batch` independent 52-card shuffle proofs
    (k = 52 -> n = 104 multipliers, Q = 208 constraints, m = 105 commitments; mode "reference-fixed").
    value : proofs/s with witness, commitments and proofs resident in HBM
    e2e   : proofs/s through the host C ABI - witness H2D, proofs D2H, proofs + commitments H2D,
            accept bytes D2H every step (bpp_acp_batch_upload_witness/prove/download_proofs/
            upload_proofs/verify/download_accept)
    multi-GPU: proofs are independent -> each rank owns `--batch` proofs, no data-path collective
            (weak scaling); value = world * batch * steps / max-over-ranks time.
workload `msm` (second half of the metric; BASELINE configs[4] at N = 2^20): reported under "msm".
    multi-GPU: points sharded, one NCCL all-gather of 128 B per rank, then add + compress.

`--impl reference` times the CPU restatement of the reference (oracle/c: dalek-ng 4.1.1 serial
backend + circuit_lib.rs flow) on all host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md 8(d): IMAD.WIDE.U32-equivalents per point operation
IMAD_MADD, IMAD_ADD, IMAD_DBL = 504, 648, 464
L_ORDER = 2**252 + 27742317777372353535851937790883648493
K_CARDS = 52


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def _ncu_traffic(names, kernel):
    """dram read + write bytes of one launch of `kernel` from a committed `ncu --set full` summary (the first of
    profiles/<names> that exists; one column per captured launch) -> (bytes, file) or (None, None)."""
    import csv
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for name in names:
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        rows = list(csv.reader(open(path)))
        col = None
        for row in rows:
            if row and row[0] == "Kernel Name":
                col = next((i for i in range(2, len(row)) if kernel in row[i]), None)
        if col is None:
            continue
        tot, seen = 0.0, set()
        for row in rows:
            if len(row) > col and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and row[0] not in seen:
                seen.add(row[0])
                tot += float(row[col]) * mult.get(row[1], 1.0)
        if tot:
            return tot, name
    return None, None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.samples, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # clocks under load = the upper half of the samples (the sampler also sees idle gaps)
        sm_sorted = sorted(sm)
        under_load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": float(np.median(under_load)) if under_load else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------- synthetic inputs
def synth_msm_inputs(n: int, rank: int, n_sets: int):
    rs = np.random.RandomState(20260000 + rank)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
    sets = []
    for _ in range(n_sets):
        s = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
        s[:, 31] &= 0x0F
        sets.append(s)
    return blobs, sets


def _sc_bytes(vals):
    return b"".join(int(v).to_bytes(32, "little") for v in vals)


def synth_shuffle_batch(k: int, count: int, rank: int):
    """`count` independent k-card shuffles: deck 1..k, a random permutation, a random challenge value X,
    uniform blindings.  Returns bytes for a_L, a_R, a_O (count x n), gamma, v (count x m), seeds."""
    import bpperm_b200
    W = bpperm_b200.weights
    rs = np.random.RandomState(777 + rank)
    aL, aR, aO, vv = [], [], [], []
    for _ in range(count):
        perm = rs.permutation(k)
        x = int.from_bytes(rs.bytes(31), "little")
        v, a_L, a_R, a_O = W.shuffle_witness(k, perm, x)
        aL.append(_sc_bytes(a_L)); aR.append(_sc_bytes(a_R)); aO.append(_sc_bytes(a_O)); vv.append(_sc_bytes(v))
    m = 2 * k + 1
    g = rs.randint(0, 256, size=(count * m, 32), dtype=np.uint8)
    g[:, 31] &= 0x0F
    seeds = rs.randint(0, 256, size=(count, 32), dtype=np.uint8)
    return b"".join(aL), b"".join(aR), b"".join(aO), g.tobytes(), b"".join(vv), seeds.tobytes()


def synth_shuffle_inputs(k: int, count: int, rank: int, salt: int):
    """What defines `count` independent k-card shuffles (the inputs of bpp_acp_batch_gen_shuffle_witness): the deck
    1..k (weights.rs:38-56 create_variables), one permutation and one challenge value X per proof, uniform blindings
    gamma (count x m) and prover RNG seeds.  numpy arrays: deck (k,32) u8, perm (count,k) u32, x (count,32) u8,
    gamma (count*m,32) u8, seeds (count,32) u8."""
    rs = np.random.RandomState(777 + 1000 * salt + rank)
    deck = np.zeros((k, 32), dtype=np.uint8)
    for i in range(k):
        deck[i, :4] = np.frombuffer((i + 1).to_bytes(4, "little"), dtype=np.uint8)
    perm = np.stack([rs.permutation(k) for _ in range(count)]).astype(np.uint32)
    x = rs.randint(0, 256, size=(count, 32), dtype=np.uint8)
    x[:, 31] = 0
    m = 2 * k + 1
    gamma = rs.randint(0, 256, size=(count * m, 32), dtype=np.uint8)
    gamma[:, 31] &= 0x0F
    seeds = rs.randint(0, 256, size=(count, 32), dtype=np.uint8)
    return deck, perm, x, gamma, seeds


def shuffle_witness_bytes(k, deck, perm_row, x_row):
    """a_L, a_R, a_O, v of one shuffle on the host (bulletproof-perm_b200/weights.py), for the CPU arm."""
    import bpperm_b200
    v, a_L, a_R, a_O = bpperm_b200.weights.shuffle_witness(k, [int(j) for j in perm_row], int.from_bytes(bytes(x_row), "little"))
    return _sc_bytes(a_L), _sc_bytes(a_R), _sc_bytes(a_O), _sc_bytes(v)


# batches in flight in the pipelined legs.  Six since round 2: on an 8-GPU host the per-GPU copy bandwidth halves (the
# one-batch-at-a-time e2e step goes from 9.5 to 11.2 ms), a lane's prove -> copy out -> copy in -> verify chain gets longer,
# and three lanes no longer cover it (8 GPUs, e2e: 3 lanes 3.56 M proofs/s, 4: 3.78 M, 6: 4.23 M, 8: 4.04 M;
# profiles/r2f_shuffle_8gpu_lanes*.json); on one GPU six are no worse than three (586 K against 570-582 K e2e).
N_LANES = int(os.environ.get("BPP_LANES", "6"))
LANE_PRIORITY_SPLIT = os.environ.get("BPP_LANE_SPLIT", "1") != "0"
FB_WINDOW_BITS = int(os.environ.get("BPP_FB_WINDOW", "16"))   # fixed-base table window: 16 windows x 32768 entries x 96 B = 50 MB per generator


def shuffle_setup(be, k: int, window_bits: int = FB_WINDOW_BITS):
    """Generators as RistrettoPoint::random (lib.rs:164-167,179-180) from a seeded byte stream, the
    corrected k-card shuffle circuit, fixed-base tables."""
    import bpperm_b200
    G = bpperm_b200.acproof
    n, Q, m, WL, WR, WO, WV, c = bpperm_b200.weights.shuffle_circuit(k)
    rs = np.random.RandomState(4242)
    pts = be.points_from_uniform(rs.randint(0, 256, size=(2 * n + 2, 64), dtype=np.uint8).tobytes())
    enc = be.compress_points(pts)
    pts.free()
    cir = G.Circuit(be, n, Q, m, WL, WR, WO, WV, c)
    gens = G.Generators(be, enc[:32], enc[32:64], [enc[64 + 32 * i: 96 + 32 * i] for i in range(n)],
                        [enc[64 + 32 * (n + i): 96 + 32 * (n + i)] for i in range(n)], window_bits)
    return cir, gens, enc, (n, Q, m)


# ---------------------------------------------------------------------------------- CPU baselines
def _cpu_instance(k, enc):
    """Dense-matrix instance for the C restatement, same generators/circuit as the GPU run."""
    from oracle import cref
    import bpperm_b200
    n, Q, m, WL, WR, WO, WV, c = bpperm_b200.weights.shuffle_circuit(k)

    def dense(tr, rows):
        M = bytearray(rows * Q * 32)
        for i, q, cf in tr:
            M[32 * (i * Q + q): 32 * (i * Q + q) + 32] = int(cf).to_bytes(32, "little")
        return bytes(M)

    return cref.AcpInstance(n, Q, m, dense(WL, n), dense(WR, n), dense(WO, n), dense(WV, m), _sc_bytes(c), enc[:32],
                            enc[32:64], enc[64:64 + 32 * n], enc[64 + 32 * n: 64 + 64 * n])


_CPU_INST = None


def _cpu_one(args):
    aL, aR, aO, gamma, v, seed = args
    Vp = _CPU_INST.commit(v, gamma)
    t0 = time.time()
    pb, rc = _CPU_INST.prove_verify(aL, aR, aO, gamma, Vp, seed, 1)
    return time.time() - t0, rc, pb


def cpu_shuffle_baseline(k, enc, batch_bytes, n_single=8):
    """The reference's CPU path (C restatement of dalek-ng 4.1.1 + circuit_lib.rs, dense matrices) on the
    same inputs: single core (the reference is single-threaded) and all cores over independent proofs."""
    global _CPU_INST
    import multiprocessing as mp
    _CPU_INST = _cpu_instance(k, enc)
    n, m = 2 * k, 2 * k + 1
    aL, aR, aO, gamma, v, seeds = batch_bytes
    cores = os.cpu_count() or 1

    def job(i):
        return (aL[32 * n * i:32 * n * (i + 1)], aR[32 * n * i:32 * n * (i + 1)], aO[32 * n * i:32 * n * (i + 1)],
                gamma[32 * m * i:32 * m * (i + 1)], v[32 * m * i:32 * m * (i + 1)], seeds[32 * i:32 * (i + 1)])

    res = [_cpu_one(job(i)) for i in range(n_single)]
    t1 = sum(r[0] for r in res)
    out = {"value": n_single / t1, "unit": "proofs/s", "cores": 1, "kind": "port",
           "sample": f"{n_single} of the batch's 52-card proofs, prove+verify each, one core ({t1 / n_single * 1e3:.1f} ms/proof)",
           "impl": "C restatement of circuit_lib.rs over curve25519-dalek-ng 4.1.1's serial u64 algorithms (oracle/c)",
           "accepted": all(r[1] == 1 for r in res), "proofs": [r[2] for r in res]}
    try:
        ctx = mp.get_context("fork")
        jobs = [job(i % n_single) for i in range(cores * 2)]
        with ctx.Pool(cores) as pool:
            pool.map(_cpu_one, jobs[:cores])  # warm the workers
            t0 = time.time()
            pool.map(_cpu_one, jobs)
            tall = time.time() - t0
        out["all_cores"] = {"value": len(jobs) / tall, "cores": cores}
    except Exception as e:  # pragma: no cover
        out["all_cores"] = {"error": str(e)}
    return out


def cpu_msm_baseline():
    from oracle import cref
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    n = 1 << 16
    rs = np.random.RandomState(7)
    pts = cref.from_uniform(rs.randint(0, 256, size=(n, 64), dtype=np.uint8).tobytes())
    sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x0F
    scb = sc.tobytes()
    t0 = time.time()
    r1 = cref.msm(scb, pts)
    t1 = time.time() - t0
    out = {"value": n / t1, "unit": "points/s", "cores": 1, "kind": "port",
           "sample": f"one 2^16-point MSM (dalek Pippenger w=8 restated in C, {t1:.2f} s); 2^20 scales linearly"}
    try:
        import ctypes
        per = n // cores
        ctx = mp.get_context("fork")
        jobs = [(scb[32 * i * per:32 * (i + 1) * per], pts[160 * i * per:160 * (i + 1) * per]) for i in range(cores)]
        with ctx.Pool(cores) as pool:
            pool.starmap(cref.msm_raw, [(j[0][:32 * 64], j[1][:160 * 64]) for j in jobs])   # workers forked and warm
            t0 = time.time()                                                              # the clock starts with a warm pool
            parts = pool.starmap(cref.msm_raw, jobs)
            acc = parts[0]
            for p in parts[1:]:
                o = ctypes.create_string_buffer(160)
                cref.lib().orc_point_add(acc, p, o)
                acc = o.raw
            tall = time.time() - t0
        out["all_cores"] = {"value": n / tall, "cores": cores,
                            "matches_1core": (cref.compress(acc) == r1) if per * cores == n else None}
    except Exception as e:  # pragma: no cover
        out["all_cores"] = {"error": str(e)}
    return out


def run_reference_msm_sweep(args):
    """--impl reference --workload msm: the CPU restatement of dalek's vartime_multiscalar_mul on the inputs of
    tools/msm_sweep.py (same seeds), one core and all cores (orc_msm_vartime_mt: points split over threads, partial
    results added), at every N of the sweep up to 2^20 (BASELINE configs[4] "vs dalek ... on host cores")."""
    from oracle import cref
    cores = os.cpu_count() or 1
    rows = []
    for log_n in range(10, 21, 2):
        n = 1 << log_n
        rs = np.random.RandomState(5000 + log_n)
        blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
        sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
        sc[:, 31] &= 0x0F
        pts = cref.from_uniform(blobs.tobytes())
        scb = sc.tobytes()
        reps = 3 if log_n <= 16 else 1
        t0 = time.time()
        for _ in range(reps):
            r1 = cref.msm(scb, pts)
        t1 = (time.time() - t0) / reps
        cref.msm(scb[:32 * 1024], pts[:160 * 1024], threads=cores)   # thread pool warm
        t0 = time.time()
        for _ in range(reps):
            rN = cref.msm(scb, pts, threads=cores)
        tN = (time.time() - t0) / reps
        rows.append({"log_n": log_n, "n": n, "cpu_1core_ms": t1 * 1e3, "cpu_all_cores_ms": tN * 1e3, "cores": cores,
                     "points_per_s_1core": n / t1, "points_per_s_all_cores": n / tN, "result": r1.hex(), "mt_equal": rN == r1})
    line = {"impl": "reference", "metric": "MSM points/sec (sweep 2^10..2^20)", "unit": "points/s", "n_gpus": args.gpus,
            "value": rows[-1]["points_per_s_all_cores"], "higher_is_better": True, "data": "synthetic", "dtype": "u64 (5x51-bit limbs)",
            "config": {"workload": "ristretto255 vartime MSM sweep, inputs of tools/msm_sweep.py (seed 5000 + log2 N)"},
            "cpu_baseline": {"kind": "port", "cores": cores, "value": rows[-1]["points_per_s_all_cores"], "unit": "points/s",
                             "sample": "one MSM per size (three up to 2^16): C restatement of dalek-ng 4.1.1 Straus / Pippenger"},
            "sweep": rows}
    _emit(line)
    return 0


def run_reference(args):
    """--impl reference: the reference's CPU path on all host cores, bounded sample per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    if args.workload == "msm":
        return run_reference_msm_sweep(args)
    global _CPU_INST
    import multiprocessing as mp
    from oracle import cref
    cores = os.cpu_count() or 1
    k = K_CARDS
    n, m = 2 * k, 2 * k + 1
    # same generator stream as the GPU arm; points derived on the CPU
    rs = np.random.RandomState(4242)
    enc = cref.compress(cref.from_uniform(rs.randint(0, 256, size=(2 * n + 2, 64), dtype=np.uint8).tobytes()))
    _CPU_INST = _cpu_instance(k, enc)
    aL, aR, aO, gamma, v, seeds = synth_shuffle_batch(k, cores, 0)
    jobs = [(aL[32 * n * i:32 * n * (i + 1)], aR[32 * n * i:32 * n * (i + 1)], aO[32 * n * i:32 * n * (i + 1)],
             gamma[32 * m * i:32 * m * (i + 1)], v[32 * m * i:32 * m * (i + 1)], seeds[32 * i:32 * (i + 1)])
            for i in range(cores)]
    ctx = mp.get_context("fork")
    ok = True
    with ctx.Pool(cores) as pool:
        for _ in range(args.warmup):
            pool.map(_cpu_one, jobs)
        t0 = time.time()
        for _ in range(args.steps):
            ok = ok and all(r[1] == 1 for r in pool.map(_cpu_one, jobs))
        dt = time.time() - t0
    value = args.steps * cores / dt
    line = {
        "impl": "reference", "metric": "shuffle proofs/sec prove+verify (52-card)", "value": value, "unit": "proofs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (5x51-bit field limbs, 4x64 scalars)",
        "data": "synthetic",
        "config": {"workload": "52-card shuffle proof prove+verify (k=52, n=104, Q=208, m=105), mode reference-fixed",
                   "all_accepted": ok},
        "cpu_baseline": {"value": value, "unit": "proofs/s", "cores": cores, "kind": "port",
                         "sample": f"each step: {cores} independent 52-card proofs (one per core), prove+verify; "
                                   "C restatement of circuit_lib.rs + dalek-ng 4.1.1 serial algorithms, dense W matrices"},
        "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)
    return 0


# ---------------------------------------------------------------------------------- algorithmic work
DECOMP_IMAD = 275 * 72   # one Ristretto (de)compression: an inverse square root (254 squarings + 11 multiplications) and
                         # ~10 more multiplications at 72 IMAD.WIDE.U32 per field multiplication (SURVEY 8(d): madd = 7 x 72)
SC_MUL_IMAD = 136        # one scalar product mod l: 64 (product) + 64 (Montgomery reduction) + 8 (final subtraction)


def _next_pow2(n):
    p = 1
    while p < n:
        p *= 2
    return p


def shuffle_imad_per_proof(n, Q, m, mode, table_windows, rlc_windows):
    """Algorithmic IMAD.WIDE.U32 per proof of one prove + verify (DESIGN.md section 6): fixed-base mixed adds of the
    prover's commitments (and, in `fixed` mode, of the lg n' rounds of L_j, R_j over 2 n' + 2 generators), the
    verifier's share of the batch MSM, point (de)compressions and the scalar products of the vector work."""
    fixed = mode == "fixed"
    np_ = _next_pow2(n) if fixed else n
    lg = np_.bit_length() - 1 if fixed else 0
    terms = (2 * n + 1) + (n + 1) + (2 * n + 1) + 5 * 2 + lg * (2 * np_ + 2)
    dyn = m + 8 + 2 * lg
    madds = terms * table_windows + dyn * rlc_windows
    points = (8 + 2 * lg) + dyn
    sc_mults = 25 * n + (12 * n + 3 * m + Q) + (dyn + 2 * np_ + 2) + (lg * 3 * np_ + 6 * np_ if fixed else 0)
    return {"mixed_adds": madds, "compress_decompress": points, "scalar_products": sc_mults,
            "imad": madds * IMAD_MADD + points * DECOMP_IMAD + sc_mults * SC_MUL_IMAD}


# ---------------------------------------------------------------------------------- GPU arm: shuffle proofs
def _pin(arr):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    return t


# ---------------------------------------------------------------------------------- --dump-outputs
DUMP_ROWS = 1024            # proofs kept per leg: 1024 x 7008 B x 4 = 29 MB for the 52-card `reference-fixed` proofs
DUMP_LIMIT = 64 << 20       # bytes of all dumped arrays together


def dump_rows(n):
    """A fixed, seeded sample of min(n, DUMP_ROWS) row indices in ascending order: the same rows in every run."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.RandomState(0).choice(n, DUMP_ROWS, replace=False))


def bytes_f32(buf, rows=1):
    """Bytes (or a uint8 array) as a (rows, len / rows) float32 array; every byte value is exact in float32."""
    return np.frombuffer(bytes(buf), dtype=np.uint8).reshape(rows, -1).astype(np.float32)


def write_dump(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy, float32 or float64 only, DUMP_LIMIT bytes in all."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"outputs to dump take {total} bytes, more than {DUMP_LIMIT}")
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"{name}: {a.dtype}, expected float32 or float64")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def shuffle_setup_mode(be, k, mode, window_bits):
    """Generators as RistrettoPoint::random (lib.rs:164-167,179-180) from a seeded byte stream (the first 2 n + 2 are
    the stream of the `reference-fixed` runs; `fixed` needs next_pow2(n) per vector), the library-built k-card shuffle
    circuit, fixed-base tables.  Returns (circuit, generators, encodings g | h | G | H, (n, Q, m, ng), table build s)."""
    import bpperm_b200
    G = bpperm_b200.acproof
    n, Q, m = 2 * k, 4 * k, 2 * k + 1
    ng = _next_pow2(n) if mode == "fixed" else n
    rs = np.random.RandomState(4242)
    blobs = rs.randint(0, 256, size=(2 * n + 2, 64), dtype=np.uint8)
    if ng > n:   # g, h, G[0..n), H[0..n) as before, then the padding generators
        extra = np.random.RandomState(4243).randint(0, 256, size=(2 * (ng - n), 64), dtype=np.uint8)
        blobs = np.concatenate([blobs[:2 + n], extra[:ng - n], blobs[2 + n:], extra[ng - n:]])
    pts = be.points_from_uniform(blobs.tobytes())
    enc = be.compress_points(pts)
    pts.free()
    cir = G.Circuit.shuffle(be, k)
    t0 = time.time()
    gens = G.Generators(be, enc[:32], enc[32:64], [enc[64 + 32 * i: 96 + 32 * i] for i in range(ng)],
                        [enc[64 + 32 * (ng + i): 96 + 32 * (ng + i)] for i in range(ng)], window_bits)
    be.synchronize()
    return cir, gens, enc, (n, Q, m, ng), time.time() - t0


def bench_shuffle(E, mode, steps, warmup, want_cpu):
    """prove + verify of `--batch` independent 52-card proofs per GPU and step, inputs resident (value) and through
    host buffers (e2e).  Every step works on the next of N_SETS input sets (permutations, challenge values, blindings,
    prover seeds); the witness is generated on the device from them (bpp_acp_batch_gen_shuffle_witness)."""
    import torch
    import bpperm_b200
    G = bpperm_b200.acproof
    be, dev, stream, world, rank, args, dist = E["be"], E["dev"], E["stream"], E["world"], E["rank"], E["args"], E["dist"]
    timed, timed_block, imad_peak = E["timed"], E["timed_block"], E["imad_peak"]
    k, B = K_CARDS, args.batch
    cir, gens, enc, (n, Q, m, ng), table_s = shuffle_setup_mode(be, k, mode, FB_WINDOW_BITS)
    Wn = (256 + FB_WINDOW_BITS - 1) // FB_WINDOW_BITS
    N_SETS = 4
    sets = [synth_shuffle_inputs(k, B, rank, s) for s in range(N_SETS)]
    h_deck = _pin(sets[0][0])
    d_deck = h_deck.to(dev)
    hs = [dict(perm=_pin(p), x=_pin(x), gamma=_pin(g), seeds=_pin(sd)) for (_, p, x, g, sd) in sets]
    ds = [{kk: v.to(dev) for kk, v in h.items()} for h in hs]
    batch = G.Batch(be, cir, gens, B, mode, b"test")
    plen = batch.proof_len
    # commit_variables for every input set: input generation, not timed
    for s_i in range(N_SETS):
        batch.gen_shuffle_witness(d_deck.data_ptr(), ds[s_i]["perm"].data_ptr(), ds[s_i]["x"].data_ptr(), ds[s_i]["gamma"].data_ptr(),
                                  ds[s_i]["seeds"].data_ptr())
        Vc = batch.commit(None)
        hs[s_i]["V"] = _pin(np.frombuffer(Vc, dtype=np.uint8))
        ds[s_i]["V"] = hs[s_i]["V"].to(dev)

    def resident_step(bt, i):
        d = ds[i % N_SETS]
        bt.gen_shuffle_witness(d_deck.data_ptr(), d["perm"].data_ptr(), d["x"].data_ptr(), d["gamma"].data_ptr(), d["seeds"].data_ptr())
        bt.upload_commitments(d["V"].data_ptr())
        bt.prove()
        bt.verify(None)          # verifier weights from the OS RNG, bound to each proof's transcript

    def e2e_step(bt, i, h_proofs, h_accept):
        h = hs[i % N_SETS]
        bt.gen_shuffle_witness(h_deck.data_ptr(), h["perm"].data_ptr(), h["x"].data_ptr(), h["gamma"].data_ptr(), h["seeds"].data_ptr())
        bt.upload_commitments(h["V"].data_ptr())                 # the prover binds V to its transcript
        bt.prove()
        bt.download_proofs_ptr(h_proofs.data_ptr())              # proofs leave the device ...
        bt.upload_proofs_ptr(h_proofs.data_ptr(), h["V"].data_ptr())   # ... and come back with the commitments
        bt.verify(None)
        bt.download_accept_ptr(h_accept.data_ptr())

    h_proofs = torch.empty(B * plen, dtype=torch.uint8).pin_memory()
    h_accept = torch.empty(B, dtype=torch.uint8).pin_memory()
    state = {"ok": True}

    def step_resident(i):
        resident_step(batch, i)

    def step_e2e(i):
        e2e_step(batch, i, h_proofs, h_accept)
        state["ok"] = state["ok"] and bytes(h_accept.numpy().tobytes()) == b"\x01" * B

    l0 = be.launch_count
    ms_res = timed(step_resident, steps, warmup)
    launches = (be.launch_count - l0) * steps // (steps + warmup)
    batch.download_accept_ptr(h_accept.data_ptr())
    be.synchronize()
    state["ok"] = bytes(h_accept.numpy().tobytes()) == b"\x01" * B
    ms_e2e_serial = timed(step_e2e, steps, warmup)
    serial_last = (warmup + steps - 1) % N_SETS
    serial_proofs = bytes(h_proofs.numpy().tobytes())
    # several batches in flight on several streams, one host thread each, so that the copies and the short dependent
    # kernels of one batch overlap the GPU-filling kernels of another.  Same public calls, same bytes per step; a step
    # is still one batch of B proofs proved and verified.
    lanes = []
    for _ in range(N_LANES):
        st = torch.cuda.Stream(dev, priority=-1) if LANE_PRIORITY_SPLIT else torch.cuda.Stream(dev)
        be_l = bpperm_b200.Backend(E["local"])
        be_l.set_stream(st.cuda_stream)
        b_l = G.Batch(be_l, cir, gens, B, mode, b"test")
        b_l.set_priority_split(LANE_PRIORITY_SPLIT)
        lanes.append({"stream": st, "be": be_l, "batch": b_l, "proofs": torch.empty(B * plen, dtype=torch.uint8).pin_memory(),
                      "accept": torch.empty(B, dtype=torch.uint8).pin_memory(), "ok": True, "last": None})

    def run_lanes(body):
        def run(cnt, first):
            idx = [[first + j for j in range(cnt) if j % N_LANES == kk] for kk in range(N_LANES)]
            th = [threading.Thread(target=body, args=(lanes[kk], idx[kk])) for kk in range(N_LANES) if idx[kk]]
            for t in th:
                t.start()
            for t in th:
                t.join()
        return run

    def lane_resident(lane, idx):
        for i in idx:
            resident_step(lane["batch"], i)

    def lane_e2e(lane, idx):
        for i in idx:
            e2e_step(lane["batch"], i, lane["proofs"], lane["accept"])
            lane["ok"] = lane["ok"] and bytes(lane["accept"].numpy().tobytes()) == b"\x01" * B
            lane["last"] = i

    lane_warm = max(2 * N_LANES, warmup)
    l2_0 = sum(ln["be"].launch_count for ln in lanes)
    ms_res2 = timed_block(run_lanes(lane_resident), steps, lane_warm, [ln["stream"] for ln in lanes])
    launches2 = (sum(ln["be"].launch_count for ln in lanes) - l2_0) * steps // (steps + lane_warm)
    for ln in lanes:
        ln["batch"].download_accept_ptr(ln["accept"].data_ptr())
        ln["be"].synchronize()
        ln["ok"] = ln["ok"] and bytes(ln["accept"].numpy().tobytes()) == b"\x01" * B
    ms_e2e = timed_block(run_lanes(lane_e2e), steps, lane_warm, [ln["stream"] for ln in lanes])
    if E["dump"] is not None:
        # the proofs and accept bytes the last timed step copied to the host
        last = next(ln for ln in lanes if ln["last"] == lane_warm + steps - 1)
        rows = dump_rows(B)
        name = "fixed" if mode == "fixed" else "shuffle"
        E["dump"][f"{name}_proofs"] = bytes_f32(last["proofs"].numpy(), B)[rows]
        E["dump"][f"{name}_proof_rows"] = rows.astype(np.float32)
        E["dump"][f"{name}_accept"] = bytes_f32(last["accept"].numpy())[0]
    all_ok = state["ok"] and all(ln["ok"] for ln in lanes)
    # the same input set gives the same proof bytes on a lane as in the serial run
    same_bytes = None
    for ln in lanes:
        if ln["last"] is not None and ln["last"] % N_SETS == serial_last:
            same_bytes = bytes(ln["proofs"].numpy().tobytes()) == serial_proofs
    for ln in lanes:
        ln["batch"].free()
        ln["be"].close()
    fb_ms, fb_madd, fb_add = batch.time_commit_msm(5)
    if world > 1:
        okt = torch.tensor([1 if all_ok else 0], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        all_ok = bool(okt.item())
    out = None
    if rank == 0:
        total = B * world
        value_single = total * steps / (ms_res * 1e-3)
        value_lanes = total * steps / (ms_res2 * 1e-3)
        two = value_lanes > value_single
        value, ms_step = (value_lanes, ms_res2 / steps) if two else (value_single, ms_res / steps)
        e2e = total * steps / (ms_e2e * 1e-3)
        fb_imads = fb_madd * IMAD_MADD + fb_add * IMAD_ADD
        ach = fb_imads / (fb_ms * 1e-3)
        alg = shuffle_imad_per_proof(n, Q, m, mode, Wn, 16)
        lg = (ng.bit_length() - 1) if mode == "fixed" else 0
        h2d = k * 32 + B * (4 * k + 32 + 32 * m + 32) + B * 32 * m + B * plen + B * 32 * m
        fb_kernel = "k_fb_msm_warp_d" if B >= 16 * 148 and FB_WINDOW_BITS in (8, 16) else ("k_fb_msm_warp" if B >= 16 * 148 else "k_fb_msm")
        traffic, traffic_file = _ncu_traffic(["r2f_ncu_full_fb_msm_warp.csv", "r2f_ncu_full_fb_msm_warp_d.csv"], fb_kernel)
        gens_n = 2 * ng + 2
        table_gib = gens_n * Wn * 2 ** (FB_WINDOW_BITS - 1) * 96 / 2**30
        out = {
            "metric": "shuffle proofs/sec prove+verify (52-card)", "value": value, "unit": "proofs/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 (8x32-bit limbs, IMAD.WIDE.U32)", "data": "synthetic",
            "mode": (f"{N_LANES} batches in flight on {N_LANES} urgent streams (one host thread each; table-gather MSMs on "
                     "lowest-priority streams), inputs resident" if two else "one batch at a time on one stream, inputs resident"),
            "single_stream": {"value": value_single, "ms_per_step": ms_res / steps, "steps": steps},
            "multi_lane": {"lanes": N_LANES, "value": value_lanes, "ms_per_step": ms_res2 / steps, "steps": steps},
            "config": {"workload": f"52-card shuffle prove+verify, batch of {B} independent proofs per GPU "
                                   f"(k=52, n={n}, Q={Q}, m={m}; BASELINE configs[1])",
                       "mode": ("reference-fixed (SURVEY A.3: the reference's own flow never verifies); l, r in the clear, "
                                f"{plen}-byte proofs" if mode != "fixed" else
                                f"fixed: l, r replaced by the inner-product argument (n' = {ng}, {lg} rounds), {plen}-byte proofs"),
                       "inputs": f"{N_SETS} rotating input sets per GPU (a different one every step): deck 1..52, a random permutation and "
                                 "challenge value per proof, uniform blindings, prover RNG = ChaCha20 per proof and seed; witness "
                                 "a_L, a_R, a_O generated on the device from them; generators = from_uniform_bytes(seeded bytes); "
                                 "value commitments bound to every transcript; verifier weights from the OS RNG",
                       "tables": f"fixed-base window tables, c = {FB_WINDOW_BITS}: {table_gib:.1f} GiB in HBM for {gens_n} generators, "
                                 f"built once per generator set in {table_s:.2f} s (not timed) = the time of "
                                 f"{table_s / (ms_step * 1e-3) * B:.0f} proofs at this rate",
                       "verify": "one random-linear-combination MSM over the batch's decompressed points + shared generators "
                                 "(Pippenger), per-proof kernels only on failure; accept bytes are per proof",
                       "l2": f"per-step working set {B * plen / 2**20:.0f} MiB proofs + {B * batch_stride_bytes(n, Q, m, ng, lg) / 2**20:.0f} MiB "
                             f"scalar blocks + randomly gathered {table_gib:.0f} GiB tables + {B * (m + 8 + 2 * lg) * 96 / 2**20:.0f} MiB decompressed points > 126 MB L2",
                       "parallelism": f"proofs sharded over {world} GPU(s), no data-path collective" if world > 1 else "single GPU",
                       "all_accepted": all_ok},
            "e2e": {"value": e2e, "unit": "proofs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": B * plen + B,
                    "ms_per_step": ms_e2e / steps,
                    "serial": {"value": total * steps / (ms_e2e_serial * 1e-3), "ms_per_step": ms_e2e_serial / steps,
                               "note": "one batch at a time: every copy waits for the kernels before it"},
                    "proof_bytes_equal_serial_run": same_bytes,
                    "note": "every step, inside the timed region: permutations + challenge values + blindings + seeds H2D (the witness is "
                            "generated on the device: round 1 sent a_L, a_R, a_O, 3 n x 32 more bytes per proof), commitments H2D, "
                            "proofs D2H, proofs + commitments H2D, accept bytes D2H; pinned host buffers; "
                            f"{N_LANES} batches in flight on {N_LANES} streams; Fiat-Shamir transcripts on the device"},
            "gpu_launches": launches2 if two else launches,
            "roofline": {"bound": "imad", "kernel": f"{fb_kernel} (A_I-shaped commitment MSM, {2 * n + 1} terms x {Wn} windows per proof)",
                         "achieved": ach / 1e12, "peak": imad_peak / 1e12, "unit": "T IMAD.WIDE.U32/s",
                         "frac": ach / imad_peak, "kernel_ms": fb_ms, "point_adds_per_s": (fb_madd + fb_add) / (fb_ms * 1e-3),
                         "peak_source": E["peak_src"], "imad_probes": E["imad_probes"],
                         "traffic": traffic,
                         "traffic_source": f"profiles/{traffic_file} (dram read+write of one A_I-shaped launch; algorithmic gathers = "
                                           f"mixed adds x 96 B = {fb_madd * 96 / 1e9:.2f} GB; a 96-byte entry lies in one or two 128-byte "
                                           "lines, 1.5 on average, and the L2 fills whole lines: 192 B per gather - DESIGN.md section 3.2)",
                         "whole_step": {"imad_per_proof": alg["imad"], "breakdown": alg,
                                        "frac_of_peak": alg["imad"] * B / (ms_step * 1e-3) / imad_peak,
                                        "note": "algorithmic IMAD.WIDE.U32 of one prove + verify (DESIGN.md section 6) x batch / ms_per_step / peak"},
                         "hbm_peak_gbs": E["peaks"].get("hbm_gbs"), "hbm_peak_source": E["peaks_src"]},
        }
        if want_cpu:
            out["cpu_baseline"] = cpu_shuffle_baseline_mode(k, mode, enc, ng, sets[serial_last], serial_proofs, plen)
    batch.free()
    gens.free()
    cir.free()
    return out


def _event_ms(stream, fn, reps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def bench_large_deck(E, k=4096, window_bits=8):
    """BASELINE configs[2]: one proof of a k = 4096-card shuffle (n = 8192 multipliers, 2^14 + 2 generators, 13
    inner-product rounds) on one GPU: prover and verifier latency, device events around each call."""
    import bpperm_b200
    G = bpperm_b200.acproof
    be, stream = E["be"], E["stream"]
    if E["rank"] != 0:
        return None
    cir, gens, enc, (n, Q, m, ng), table_s = shuffle_setup_mode(be, k, "fixed", window_bits)
    deck, perm, x, gamma, seeds = synth_shuffle_inputs(k, 1, 0, 99)
    batch = G.Batch(be, cir, gens, 1, "fixed", b"test")
    batch.gen_shuffle_witness(deck.tobytes(), perm.tobytes(), x.tobytes(), gamma.tobytes(), seeds.tobytes())
    batch.commit(None, want=False)
    for _ in range(3):
        batch.prove()
        batch.verify(None)
    steps = E["args"].steps
    l0 = be.launch_count
    tp = _event_ms(stream, batch.prove, steps)
    lp = (be.launch_count - l0) // steps
    tv = _event_ms(stream, lambda: batch.verify(None), steps)
    ok = batch.download_accept() == b"\x01"
    if E["dump"] is not None:
        E["dump"]["large_deck_proof"] = bytes_f32(batch.download_proofs())[0]
        E["dump"]["large_deck_accept"] = bytes_f32(batch.download_accept())[0]
    Wn = (256 + window_bits - 1) // window_bits
    alg = shuffle_imad_per_proof(n, Q, m, "fixed", Wn, 16)
    out = {"workload": f"large-deck shuffle, k = {k} committed card values, single proof, `fixed` mode (BASELINE configs[2])",
           "n": n, "generators": 2 * ng + 2, "ipa_rounds": ng.bit_length() - 1, "proof_bytes": batch.proof_len,
           "prove_ms": tp, "verify_ms": tv, "proofs_per_s": 1e3 / (tp + tv), "accepted": ok, "prover_launches": lp,
           "tables": f"fixed-base window tables, c = {window_bits}: {(2 * ng + 2) * Wn * 2 ** (window_bits - 1) * 96 / 2**30:.1f} GiB, built in {table_s:.2f} s",
           "whole_step": {"imad_per_proof": alg["imad"], "frac_of_peak": alg["imad"] / ((tp + tv) * 1e-3) / E["imad_peak"],
                          "note": "one proof cannot fill the GPU: the 13 rounds are a chain of dependent launches (latency, not throughput)"}}
    batch.free()
    gens.free()
    cir.free()
    return out


def bench_batch_verify(E, total=4096, corrupt_every=97):
    """BASELINE configs[3]: batch verification of 4096 independent 52-card proofs IN TOTAL (strong scaling), `fixed`
    mode, sharded over the ranks (bulletproof-perm_b200.parallel.shard_bounds), >= 1 % of them corrupted; every rank
    verifies its slice (one random-linear-combination MSM, bisection on failure), the accept bytes are gathered to
    every rank through NCCL and compared with the expected decisions."""
    import torch
    import bpperm_b200
    G = bpperm_b200.acproof
    par = bpperm_b200.parallel
    be, dev, stream, world, rank, args, dist = E["be"], E["dev"], E["stream"], E["world"], E["rank"], E["args"], E["dist"]
    k, mode = K_CARDS, "fixed"
    cir, gens, enc, (n, Q, m, ng), _ = shuffle_setup_mode(be, k, mode, FB_WINDOW_BITS)
    off, cnt = par.shard_bounds(total, world, rank)
    # proofs are produced where they are verified (synthetic input generation, not timed): the same global set for any N
    deck, perm, x, gamma, seeds = synth_shuffle_inputs(k, total, 0, 7)
    sl = slice(off, off + cnt)
    batch = G.Batch(be, cir, gens, cnt, mode, b"test")
    plen = batch.proof_len
    batch.gen_shuffle_witness(deck.tobytes(), perm[sl].tobytes(), x[sl].tobytes(), gamma[m * off:m * (off + cnt)].tobytes(),
                              seeds[sl].tobytes())
    Vc = batch.commit(None)
    batch.prove()
    good = batch.download_proofs()
    bad = bytearray(good)
    expect = bytearray(b"\x01" * cnt)
    fields = [0, 5, 8, 11, 12, plen // 32 - 1]         # A_I, T_4, t_x, L_0, R_0, b
    j = 0
    for g in range(total):
        if g % corrupt_every == 3 and off <= g < off + cnt:
            i, f = g - off, fields[j % len(fields)]
            bad[i * plen + 32 * f + 1] ^= 0x20
            expect[i] = 0
        if g % corrupt_every == 3:
            j += 1
    n_bad_total = len([g for g in range(total) if g % corrupt_every == 3])
    d_good = torch.frombuffer(bytearray(good), dtype=torch.uint8).to(dev)
    d_bad = torch.frombuffer(bad, dtype=torch.uint8).to(dev)
    d_V = torch.frombuffer(bytearray(Vc), dtype=torch.uint8).to(dev)
    per = (total + world - 1) // world
    d_acc = torch.zeros(per, dtype=torch.uint8, device=dev)
    d_all = {"good": torch.zeros(per * world, dtype=torch.uint8, device=dev), "bad": torch.zeros(per * world, dtype=torch.uint8, device=dev)}
    res = {}

    def run(d_proofs, key):
        def step(i):
            batch.upload_proofs_ptr(d_proofs.data_ptr(), d_V.data_ptr())      # D2D: proofs + commitments resident in HBM
            batch.verify(None)
            batch.download_accept_ptr(d_acc.data_ptr())
            be.all_gather_dev(d_acc.data_ptr(), per, d_all[key].data_ptr())   # the library's NCCL communicator (bpp_comm_all_gather_dev)
            res[key] = d_all[key]
        return step

    steps = args.steps
    ms_good = E["timed"](run(d_good, "good"), steps, args.warmup)
    ms_bad = E["timed"](run(d_bad, "bad"), steps, args.warmup)
    acc_all = bytes(res["bad"].cpu().numpy().tobytes())
    mine = acc_all[per * rank: per * rank + cnt]
    ok = mine == bytes(expect)
    okg = bytes(res["good"].cpu().numpy().tobytes())[per * rank: per * rank + cnt] == b"\x01" * cnt
    if world > 1:
        t = torch.tensor([1 if (ok and okg) else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        ok = okg = bool(t.item())
    out = None
    if rank == 0:
        rebuilt = b"".join(acc_all[per * r: per * r + par.shard_bounds(total, world, r)[1]] for r in range(world))
        if E["dump"] is not None:
            E["dump"]["batch_verify_accept"] = bytes_f32(rebuilt)[0]
        out = {"metric": "batch verification proofs/sec (52-card, `fixed` mode)", "unit": "proofs/s", "scaling": "strong",
               "workload": f"{total} independent 52-card proofs in total, sharded over {world} GPU(s) ({cnt} on rank 0), "
                           f"{n_bad_total} of them ({100.0 * n_bad_total / total:.1f} %) corrupted in different fields; verify only; "
                           "accept bytes all-gathered over NCCL (BASELINE configs[3])",
               "n_gpus": world, "steps": steps,
               "value": total / (ms_bad / steps * 1e-3), "ms_per_step": ms_bad / steps,
               "all_valid": {"value": total / (ms_good / steps * 1e-3), "ms_per_step": ms_good / steps},
               "corrupted_over_all_valid": ms_bad / ms_good,
               "rejected": rebuilt.count(b"\x00"), "decisions_match_expected": bool(ok and okg),
               "note": "value = the batch with corrupted proofs (the combined check fails, then every proof is checked on its own: "
                       "DESIGN.md section 3.2 on why group testing does not pay at 1 %); all_valid = the same batch untouched (one combined check)"}
    batch.free()
    gens.free()
    cir.free()
    return out


def bench_small_msm(E):
    """The reference's own call sites (circuit_lib.rs:187-575: 2, 105, 209 points) through the trait-level host call
    bpp_msm_vartime_host (scalars + compressed points in, compressed point out), and `count` of them per launch through
    bpp_msm_vartime_batch; CPU restatement beside it."""
    import bpperm_b200
    from oracle import cref
    be = E["be"]
    if E["rank"] != 0:
        return None
    rs = np.random.RandomState(31)
    rows = []
    for npts in (2, 105, 209):
        blobs = rs.randint(0, 256, size=(npts, 64), dtype=np.uint8).tobytes()
        pts = be.points_from_uniform(blobs)
        enc = be.compress_points(pts)
        sc = rs.randint(0, 256, size=(npts, 32), dtype=np.uint8)
        sc[:, 31] &= 0x0F
        scb = sc.tobytes()
        want = cref.msm(scb, cref.decompress(enc))
        for _ in range(3):
            got = be.msm_host(scb, enc)
        R = E["args"].steps
        t0 = time.time()
        for _ in range(R):
            got = be.msm_host(scb, enc)
        t_host = (time.time() - t0) / R
        t0 = time.time()
        for _ in range(R):
            got_res = be.vartime_multiscalar_mul(scb, pts)
        t_res = (time.time() - t0) / R
        cp = cref.decompress(enc)
        t0 = time.time()
        for _ in range(R):
            cref.msm(scb, cp)
        t_cpu = (time.time() - t0) / R
        t0 = time.time()
        be.precompute(pts, 8)                 # window table of the point set, once (c = 8)
        t_table = time.time() - t0
        for _ in range(3):
            got_tab = be.vartime_multiscalar_mul(scb, pts)
        t0 = time.time()
        for _ in range(R):
            got_tab = be.vartime_multiscalar_mul(scb, pts)
        t_tab = (time.time() - t0) / R
        row = {"points": npts, "host_call_us": t_host * 1e6, "resident_points_call_us": t_res * 1e6,
               "precomputed_points_call_us": t_tab * 1e6, "precompute_once_ms": t_table * 1e3, "cpu_restatement_us": t_cpu * 1e6,
               "matches_cpu": got == want and got_res == want and got_tab == want}
        cnt = 4096
        scs = rs.randint(0, 256, size=(cnt * npts, 32), dtype=np.uint8)
        scs[:, 31] &= 0x0F
        for _ in range(2):
            outs = be.msm_batch(scs.tobytes(), pts, npts, cnt)
        t0 = time.time()
        for _ in range(R):
            outs = be.msm_batch(scs.tobytes(), pts, npts, cnt)
        t_b = (time.time() - t0) / R
        row["batch_4096_shared_points_us_per_msm"] = t_b / cnt * 1e6
        row["batch_first_matches_cpu"] = outs[:32] == cref.msm(scs[:npts].tobytes(), cp)
        if E["dump"] is not None:
            E["dump"][f"trait_call_msm_{npts}"] = bytes_f32(got + got_res + got_tab, 3)
            E["dump"][f"trait_call_msm_batch_{npts}"] = bytes_f32(outs, cnt)
        rows.append(row)
        pts.free()
    return {"note": "wall clock around the public call (host buffers in and out, one synchronisation per call): host_call = "
                    "bpp_msm_vartime_host (points sent, decompressed and bucket-sorted every call, 253 dependent doublings); "
                    "resident_points = bpp_msm_vartime over uploaded points; precomputed_points = the same after "
                    "bpp_points_precompute (table look-ups + mixed adds, no doublings); batch = bpp_msm_vartime_batch: 4096 MSMs "
                    "over the same points with different scalars in one launch",
            "cpu_cores": 1, "rows": rows}


def batch_stride_bytes(n, Q, m, ng, lg):
    """Approximate bytes of one proof's scalar block (acp_make_layout)."""
    return 32 * (8 * n + 3 * m + Q + 12 * n + 6 * ng + 2 * lg + 90 + (2 * ng + 60 if lg else 0))


def cpu_shuffle_baseline_mode(k, mode, enc, ng, input_set, gpu_proofs, plen, n_single=6):
    """The CPU restatement (oracle/c) on the first proofs of the step the GPU's serial e2e run ended on: single core
    (the reference is single-threaded) and all cores over independent proofs; proof bytes compared with the GPU's."""
    global _CPU_INST
    import multiprocessing as mp
    from oracle import cref
    import bpperm_b200
    n, m = 2 * k, 2 * k + 1
    deck, perm, x, gamma, seeds = input_set
    if mode == "fixed":
        _n, Q, _m, WL, WR, WO, WV, c = bpperm_b200.weights.shuffle_circuit(k)
        _CPU_INST = cref.AcpFixedInstance(n, Q, m, WL, WR, WO, WV, _sc_bytes(c), enc[:32], enc[32:64], enc[64:64 + 32 * ng],
                                          enc[64 + 32 * ng:64 + 64 * ng])
    else:
        _CPU_INST = _cpu_instance(k, enc)
    cores = os.cpu_count() or 1

    def job(i):
        aL, aR, aO, v = shuffle_witness_bytes(k, deck, perm[i], x[i])
        return (aL, aR, aO, gamma[m * i:m * (i + 1)].tobytes(), v, seeds[i].tobytes(), mode)

    jobs1 = [job(i) for i in range(n_single)]
    res = [_cpu_one_mode(j) for j in jobs1]
    t1 = sum(r[0] for r in res)
    out = {"value": n_single / t1, "unit": "proofs/s", "cores": 1, "kind": "port",
           "sample": f"the first {n_single} proofs of one GPU step, prove+verify each, one core ({t1 / n_single * 1e3:.1f} ms/proof)",
           "impl": ("C restatement of circuit_lib.rs over curve25519-dalek-ng 4.1.1's serial u64 algorithms (oracle/c), dense W matrices"
                    if mode != "fixed" else
                    "C restatement of the `fixed` flow (oracle/c: sparse weights, bulletproofs 4.0.0 inner-product argument with "
                    "explicit generator folding) over dalek-ng 4.1.1's serial algorithms"),
           "accepted": all(r[1] == 1 for r in res),
           "proof_bytes_equal_gpu": [r[2] for r in res] == [gpu_proofs[i * plen:(i + 1) * plen] for i in range(n_single)]}
    try:
        ctx = mp.get_context("fork")
        jobs = [jobs1[i % n_single] for i in range(cores * 2)]
        with ctx.Pool(cores) as pool:
            pool.map(_cpu_one_mode, jobs[:cores])  # warm the workers
            t0 = time.time()
            pool.map(_cpu_one_mode, jobs)
            tall = time.time() - t0
        out["all_cores"] = {"value": len(jobs) / tall, "cores": cores}
    except Exception as e:  # pragma: no cover
        out["all_cores"] = {"error": str(e)}
    return out


def _cpu_one_mode(args):
    aL, aR, aO, gamma, v, seed, mode = args
    from oracle import cref
    Vp = _CPU_INST.commit(v, gamma)
    if mode == "fixed":
        Ve = cref.compress(Vp)
        t0 = time.time()
        pb = _CPU_INST.prove(aL, aR, aO, gamma, Vp, seed, V_enc=Ve)
        rc = 1 if _CPU_INST.verify(pb, Vp, V_enc=Ve) else 0
        return time.time() - t0, rc, pb
    t0 = time.time()
    pb, rc = _CPU_INST.prove_verify(aL, aR, aO, gamma, Vp, seed, 1)
    return time.time() - t0, rc, pb


# ---------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    import bpperm_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("BPP_BLOCKING_SYNC") == "1":
        # tuning hook: host threads sleep in cudaStreamSynchronize instead of spinning (cudaDeviceScheduleBlockingSync);
        # must precede the creation of the device's primary context
        import ctypes
        rt = ctypes.CDLL("libcudart.so.12")
        rt.cudaSetDevice(local)
        rt.cudaSetDeviceFlags(4)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # one slice of the host cores per rank (round 1: every rank's lane threads roamed over all cores of one NUMA
        # node and the end-to-end legs lost 22 % at 8 GPUs): the rank's threads and its pinned buffers stay together
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            os.sched_setaffinity(0, set(cores[local * per:(local + 1) * per]) or set(cores))
        except Exception:
            pass
    be = bpperm_b200.Backend(local)
    stream = torch.cuda.current_stream(dev)
    be.set_stream(stream.cuda_stream)
    bpperm_b200.parallel.init_comm(be, world, rank, dev)   # the library's own NCCL communicator (bpp_comm_init)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            fn(warmup + i)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed_block(run, steps, warmup, side_streams=()):
        """like timed(), for a body that runs `n` steps at once (pipelined over side streams): run(n, first_index)"""
        run(warmup, 0)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for st in side_streams:
            st.wait_stream(stream)
        run(steps, warmup)
        for st in side_streams:
            stream.wait_stream(st)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # Roofline denominator: the IMAD.WIDE.U32 issue limit (32 lanes/clk/SM = one warp instruction per 4 clocks
    # per sub-partition, confirmed by ncu: fmaheavy cycles per IMAD.WIDE = 4.0) at the maximum SM clock.  The
    # microbenchmarks measured in this run are reported next to it.
    imad_peak = be.imad_pipe_limit()
    imad_probes = {"imad_wide_plain": max(be.pipe_probe(0, 2048) for _ in range(2)),
                   "imad_wide_carry_chained": max(be.pipe_probe(1, 2048) for _ in range(2)),
                   "imad_32": max(be.pipe_probe(2, 2048) for _ in range(2)),
                   "fe_mul_chain_x72": max(be.pipe_probe(4, 512) for _ in range(2)),
                   "ge_madd_chain_x504": max(be.pipe_probe(5, 256) for _ in range(2))}
    imad_probes = {k: v / 1e12 for k, v in imad_probes.items()}
    peak_src = ("IMAD.WIDE.U32 pipe limit = SMs x 32 lanes/clk x max SM clock (4-cycle issue per warp instruction per "
                "sub-partition; ncu fmaheavy cycles per IMAD.WIDE = 4.0, profiles/r1_imad_rate.md); microbenchmarks of "
                "this run in imad_probes (T ops/s)")
    peaks, peaks_src = _peaks()
    line = {}
    sampler = ClockSampler(local)

    E = dict(be=be, dev=dev, stream=stream, world=world, rank=rank, local=local, timed=timed, timed_block=timed_block,
             imad_peak=imad_peak, imad_probes=imad_probes, peak_src=peak_src, peaks=peaks, peaks_src=peaks_src, args=args, dist=dist,
             dump={} if args.dump_outputs else None)
    # ------------------------------------------------------------------ shuffle proofs (headline)
    if args.workload in ("shuffle", "both"):
        if rank == 0:
            sampler.start()
        line = bench_shuffle(E, "reference-fixed", args.steps, args.warmup, want_cpu=(world == 1 and not args.no_cpu))
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            line["clocks"] = clocks
        if not args.no_fixed:
            # the north_star's own protocol: l, r replaced by the inner-product argument (SURVEY 8 row a16)
            fx = bench_shuffle(E, "fixed", args.steps, args.warmup, want_cpu=(world == 1 and not args.no_cpu))
            if rank == 0:
                line["fixed"] = fx
        if not args.no_extra:
            bv = bench_batch_verify(E)          # BASELINE configs[3]: 4096 proofs in total, sharded, >= 1 % corrupted
            ld = bench_large_deck(E) if world == 1 else None   # BASELINE configs[2]: single-GPU by definition
            sm = bench_small_msm(E) if world == 1 else None    # the reference's 15 call sites through the trait-level call
            if rank == 0:
                line["batch_verify"] = bv
                if ld:
                    line["large_deck"] = ld
                if sm:
                    line["trait_call_msm"] = sm

    # ------------------------------------------------------------------ MSM at 2^20 (second metric)
    if args.workload in ("msm", "both"):
        n = 1 << args.log_n
        n_sets = 4
        blobs, sets = synth_msm_inputs(n, rank, n_sets)
        table = be.points_from_uniform(blobs.tobytes())
        d_sets = [torch.from_numpy(s).to(dev) for s in sets]
        h_sets = [torch.from_numpy(s).pin_memory() for s in sets]
        smsm = bpperm_b200.parallel.ShardedMsm(be, table, world, dev)
        d_out = smsm.d_out
        h_out = torch.zeros(32, dtype=torch.uint8).pin_memory()

        def msm_once(d_sc):
            smsm.run(d_sc)

        def msm_resident(i):
            msm_once(d_sets[i % n_sets])

        def msm_e2e(i):
            d_sc = d_sets[i % n_sets]
            d_sc.copy_(h_sets[(i + 1) % n_sets], non_blocking=True)
            msm_once(d_sc)
            h_out.copy_(d_out[:32], non_blocking=True)
            stream.synchronize()

        # throughput form (single GPU): every step is one bpp_msm_submit_dev, two MSMs in flight on the library's
        # internal streams (the dependent tail of one beside the sort + accumulate of the next), one bpp_msm_wait
        # before the closing event; results alternate between two output buffers
        d_outs = [torch.zeros(160, dtype=torch.uint8, device=dev) for _ in range(2)]

        def msm_submitted(cnt, first):
            if world > 1:   # sharded: the 128-byte all-gather of step i-1 on a side stream beside the MSM of step i
                smsm.run_many([d_sets[(first + i) % n_sets] for i in range(cnt)])
                return
            for i in range(cnt):
                be.msm_submit_dev(d_sets[(first + i) % n_sets].data_ptr(), table, 0, n, d_outs[i & 1].data_ptr())
            be.msm_wait()

        msm_steps = args.steps
        l0 = be.launch_count
        samp2 = ClockSampler(local)
        if rank == 0 and args.workload == "msm":
            samp2.start()
        ms_single = timed(msm_resident, msm_steps, args.warmup)
        launches = (be.launch_count - l0) * msm_steps // (msm_steps + args.warmup)
        ms_res = timed_block(msm_submitted, msm_steps, args.warmup)
        # the submitted results of the last two timed steps are the single-call results
        last_two = range(max(0, msm_steps - 2), msm_steps)
        want = []
        for i in last_two:
            msm_once(d_sets[(args.warmup + i) % n_sets])
            want.append(bytes(d_out[:32].cpu().numpy().tobytes()))
        if world == 1:
            got = [bytes(d_outs[i & 1][:32].cpu().numpy().tobytes()) for i in last_two]
        else:
            got = [bytes(smsm.d_outs[i % 3][:32].cpu().numpy().tobytes()) for i in last_two]
        assert got == want, "submitted MSM results differ from the single-call results"
        sharded_check = None
        if world > 1:
            # independent of the library's communicator: every rank's partial point (bpp_msm_partial_dev) all-gathered by
            # torch.distributed, summed and compressed by one rank-local kernel - must be the sharded call's result
            d_part = torch.zeros(128, dtype=torch.uint8, device=dev)
            d_allp = torch.zeros(128 * world, dtype=torch.uint8, device=dev)
            d_chk = torch.zeros(32, dtype=torch.uint8, device=dev)
            last = d_sets[(args.warmup + msm_steps - 1) % n_sets]
            be.msm_partial_dev(last.data_ptr(), table, 0, n, d_part.data_ptr())
            stream.synchronize()
            dist.all_gather_into_tensor(d_allp, d_part)
            torch.cuda.synchronize()
            be.points_sum_compress_dev(d_allp.data_ptr(), world, d_chk.data_ptr())
            sharded_check = bytes(d_chk.cpu().numpy().tobytes()) == want[-1]
            assert sharded_check, "sharded MSM (library NCCL) differs from partials gathered by torch.distributed"
        clocks2 = samp2.stop() if (rank == 0 and args.workload == "msm") else None
        ms_e2e_serial = timed(msm_e2e, msm_steps, args.warmup)
        # e2e, double buffered: the next step's scalars travel on a copy stream while this step's MSM runs
        copy_stream = torch.cuda.Stream(dev)
        bufs3 = [torch.empty_like(d_sets[0]) for _ in range(3)]
        ready3 = [torch.cuda.Event() for _ in range(3)]
        free3 = [torch.cuda.Event() for _ in range(3)]

        def msm_pipelined(cnt, first):
            if world == 1:
                # submit(i) / wait_previous / read result i-1: scalars of step i+1 travel on the copy stream meanwhile;
                # three scalar buffers because two MSMs are in flight while the third buffer is being filled
                used = [False] * 3
                with torch.cuda.stream(copy_stream):
                    bufs3[0].copy_(h_sets[first % n_sets], non_blocking=True)
                    ready3[0].record(copy_stream)
                for i in range(cnt):
                    b, nb = i % 3, (i + 1) % 3
                    if i + 1 < cnt:
                        with torch.cuda.stream(copy_stream):
                            if used[nb]:
                                copy_stream.wait_event(free3[nb])
                            bufs3[nb].copy_(h_sets[(first + i + 1) % n_sets], non_blocking=True)
                            ready3[nb].record(copy_stream)
                    stream.wait_event(ready3[b])
                    be.msm_submit_dev(bufs3[b].data_ptr(), table, 0, n, d_outs[i & 1].data_ptr())
                    be.msm_wait_previous()
                    if i:
                        pb = (i - 1) % 3
                        free3[pb].record(stream)   # MSM i-1 is complete here in stream order: its scalars may be replaced
                        used[pb] = True
                        h_out.copy_(d_outs[(i - 1) & 1][:32], non_blocking=True)
                be.msm_wait()
                h_out.copy_(d_outs[(cnt - 1) & 1][:32], non_blocking=True)
                return
            # sharded: bpp_msm_sharded_submit_dev(i) leaves the caller's stream behind MSM i - 1 (its scalars may be
            # replaced) and behind the gathered result of MSM i - 2 (it may be read); scalars of step i + 1 travel on
            # the copy stream meanwhile
            used = [False] * 3
            with torch.cuda.stream(copy_stream):
                bufs3[0].copy_(h_sets[first % n_sets], non_blocking=True)
                ready3[0].record(copy_stream)
            for i in range(cnt):
                b, nb = i % 3, (i + 1) % 3
                if i + 1 < cnt:
                    with torch.cuda.stream(copy_stream):
                        if used[nb]:
                            copy_stream.wait_event(free3[nb])
                        bufs3[nb].copy_(h_sets[(first + i + 1) % n_sets], non_blocking=True)
                        ready3[nb].record(copy_stream)
                stream.wait_event(ready3[b])
                be.msm_sharded_submit_dev(bufs3[b].data_ptr(), table, 0, n, smsm.d_outs[i % 3].data_ptr())
                if i >= 1:
                    free3[(i - 1) % 3].record(stream)
                    used[(i - 1) % 3] = True
                if i >= 2:
                    h_out.copy_(smsm.d_outs[(i - 2) % 3][:32], non_blocking=True)
            be.msm_sharded_wait()
            if cnt >= 2:
                h_out.copy_(smsm.d_outs[(cnt - 2) % 3][:32], non_blocking=True)
            h_out.copy_(smsm.d_outs[(cnt - 1) % 3][:32], non_blocking=True)

        ms_e2e = timed_block(msm_pipelined, msm_steps, args.warmup, [copy_stream])
        if E["dump"] is not None:
            E["dump"]["msm_result"] = bytes_f32(h_out.numpy())[0]    # the last step's result, on the host
        be.set_profiling(True)
        acc_ms = []
        for i in range(5):
            be.msm_dev(d_sets[i % n_sets].data_ptr(), table, 0, n, d_out.data_ptr())
            ph = be.last_phase_ms()
            acc_ms.append([ph[kk] for kk in bpperm_b200.backend.PHASES])
        be.set_profiling(False)
        ops = be.last_op_counts()
        if rank == 0:
            total_points = n * world
            phases = np.median(np.array(acc_ms), axis=0)
            acc_t = float(phases[3]) * 1e-3
            imads_acc = ops["mixed_adds"] * IMAD_MADD
            imads_all = imads_acc + ops["full_adds"] * IMAD_ADD + ops["doublings"] * IMAD_DBL
            c_win = 8 if n <= 1500 else 11 if n <= 96000 else 15 if n < 1000000 else 16      # pick_window (capi_core.cu)
            W_win = (253 + c_win - 1) // c_win
            imads_alg = IMAD_MADD * n * W_win + IMAD_ADD * 2 * (2 ** (c_win - 1) - 1) * W_win + IMAD_DBL * c_win * (W_win - 1)
            ach = imads_acc / acc_t
            acc_traffic, acc_traffic_file = _ncu_traffic(["r2f_ncu_full_msm2p20.csv", "r2_ncu_full_msm2p20.csv"], "k_bucket_accum")
            msm = {
                "metric": "MSM points/sec at 2^20", "value": total_points * msm_steps / (ms_res * 1e-3), "unit": "points/s",
                "n_gpus": world, "steps": msm_steps, "ms_per_step": ms_res / msm_steps, "scaling": "weak",
                "mode": ("throughput: one bpp_msm_submit_dev per step, two MSMs in flight (the tail of one beside the sort "
                         "and accumulate of the next), one bpp_msm_wait before the closing event; results checked against "
                         "the single-call results") if world == 1 else
                        ("throughput, sharded: bpp_msm_submit_partial_dev per step on every rank (two in flight), the 128-byte "
                         "all-gather of step i-1 on a side stream beside the MSM of step i, its sum one step later; results "
                         "checked against the single-call results"),
                "single_call": {"value": total_points * msm_steps / (ms_single * 1e-3), "ms_per_step": ms_single / msm_steps,
                                "note": "bpp_msm_vartime_dev one call at a time: the caller's stream joins every MSM"},
                "config": {"workload": f"ristretto255 vartime MSM, 2^{args.log_n} points per GPU (BASELINE configs[4])",
                           "points": "from_uniform_bytes(seeded bytes), resident as affine Niels (96 B/pt), no precomputed multiples",
                           "scalars": "uniform < 2^252, 4 rotating sets",
                           "l2": "96 MiB table + 32 MiB scalars + 100 MiB sort scratch + 64 MiB buckets > 126 MB L2",
                           "parallelism": f"points sharded over {world} GPUs, one NCCL all-gather of 128 B/rank" if world > 1 else "single GPU",
                           "result": bytes(d_out[:32].cpu().numpy().tobytes()).hex(),
                           "sharded_result_equals_partials_gathered_by_torch": sharded_check},
                "e2e": {"value": total_points * msm_steps / (ms_e2e * 1e-3), "unit": "points/s", "h2d_bytes_per_step": n * 32,
                        "d2h_bytes_per_step": 32, "ms_per_step": ms_e2e / msm_steps,
                        "serial": {"value": total_points * msm_steps / (ms_e2e_serial * 1e-3), "ms_per_step": ms_e2e_serial / msm_steps},
                        "note": "scalars pinned-host->HBM and result HBM->host every step; generator table resident; the next "
                                "step's scalars are copied on a second stream during this step's MSM; submitted form (two MSMs "
                                "in flight per GPU; sharded: bpp_msm_sharded_submit_dev, the 128-byte gather of step i-1 beside step i)"},
                "gpu_launches": launches,
                "roofline": {"bound": "imad", "kernel": "k_bucket_accum", "achieved": ach / 1e12, "peak": imad_peak / 1e12,
                             "unit": "T IMAD.WIDE.U32/s", "frac": ach / imad_peak, "kernel_ms": float(phases[3]),
                             "point_adds_per_s": ops["mixed_adds"] / acc_t, "peak_source": peak_src,
                             "traffic": acc_traffic if args.log_n == 20 else None,
                             "traffic_source": f"profiles/{acc_traffic_file} (dram read+write of one k_bucket_accum launch, 2^20 points, one window group)",
                             "whole_msm": {"imad_algorithmic": imads_alg, "formula": "SURVEY 8(d): 504 N W + 648 * 2 (2^(c-1) - 1) W + 464 c (W - 1), "
                                                                                     f"c = {c_win}, W = {W_win}",
                                           "frac_of_peak": imads_alg / (ms_res / msm_steps * 1e-3) / imad_peak,
                                           "frac_of_peak_single_call": imads_alg / (ms_single / msm_steps * 1e-3) / imad_peak,
                                           "imad_executed": imads_all},
                             "phases_ms": dict(zip(bpperm_b200.backend.PHASES, [float(x) for x in phases]))},
            }
            if clocks2:
                msm["clocks"] = clocks2
            if world == 1 and not args.no_cpu:
                msm["cpu_baseline"] = cpu_msm_baseline()
            if line:
                line["msm"] = msm
            else:
                line = dict(msm)
                line.update({"warmup": args.warmup, "higher_is_better": True, "vs_baseline": None,
                             "dtype": "u32 (8x32-bit limbs, IMAD.WIDE.U32)", "data": "synthetic"})

    if rank == 0:
        if E["dump"] is not None:
            write_dump(args.dump_outputs, E["dump"])
        _emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def _emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="both", choices=["shuffle", "msm", "both"])
    ap.add_argument("--batch", type=int, default=4096, help="independent 52-card proofs per GPU per step")
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline legs")
    ap.add_argument("--no-fixed", action="store_true", help="skip the `fixed` (inner-product) mode leg of the shuffle workload")
    ap.add_argument("--no-extra", action="store_true", help="skip batch_verify / large_deck / trait_call_msm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of each leg's last step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    # The contract is ONE JSON line on stdout.  Libraries write to file descriptor 1 behind Python's back (NCCL prints
    # its version banner there): keep the real stdout aside for the JSON line and point fd 1 at stderr meanwhile.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
