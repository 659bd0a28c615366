"""One prove + one verify of a k-card batch inside a cudaProfilerStart/Stop range (for `ncu --profile-from-start off`),
with CUDA-event times of both printed first.  argv: k, mode, batch, table window bits, [out json]"""
import ctypes
import json
import sys

import numpy as np

sys.path.insert(0, ".")
import bench, bpperm_b200

k = int(sys.argv[1]) if len(sys.argv) > 1 else 52
mode = sys.argv[2] if len(sys.argv) > 2 else "fixed"
B = int(sys.argv[3]) if len(sys.argv) > 3 else 4096
cb = int(sys.argv[4]) if len(sys.argv) > 4 else 16
out = sys.argv[5] if len(sys.argv) > 5 else None

import torch

be = bpperm_b200.Backend(0)
stream = torch.cuda.current_stream()
be.set_stream(stream.cuda_stream)
import os
if os.environ.get("BPP_GROUPS"):
    be.set_msm_groups(int(os.environ["BPP_GROUPS"]))
G = bpperm_b200.acproof
n, Q, m, WL, WR, WO, WV, c = bpperm_b200.weights.shuffle_circuit(k)
ng = G.next_pow2(n) if mode == "fixed" else n
rs = np.random.RandomState(4242)
pts = be.points_from_uniform(rs.randint(0, 256, size=(2 * ng + 2, 64), dtype=np.uint8).tobytes())
enc = be.compress_points(pts)
cir = G.Circuit(be, n, Q, m, WL, WR, WO, WV, c)
gens = G.Generators(be, enc[:32], enc[32:64], [enc[64 + 32 * i: 96 + 32 * i] for i in range(ng)],
                    [enc[64 + 32 * (ng + i): 96 + 32 * (ng + i)] for i in range(ng)], cb)
aL, aR, aO, gamma, v, seeds = bench.synth_shuffle_batch(k, B, 0)
batch = G.Batch(be, cir, gens, B, mode, b"test")
batch.upload_witness(aL, aR, aO, gamma, seeds)
batch.commit(v)
for _ in range(3):
    batch.prove()
    batch.verify(b"\x01" * 32)
be.synchronize()


def timed(fn, reps=5):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


tp = timed(batch.prove)
tv = timed(lambda: batch.verify(b"\x01" * 32))
fb_ms, fb_madd, _ = batch.time_commit_msm(10)
import os
row = {"k": k, "mode": mode, "batch": B, "table_window_bits": cb, "prove_ms": tp, "verify_ms": tv, "a_i_msm_ms": fb_ms,
       "a_i_msm_frac_of_imad_limit": fb_madd * 504 / (fb_ms * 1e-3) / be.imad_pipe_limit(), "lib": os.environ.get("BPPERM_LIB", "product"),
       "proofs_per_s": B / ((tp + tv) * 1e-3), "accepted": batch.download_accept() == b"\x01" * B}
print(json.dumps(row), flush=True)
if out:
    json.dump(row, open(out, "w"))
torch.cuda.synchronize()
torch.cuda.profiler.start()
batch.prove()
batch.verify(b"\x01" * 32)
torch.cuda.synchronize()
torch.cuda.profiler.stop()
