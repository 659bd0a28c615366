"""GPU parity: RistrettoPoint::vartime_multiscalar_mul through the C ABI vs the CPU oracle.
Bit-exact on the 32-byte compressed result."""
import os
import random

import pytest

from oracle import ristretto255 as R
from oracle.chacha import ChaChaRng

pytestmark = pytest.mark.gpu


def _inputs(n, seed):
    rng = ChaChaRng(bytes([seed]) * 32)
    pts = [rng.point() for _ in range(n)]
    sc = [rng.scalar() for _ in range(n)]
    return sc, pts


def test_survey_e2_golden_vector(backend):
    rng = ChaChaRng(bytes(range(32)))
    pts = [rng.point() for _ in range(4)]
    sc = [rng.scalar() for _ in range(4)]
    out = backend.vartime_multiscalar_mul(sc, [R.compress(p) for p in pts])
    assert out.hex() == "ac0188282e26885b30102aa5ee4e91734b3328dba689b17245af361585d58d6f"


# the reference's own MSM sizes at 52 cards (SURVEY 2.2) plus ragged / tiny cases
@pytest.mark.parametrize("n", [1, 2, 3, 17, 104, 105, 110, 111, 209, 600])
def test_msm_matches_oracle(backend, n):
    sc, pts = _inputs(n, n % 251)
    want = R.compress(R.msm_naive(sc, pts))
    got = backend.vartime_multiscalar_mul(sc, [R.compress(p) for p in pts])
    assert got == want


@pytest.mark.parametrize("c", list(range(4, 17)))
def test_every_window_width_gives_identical_bytes(backend, c):
    sc, pts = _inputs(64, 77)
    want = R.compress(R.msm_naive(sc, pts))
    backend.set_window_bits(c)
    try:
        assert backend.vartime_multiscalar_mul(sc, [R.compress(p) for p in pts]) == want
    finally:
        backend.set_window_bits(0)


def test_edge_scalars_and_points(backend):
    sc, pts = _inputs(12, 3)
    sc[0] = 0
    sc[1] = 1
    sc[2] = R.L - 1
    sc[3] = 2**252
    sc[4] = R.L - 2**128
    pts[5] = R.IDENTITY
    pts[6] = pts[7]                      # repeated point
    sc[8], sc[9] = 12345, R.L - 12345    # s*P + (-s)*P
    pts[9] = pts[8]
    sc[10] = (1 << 255) - 1 - (1 << 254)  # non-canonical but bit 255 clear (dalek allows < 2^255)
    want = R.compress(R.msm_naive([s % R.L for s in sc], pts))
    got = backend.vartime_multiscalar_mul(sc, [R.compress(p) for p in pts])
    assert got == want


def test_cancelling_terms_give_identity(backend):
    sc, pts = _inputs(5, 4)
    sc2 = sc + [R.L - s for s in sc]
    enc = [R.compress(p) for p in pts] * 2
    assert backend.vartime_multiscalar_mul(sc2, enc) == bytes(32)
    assert backend.vartime_multiscalar_mul([0] * 10, enc) == bytes(32)


def test_empty_and_error_behaviour(backend):
    import bpperm_b200
    assert backend.vartime_multiscalar_mul([], []) == bytes(32)   # empty sum = identity (dalek: same)
    sc, pts = _inputs(3, 5)
    enc = [R.compress(p) for p in pts]
    with pytest.raises(bpperm_b200.BppError) as ei:              # dalek asserts equal lengths
        backend.vartime_multiscalar_mul(sc[:2], enc)
    assert ei.value.status == -4
    with pytest.raises(bpperm_b200.BppError) as ei:
        backend.vartime_multiscalar_mul([1 << 255, 1, 1], enc)
    assert ei.value.status == -6
    with pytest.raises(bpperm_b200.BppError) as ei:              # decompress().unwrap() on a bad point
        backend.vartime_multiscalar_mul(sc, enc[:2] + [b"\x01" + bytes(31)])
    assert ei.value.status == -5


def test_resident_points_offsets_and_ext_output(backend):
    sc, pts = _inputs(40, 6)
    table = backend.upload_points([R.compress(p) for p in pts])
    for off, n in ((0, 40), (5, 10), (39, 1), (13, 27)):
        want = R.msm_naive(sc[:n], pts[off:off + n])
        got, ext = backend.vartime_multiscalar_mul(sc[:n], table, off=off, n=n, want_ext=True)
        assert got == R.compress(want)
        X, Y, Z, T = (int.from_bytes(ext[32 * k:32 * k + 32], "little") for k in range(4))
        assert max(X, Y, Z, T) < R.P
        assert R.compress((X, Y, Z, T)) == got and (X * Y - Z * T) % R.P == 0


def _np_scalars(n, seed):
    import numpy as np
    rs = np.random.RandomState(seed)
    b = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    b[:, 31] &= 0x0F      # < 2^252 < l: canonical
    return b


@pytest.mark.parametrize("logn", [14, 20])
def test_large_msm_properties(backend, logn):
    """BASELINE sizes: no CPU oracle finishes 2^20 in seconds, so check size-independent properties:
    (1) identical bytes for two different window widths (two different bucket decompositions),
    (2) split linearity: MSM(all) == sum of the two half-MSMs' partial points,
    (3) scalar linearity: MSM(s) + MSM(l - s) == identity,
    (4) a 600-point slice equals the CPU oracle."""
    import numpy as np
    import torch
    n = 1 << logn
    seed_bytes = np.random.RandomState(logn).randint(0, 256, size=(n, 64), dtype=np.uint8).tobytes()
    table = backend.points_from_uniform(seed_bytes)
    sc = _np_scalars(n, 1000 + logn)
    scb = sc.tobytes()
    full = backend.vartime_multiscalar_mul(scb, table)
    backend.set_window_bits(13)
    try:
        assert backend.vartime_multiscalar_mul(scb, table) == full
    finally:
        backend.set_window_bits(0)
    # (2) halves via the device-pointer partial API
    dev = torch.device("cuda:0")
    d_sc = torch.from_numpy(sc).to(dev)
    parts = torch.zeros(2, 128, dtype=torch.uint8, device=dev)
    out32 = torch.zeros(32, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    h = n // 2
    backend.msm_partial_dev(d_sc.data_ptr(), table, 0, h, parts[0].data_ptr())
    backend.msm_partial_dev(d_sc[h:].data_ptr(), table, h, n - h, parts[1].data_ptr())
    backend.points_sum_compress_dev(parts.data_ptr(), 2, out32.data_ptr())
    backend.synchronize()
    assert bytes(out32.cpu().numpy().tobytes()) == full
    # (3) negated scalars
    neg = np.zeros_like(sc)
    for i in range(0, n, max(1, n // 4096)):   # negate a subset exactly on the host (python ints)
        pass
    sub = 2048
    s_int = [int.from_bytes(sc[i].tobytes(), "little") for i in range(sub)]
    both = b"".join(x.to_bytes(32, "little") for x in s_int) + b"".join((R.L - x).to_bytes(32, "little") for x in s_int)
    enc = backend.compress_points(table, 0, sub)
    t2 = backend.upload_points(enc + enc)
    assert backend.vartime_multiscalar_mul(both, t2) == bytes(32)
    # (4) slice against the oracle
    k = 600
    pts = [R.decompress(enc[32 * i:32 * i + 32]) for i in range(k)]
    want = R.compress(R.msm_naive(s_int[:k], pts))
    assert backend.vartime_multiscalar_mul(scb[:32 * k], table, off=0, n=k) == want


@pytest.mark.parametrize("log_n", [10, 12, 14, 16])
def test_sweep_inputs_match_oracle(backend, log_n):
    """BASELINE configs[4]: the seeded inputs of tools/msm_sweep.py (seed 5000 + log2 N) against the C restatement
    of dalek's vartime_multiscalar_mul; pins the `result` bytes recorded in profiles/*msm_sweep*.json."""
    import numpy as np
    from oracle import cref
    n = 1 << log_n
    rs = np.random.RandomState(5000 + log_n)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
    sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x0F
    table = backend.points_from_uniform(blobs.tobytes())
    got = backend.vartime_multiscalar_mul(sc.tobytes(), table)
    table.free()
    assert got == cref.msm(sc.tobytes(), cref.from_uniform(blobs.tobytes()))


@pytest.mark.parametrize("groups,c", [(2, 16), (3, 11), (4, 16), (5, 13), (8, 8), (8, 16), (4, 0)])
def test_window_groups_match_oracle(backend, groups, c):
    """The pipelined form (window groups on side streams, bpp_set_msm_groups) against the C restatement: 2^14 random
    terms plus a skewed tail (repeated and tiny scalars: hot buckets and the long-bucket queue inside every group,
    zero scalars: empty windows).  The bytes must not depend on the grouping or on the window width."""
    import numpy as np
    from oracle import cref
    n = (1 << 14) + 3000
    rs = np.random.RandomState(900 + groups)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
    sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x0F
    sc[1 << 14:(1 << 14) + 2000] = sc[7]          # one scalar 2000 times: every window has a hot bucket
    sc[(1 << 14) + 2000:(1 << 14) + 2500, 1:] = 0  # tiny scalars: only window 0 is populated
    sc[(1 << 14) + 2500:] = 0                      # zero scalars
    table = backend.points_from_uniform(blobs.tobytes())
    backend.set_window_bits(c)
    backend.set_msm_groups(groups)
    try:
        got = backend.vartime_multiscalar_mul(sc.tobytes(), table)
        again = backend.vartime_multiscalar_mul(sc.tobytes(), table)   # scratch reuse across calls
        backend.set_msm_groups(1)
        in_order = backend.vartime_multiscalar_mul(sc.tobytes(), table)
    finally:
        backend.set_window_bits(0)
        backend.set_msm_groups(0)
        table.free()
    assert got == again == in_order
    assert got == cref.msm(sc.tobytes(), cref.from_uniform(blobs.tobytes()))


def test_submitted_msms_match_joined(backend):
    """bpp_msm_submit_dev / bpp_msm_wait: six independent MSMs submitted back to back (two in flight on the internal
    streams, scratch slots reused three times) give the bytes of the one-at-a-time calls and of the C restatement."""
    import numpy as np
    import torch
    from oracle import cref
    n = 1 << 14
    rs = np.random.RandomState(4242)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
    table = backend.points_from_uniform(blobs.tobytes())
    dev = torch.device("cuda:0")
    sets = []
    for i in range(6):
        sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
        sc[:, 31] &= 0x0F
        if i == 3:
            sc[:5000] = sc[0]     # a skewed one in the middle
        sets.append(sc)
    d_sets = [torch.from_numpy(s).to(dev) for s in sets]
    outs = torch.zeros(6, 160, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    backend.set_msm_groups(4)
    try:
        for i in range(6):
            backend.msm_submit_dev(d_sets[i].data_ptr(), table, 0, n, outs[i].data_ptr())
        backend.msm_wait()
        backend.synchronize()
        got = [bytes(outs[i, :32].cpu().numpy().tobytes()) for i in range(6)]
        outs.zero_()
        # mixed: submitted, then a joined call, then a partial (uncompressed) one
        backend.msm_submit_dev(d_sets[0].data_ptr(), table, 0, n, outs[0].data_ptr())
        backend.msm_dev(d_sets[1].data_ptr(), table, 0, n, outs[1].data_ptr())
        backend.synchronize()
        assert bytes(outs[0, :32].cpu().numpy().tobytes()) == got[0]
        assert bytes(outs[1, :32].cpu().numpy().tobytes()) == got[1]
    finally:
        backend.set_msm_groups(0)
    pts = cref.from_uniform(blobs.tobytes())
    for i in (0, 3, 5):
        assert got[i] == cref.msm(sets[i].tobytes(), pts)
    backend.set_msm_groups(1)
    try:
        for i in range(6):
            assert backend.vartime_multiscalar_mul(sets[i].tobytes(), table) == got[i]
    finally:
        backend.set_msm_groups(0)
        table.free()


def test_wait_previous_producer_consumer_loop():
    """submit(i); wait_previous(); consume(i-1) on the caller's (torch) stream: the consumer copies see final bytes."""
    import numpy as np
    import torch
    import bpperm_b200
    dev = torch.device("cuda:0")
    be = bpperm_b200.Backend(0)
    stream = torch.cuda.Stream(dev)
    be.set_stream(stream.cuda_stream)
    n = 1 << 13
    rs = np.random.RandomState(77)
    table = be.points_from_uniform(rs.randint(0, 256, size=(n, 64), dtype=np.uint8).tobytes())
    sets = []
    for i in range(5):
        sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
        sc[:, 31] &= 0x0F
        sets.append(sc)
    want = [be.vartime_multiscalar_mul(s.tobytes(), table) for s in sets]
    d_sets = [torch.from_numpy(s).to(dev) for s in sets]
    outs = torch.zeros(5, 160, dtype=torch.uint8, device=dev)
    host = torch.zeros(5, 32, dtype=torch.uint8).pin_memory()
    torch.cuda.synchronize()
    be.set_msm_groups(3)
    with torch.cuda.stream(stream):
        for i in range(5):
            be.msm_submit_dev(d_sets[i].data_ptr(), table, 0, n, outs[i].data_ptr())
            be.msm_wait_previous()
            if i:
                host[i - 1].copy_(outs[i - 1, :32], non_blocking=True)
        be.msm_wait()
        host[4].copy_(outs[4, :32], non_blocking=True)
    stream.synchronize()
    be.set_msm_groups(0)
    for i in range(5):
        assert bytes(host[i].numpy().tobytes()) == want[i], i
    table.free()
    be.close()


@pytest.mark.parametrize("c,groups", [(16, 1), (16, 4), (15, 2), (13, 2), (12, 1), (11, 3), (8, 1), (5, 8), (4, 1), (0, 0)])
def test_skewed_scalars_match_oracle(backend, c, groups):
    """random + skewed + zero + extreme scalars against the C restatement: hot buckets (one scalar repeated 1 500 and
    15 000 times) go through the hot-bucket queue, all-ones windows exercise the recoding carry across windows."""
    import numpy as np
    from oracle import cref
    n = 40000 + 1234
    rs = np.random.RandomState(3100 + c)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
    sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x0F
    sc[100:1600] = sc[7]               # hot buckets in every window
    sc[21000:36000] = sc[8]            # 15 000 equal scalars
    sc[2000:2300, 2:] = 0              # only the lowest windows populated
    sc[2300:2400] = 0                  # zero scalars
    sc[2400:2500, :31] = 0xFF          # runs of ones: carries ripple through every window
    sc[2500:2600, :16] = 0x80          # windows equal to `half` at c = 8 / 16
    sc[2500:2600, 0] = 0x81
    sc[2600:2700, :] = 0
    sc[2600:2700, 1::2] = 0x80         # 0x8000 in every 16-bit window: digits exactly `half`, no carry
    sc[2600:2700, 31] = 0x08
    table = backend.points_from_uniform(blobs.tobytes())
    backend.set_window_bits(c)
    backend.set_msm_groups(groups)
    try:
        got = backend.vartime_multiscalar_mul(sc.tobytes(), table)
        again = backend.vartime_multiscalar_mul(sc.tobytes(), table)
    finally:
        backend.set_window_bits(0)
        backend.set_msm_groups(0)
        table.free()
    assert got == again
    assert got == cref.msm(sc.tobytes(), cref.from_uniform(blobs.tobytes()))


@pytest.mark.parametrize("log_n", [12, 13])
@pytest.mark.parametrize("groups,tile", [(0, 0), (4, 0), (8, 8), (3, 16)])
def test_hot_buckets_in_every_window_group(backend, log_n, groups, tile):
    """Small inputs in the pipelined / submitted form with hot buckets in EVERY window: each window group queues its own
    hot buckets and the groups' fix-up kernels run concurrently on different streams, so the queues must not share
    memory (ADVICE round 1: at n = 2^12 the per-group regions overlapped).  Several equal scalars repeated ~800 times
    each give every window of every group several hot buckets; submitted twice in flight + joined vs the C restatement."""
    import numpy as np
    import torch
    from oracle import cref
    n = 1 << log_n
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(5200 + log_n)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
    sets = []
    for k in range(3):
        sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
        sc[:, 31] &= 0x0F
        reps = 3 + k
        span = (n - 64) // reps
        for r in range(reps):          # `reps` different scalars, each repeated span times: hot buckets in all windows
            sc[r * span:(r + 1) * span] = sc[n - 1 - r]
        sets.append(sc)
    table = backend.points_from_uniform(blobs.tobytes())
    pts = cref.from_uniform(blobs.tobytes())
    want = [cref.msm(s.tobytes(), pts) for s in sets]
    d_sets = [torch.from_numpy(s).to(dev) for s in sets]
    outs = torch.zeros(3, 160, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    backend.set_msm_groups(groups)
    backend.set_msm_tile(tile)
    try:
        for rep in range(2):
            for i in range(3):
                backend.msm_submit_dev(d_sets[i].data_ptr(), table, 0, n, outs[i].data_ptr())
            backend.msm_wait()
            backend.synchronize()
            for i in range(3):
                assert bytes(outs[i, :32].cpu().numpy().tobytes()) == want[i], (rep, i)
        for i in range(3):
            assert backend.vartime_multiscalar_mul(sets[i].tobytes(), table) == want[i]
    finally:
        backend.set_msm_groups(0)
        backend.set_msm_tile(0)
        table.free()


def test_submitted_partials_sum_to_the_full_result(backend):
    """bpp_msm_submit_partial_dev (the sharded multi-GPU form, here two shards on one GPU): the two submitted
    partials of a split MSM, summed by bpp_points_sum_compress_dev, give the bytes of the one-call MSM."""
    import numpy as np
    import torch
    n = 1 << 15
    rs = np.random.RandomState(515)
    table = backend.points_from_uniform(rs.randint(0, 256, size=(n, 64), dtype=np.uint8).tobytes())
    sc = _np_scalars(n, 616)
    want = backend.vartime_multiscalar_mul(sc.tobytes(), table)
    dev = torch.device("cuda:0")
    d_sc = torch.from_numpy(sc).to(dev)
    parts = torch.zeros(2, 128, dtype=torch.uint8, device=dev)
    out32 = torch.zeros(32, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    h = n // 2 + 37
    backend.set_msm_groups(3)
    try:
        backend.msm_submit_partial_dev(d_sc.data_ptr(), table, 0, h, parts[0].data_ptr())
        backend.msm_submit_partial_dev(d_sc[h:].data_ptr(), table, h, n - h, parts[1].data_ptr())
        backend.msm_wait()
        backend.points_sum_compress_dev(parts.data_ptr(), 2, out32.data_ptr())
        backend.synchronize()
    finally:
        backend.set_msm_groups(0)
    assert bytes(out32.cpu().numpy().tobytes()) == want
    table.free()


@pytest.mark.parametrize("tile,c,groups", [(8, 11, 1), (48, 16, 3), (64, 16, 4), (64, 8, 1), (256, 13, 2)])
def test_tile_lengths_match_oracle(backend, tile, c, groups):
    """bpp_set_msm_tile: the accumulate's tile length (32 by default, 64 for large inputs) with skewed scalars, so that
    buckets span many tiles (the long-bucket queue at tile 8) or many buckets share one tile (tile 256)."""
    import numpy as np
    from oracle import cref
    n = 12000 + 345
    rs = np.random.RandomState(8200 + tile)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8)
    sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x0F
    sc[500:3000] = sc[1]
    sc[4000:4200, 2:] = 0
    table = backend.points_from_uniform(blobs.tobytes())
    backend.set_window_bits(c)
    backend.set_msm_groups(groups)
    backend.set_msm_tile(tile)
    try:
        got = backend.vartime_multiscalar_mul(sc.tobytes(), table)
    finally:
        backend.set_msm_tile(0)
        backend.set_msm_groups(0)
        backend.set_window_bits(0)
        table.free()
    assert got == cref.msm(sc.tobytes(), cref.from_uniform(blobs.tobytes()))


# ---- small and batched MSMs over a precomputed point set (SURVEY 2.3 K5; the reference's call-site sizes) -----------
@pytest.mark.parametrize("n", [2, 105, 209])
@pytest.mark.parametrize("window_bits", [0, 5, 11])
def test_precomputed_points_single_msm_matches_the_bucket_path_and_the_oracle(backend, n, window_bits):
    import numpy as np
    from oracle import cref
    rs = np.random.RandomState(1000 + n + window_bits)
    blobs = rs.randint(0, 256, size=(n + 3, 64), dtype=np.uint8).tobytes()
    pts_c = cref.from_uniform(blobs)
    sc = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x1F                    # up to 2^253: non-canonical values allowed below 2^255
    sc[0] = 0
    scb = sc.tobytes()
    table = backend.points_from_uniform(blobs)
    want = cref.msm(scb, pts_c[160 * 3:160 * (3 + n)])          # a sub-range of the set: points 3 .. 3 + n
    plain = backend.vartime_multiscalar_mul(scb, table, 3, n)
    backend.precompute(table, window_bits)
    l0 = backend.launch_count
    fast = backend.vartime_multiscalar_mul(scb, table, 3, n)
    assert backend.launch_count - l0 <= 3                     # table look-ups + sum + compress: no bucket pipeline
    assert plain == want and fast == want
    table.free()


# count >= 16 per SM (148 SMs): a warp per output, at c = 8 digit-staged (209), scalar-staged (350: the digit stage,
# 50 432 B, exceeds 48 KB) and unstaged (400: the scalar stage, 51 200 B, does too)
@pytest.mark.parametrize("n,count", [(2, 1), (2, 5000), (105, 7), (209, 300), (209, 2500), (33, 1), (350, 2400), (400, 2400)])
def test_batched_msm_over_shared_points_matches_the_c_restatement(backend, n, count):
    import numpy as np
    from oracle import cref
    rs = np.random.RandomState(7 * n + count)
    blobs = rs.randint(0, 256, size=(n, 64), dtype=np.uint8).tobytes()
    pts_c = cref.from_uniform(blobs)
    sc = rs.randint(0, 256, size=(count * n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x0F
    sc[n - 1] = 0
    sc[0, :] = np.frombuffer((R.L - 1).to_bytes(32, "little"), dtype=np.uint8)
    table = backend.points_from_uniform(blobs)
    out = backend.msm_batch(sc.tobytes(), table, n, count)
    assert len(out) == 32 * count
    for i in sorted(set([0, 1 % count, count // 2, count - 1])):
        assert out[32 * i:32 * i + 32] == cref.msm(sc[i * n:(i + 1) * n].tobytes(), pts_c), i
    with pytest.raises(Exception):
        bad = bytearray(sc[:n].tobytes())
        bad[31] |= 0x80                                        # bit 255 set: BPP_ERR_SCALAR_RANGE like the single call
        backend.msm_batch(bytes(bad), table, n, 1)
    table.free()
