"""GPU parity of the mixed MSM (bpp_msm_mixed*): per MSM, a static part over a sub-range of a tabled point set plus a ragged
dynamic part over caller encodings.  The oracle of MSM j is one vartime_multiscalar_mul over its static terms followed by
its dynamic terms (oracle.cref.msm, or R.vartime_multiscalar_mul for edge values): the encoding is unique, so the order in
which the library adds the two parts cannot change the bytes.  The table path (bpp_msm_vartime_batch), the caller-point path
(bpp_msm_multi, bpp_msm_multi_indexed) and the reference's call sites are checked against it as well."""
import ctypes
import random

import pytest

from oracle import acproof as A, cref, ristretto255 as R
from oracle.chacha import ChaChaRng

pytestmark = pytest.mark.gpu
L = R.L
PT = 160   # bytes of one raw point of the C oracle


def _points(n, seed):
    """n random points: (raw points of the C oracle, their encodings)."""
    rng = ChaChaRng(bytes([seed]) * 32)
    raw = cref.from_uniform(rng.fill_bytes(64 * n))
    return raw, cref.compress(raw)


def _scalars(n, rng):
    return b"".join(rng.randrange(0, 2 ** 255).to_bytes(32, "little") if rng.random() < 0.1 else
                    rng.randrange(0, L).to_bytes(32, "little") for _ in range(n))


def _static_set(backend, n, seed, c=None):
    raw, enc = _points(n, seed)
    pts = backend.upload_points(enc)
    if c is not None:
        backend.precompute(pts, c)
    return pts, raw, enc


def _oracle(st_sc, st_raw, n_static, sizes, dy_sc, dy_raw, only=None):
    """MSM j = cref.msm over its n_static static terms, then its dynamic terms.  only: the MSMs to compute (others None)."""
    out, t = [], 0
    for j, n in enumerate(sizes):
        if only is None or j in only:
            sc = st_sc[32 * n_static * j:32 * n_static * (j + 1)] + dy_sc[32 * t:32 * (t + n)]
            out.append(cref.msm(sc, st_raw + dy_raw[PT * t:PT * (t + n)]))
        else:
            out.append(None)
        t += n
    return out


def _dynamic(sizes, seed):
    rng = random.Random(seed)
    T = sum(sizes)
    raw, enc = _points(max(T, 1), seed & 0xff)
    return _scalars(T, rng), raw[:PT * T], enc[:32 * T]


def test_ragged_batch_and_permutation(backend):
    """Dynamic sizes on both sides of every size class, one 8192-term MSM among thousands of small ones, a static part over
    a sub-range (off > 0); then the same MSMs in another order."""
    rng = random.Random(1)
    off, n_static = 5, 12
    pts, raw, _ = _static_set(backend, 40, 21, 8)
    sizes = [0, 1, 2, 31, 32, 33, 1023, 1024, 1025] * 2 + [8192] + [rng.choice((0, 1, 2, 3)) for _ in range(2000)]
    rng.shuffle(sizes)
    st = _scalars(len(sizes) * n_static, rng)
    dy, dy_raw, dy_enc = _dynamic(sizes, 31)
    want = _oracle(st, raw[PT * off:PT * (off + n_static)], n_static, sizes, dy, dy_raw)
    got, ok = backend.msm_mixed(st, pts, n_static, dy, dy_enc, sizes, off)
    assert ok == [True] * len(sizes)
    assert got == want
    starts = [sum(sizes[:j]) for j in range(len(sizes))]
    perm = list(range(len(sizes)))
    rng.shuffle(perm)
    sizes_p = [sizes[j] for j in perm]
    st_p = b"".join(st[32 * n_static * j:32 * n_static * (j + 1)] for j in perm)
    dy_p = b"".join(dy[32 * starts[j]:32 * (starts[j] + sizes[j])] for j in perm)
    enc_p = b"".join(dy_enc[32 * starts[j]:32 * (starts[j] + sizes[j])] for j in perm)
    got_p, ok_p = backend.msm_mixed(st_p, pts, n_static, dy_p, enc_p, sizes_p, off)
    assert all(ok_p) and got_p == [want[j] for j in perm]


@pytest.mark.parametrize("c", [4, 5, 8, 11, 16])
def test_every_table_width_and_the_table_path(backend, c):
    """The static part at every width a set can carry, in the table kernels' block form (few MSMs, split partials) and warp
    form (many MSMs); sizes == 0 everywhere gives bpp_msm_vartime_batch's bytes.  c = 16 on a small set: 48 MiB per point."""
    rng = random.Random(c)
    n_set, off, n_static = (6, 1, 5) if c == 16 else (48, 7, 30)
    pts, raw, _ = _static_set(backend, n_set, 40 + c, c)
    st_raw = raw[PT * off:PT * (off + n_static)]
    for count in (200, 2600):
        sizes = [rng.choice((0, 1, 2, 5, 40)) for _ in range(count)]
        st = _scalars(count * n_static, rng)
        dy, dy_raw, dy_enc = _dynamic(sizes, 7 * c + count)
        sample = set(range(0, count, max(1, count // 150)))
        want = _oracle(st, st_raw, n_static, sizes, dy, dy_raw, only=sample)
        got, ok = backend.msm_mixed(st, pts, n_static, dy, dy_enc, sizes, off)
        assert all(ok)
        assert [got[j] for j in sorted(sample)] == [want[j] for j in sorted(sample)], (c, count)
        table = backend.msm_batch(st, pts, n_static, count, off)
        got0, ok0 = backend.msm_mixed(st, pts, n_static, b"", b"", [0] * count, off)
        assert all(ok0) and b"".join(got0) == table, (c, count)


@pytest.mark.parametrize("c", [5, 8, 16])
def test_edge_scalars_in_both_parts(backend, c):
    """0, 1, l - 1 and 2^255 - 1 (the largest accepted value; at c = 8 and c = 16 it drives the top digit to exactly
    2^(c-1)) in the static and the dynamic part."""
    special = [0, 1, L - 1, 2 ** 255 - 1]
    n_set = 4
    _, enc = _points(n_set, 90 + c)
    pts = backend.upload_points(enc)
    backend.precompute(pts, c)
    st_pts = [R.decompress(enc[32 * i:32 * i + 32]) for i in range(n_set)]
    P1, P2 = R.pt_mul(7, R.BASEPOINT), R.from_uniform_bytes(bytes(range(64)))
    rows, calls = [], []
    for a in special:
        for b in special:
            rows.append([a, b, a, b])
            calls.append(([b, a, 3], [P1, P2, P1]))
    rows.append([2 ** 255 - 1] * n_set)
    calls.append(([2 ** 255 - 1] * 2, [P2, P2]))
    rows.append([L - 1] * n_set)
    calls.append(([1], [st_pts[0]]))                  # a dynamic point equal to a static one
    st = b"".join(s.to_bytes(32, "little") for r in rows for s in r)
    dy = b"".join(s.to_bytes(32, "little") for ss, _ in calls for s in ss)
    enc_d = b"".join(R.compress(p) for _, pp in calls for p in pp)
    sizes = [len(ss) for ss, _ in calls]
    want = [R.compress(R.vartime_multiscalar_mul([s % L for s in r + ss], st_pts + pp)) for r, (ss, pp) in zip(rows, calls)]
    got, ok = backend.msm_mixed(st, pts, n_set, dy, enc_d, sizes)
    assert all(ok) and got == want
    got0, _ = backend.msm_mixed(st, pts, n_set, b"", b"", [0] * len(rows))
    assert b"".join(got0) == backend.msm_batch(st, pts, n_set, len(rows))


def test_zero_static_scalars_give_msm_multi(backend):
    sizes = [0, 1, 2, 31, 33, 209, 1025, 3]
    pts, _, _ = _static_set(backend, 20, 61, 8)
    dy, _, dy_enc = _dynamic(sizes, 62)
    want, want_ok = backend.msm_multi(dy, dy_enc, sizes)
    got, ok = backend.msm_mixed(bytes(32 * 20 * len(sizes)), pts, 20, dy, dy_enc, sizes)
    assert ok == want_ok == [True] * len(sizes) and got == want


def test_verifier_shape_equals_the_indexed_path(backend):
    """4096 x (209 generators + 8 proof points): the mixed call against bpp_msm_multi_indexed over a set holding the
    generators and the proof points (GPU to GPU), plus oracle spot checks."""
    count, n_static, n_dyn, pool = 4096, 209, 8, 512
    rng = random.Random(209)
    g_raw, g_enc = _points(n_static, 71)
    p_raw, p_enc = _points(pool, 72)
    gens = backend.upload_points(g_enc)
    both = backend.upload_points(g_enc + p_enc)
    st = _scalars(count * n_static, rng)
    dy = _scalars(count * n_dyn, rng)
    pick = [rng.randrange(pool) for _ in range(count * n_dyn)]
    dy_enc = b"".join(p_enc[32 * i:32 * i + 32] for i in pick)
    got, ok = backend.msm_mixed(st, gens, n_static, dy, dy_enc, [n_dyn] * count)
    assert all(ok)
    sc = b"".join(st[32 * n_static * j:32 * n_static * (j + 1)] + dy[32 * n_dyn * j:32 * n_dyn * (j + 1)] for j in range(count))
    index = [i for j in range(count) for i in list(range(n_static)) + [n_static + p for p in pick[n_dyn * j:n_dyn * (j + 1)]]]
    assert got == backend.msm_multi_indexed(sc, both, index, [n_static + n_dyn] * count)
    for j in (0, 1, 2047, 4095):
        dy_raw = b"".join(p_raw[PT * i:PT * (i + 1)] for i in pick[n_dyn * j:n_dyn * (j + 1)])
        assert got[j] == cref.msm(sc[32 * (n_static + n_dyn) * j:32 * (n_static + n_dyn) * (j + 1)], g_raw + dy_raw), j


def test_bad_encoding_fails_only_its_own_msm(backend):
    from test_gpu_decode import _invalid_encodings
    bad = [e for v in _invalid_encodings().values() for e in v]
    rng = random.Random(5)
    n_static = 16
    pts, raw, _ = _static_set(backend, n_static, 81, 8)
    sizes = [3, 40, 2, 200, 700, 1, 2500, 5] * 4
    st = _scalars(len(sizes) * n_static, rng)   # every MSM has a non-zero static part
    dy, dy_raw, dy_enc = _dynamic(sizes, 82)
    want = _oracle(st, raw, n_static, sizes, dy, dy_raw)
    starts = [sum(sizes[:j]) for j in range(len(sizes))]
    encl = bytearray(dy_enc)
    spoiled = set()
    for i, e in enumerate(bad):
        j = (3 * i + 1) % len(sizes)
        t = starts[j] + rng.randrange(sizes[j])
        encl[32 * t:32 * t + 32] = e
        spoiled.add(j)
    got, ok = backend.msm_mixed(st, pts, n_static, dy, bytes(encl), sizes)
    for j in range(len(sizes)):
        if j in spoiled:
            assert not ok[j] and got[j] == bytes(32), j
        else:
            assert ok[j] and got[j] == want[j], j


def test_errors_leave_the_outputs_untouched(backend):
    lib, ctx = backend._lib, backend._ctx
    n_set, n_static = 10, 4
    pts, _, _ = _static_set(backend, n_set, 91, 8)
    sizes = [2, 3]
    arr = (ctypes.c_uint32 * 2)(*sizes)
    rng = random.Random(3)
    st = _scalars(2 * n_static, rng)
    dy, _, enc = _dynamic(sizes, 92)
    out, ok = ctypes.create_string_buffer(b"\xa5" * 64, 64), ctypes.create_string_buffer(b"\x5a" * 2, 2)

    def untouched():
        return out.raw == b"\xa5" * 64 and ok.raw == b"\x5a" * 2

    def mixed(count=2, points=pts._h, off=0, n=n_static, s=st, z=arr, d=dy, e=enc, o=out, k=ok):
        return lib.bpp_msm_mixed(ctx, count, points, off, n, s, z, d, e, o, k)

    assert mixed() == 0 and not untouched()   # the arguments below differ from a valid call in one place each
    out.raw, ok.raw = b"\xa5" * 64, b"\x5a" * 2
    for kw in ({"s": None}, {"z": None}, {"d": None}, {"e": None}, {"o": None}, {"k": None}, {"points": None},
               {"count": 0}, {"n": 0}, {"z": (ctypes.c_uint32 * 2)(2 ** 31 - 1, 1)}):
        assert mixed(**kw) == -3, kw
    assert lib.bpp_msm_mixed(None, 2, pts._h, 0, n_static, st, arr, dy, enc, out, ok) == -3
    assert mixed(off=n_set - n_static + 1) == -4
    assert mixed(off=n_set + 1) == -4
    assert mixed(n=n_set + 1) == -4
    for region, t in (("s", 5), ("d", 4)):
        high = bytearray(st if region == "s" else dy)
        high[32 * t + 31] |= 0x80
        assert mixed(**{region: bytes(high)}) == -6, region
    # count x n_static >= 2^31: refused before the scalars are read
    assert lib.bpp_msm_mixed(ctx, 2 ** 16, pts._h, 0, 2 ** 15, st, (ctypes.c_uint32 * 2 ** 16)(), dy, enc, out, ok) == -3
    assert untouched()

    def mixed_dev(count=2, points=pts._h, off=0, n=n_static, s=1, z=arr, d=1, e=1, o=1, k=1):
        return lib.bpp_msm_mixed_dev(ctx, count, points, off, n, s, z, d, e, o, k)

    for kw in ({"s": None}, {"z": None}, {"d": None}, {"e": None}, {"o": None}, {"k": None}, {"points": None},
               {"count": 0}, {"n": 0}, {"z": (ctypes.c_uint32 * 2)(2 ** 31 - 1, 1)}):
        assert mixed_dev(**kw) == -3, kw
    assert mixed_dev(off=n_set - n_static + 1) == -4
    assert mixed_dev(n=n_set + 1) == -4


def test_launches_are_bounded_and_independent_of_count(backend):
    """A fixed handful of launches whatever count is: the table part (1), decode, Straus, Pippenger and the finish kernel.
    A static part over more than FB_THREADS work items at few MSMs takes the table kernels' split partials and their sum
    kernel (one launch more), as bpp_msm_vartime_batch does; 16 terms at c = 8 are 128 items, one block per MSM.  The
    operation counts report both parts."""
    pts, _, _ = _static_set(backend, 209, 101, 8)
    rng = random.Random(8)

    def launches(count, n_static):
        sizes = [(3, 40, 0, 2)[j % 4] for j in range(count)]
        st = _scalars(count * n_static, rng)
        dy, _, dy_enc = _dynamic(sizes, 102)
        backend.msm_mixed(st, pts, n_static, dy, dy_enc, sizes)   # warm-up: arena growth
        l0 = backend.launch_count
        backend.msm_mixed(st, pts, n_static, dy, dy_enc, sizes)
        n = backend.launch_count - l0
        ops = backend.last_op_counts()
        backend.msm_multi(dy, dy_enc, sizes)
        dyn_ops = backend.last_op_counts()
        assert ops["mixed_adds"] == dyn_ops["mixed_adds"] + count * n_static * 32
        assert ops["doublings"] == dyn_ops["doublings"] and ops["full_adds"] > dyn_ops["full_adds"] + count
        return n

    assert launches(4, 16) == launches(4096, 16) == 5
    assert launches(4, 209) <= 6 and launches(4096, 209) == 5


def test_reference_call_sites_in_one_call(backend):
    """Every vartime_multiscalar_mul of the reference's prover and verifier for 3-, 5- and 52-card proofs, recorded from the
    oracle's flow.  The points of a call that belong to the generator sets (g, h, G_vec, H_vec of every instance, one
    resident set) go into the static part, at their set position; the others into the dynamic part.  Replayed as one
    bpp_msm_mixed."""
    calls = []

    def recording_msm(scalars, points):
        scalars, points = list(scalars), list(points)
        enc = b"".join(R.compress(p) for p in points)
        sb = b"".join(R.sc_bytes(s % L) for s in scalars)
        out = cref.msm(sb, cref.decompress(enc))
        calls.append(([s % L for s in scalars], [R.compress(p) for p in points], out))
        return R.decompress(out) if out != bytes(32) else R.IDENTITY

    set_enc, where = [], {}
    for k, seed in ((3, 1), (3, 2), (5, 3), (52, 4)):
        rng = ChaChaRng(bytes([60 + seed]) * 32)
        core, prover, V = A.make_instance(k, rng)
        for p in [core["g_base"], core["h_base"]] + list(core["G_vec"]) + list(core["H_vec"]):
            e = R.compress(p)
            if e not in where:
                where[e] = len(set_enc)
                set_enc.append(e)
        _, ok, _, _ = A.run_flow(core, prover, V, ChaChaRng(bytes([seed]) * 32), "reference-fixed", b"test", recording_msm)
        assert ok
    assert len(calls) == 4 * 15
    n_static = len(set_enc)
    pts = backend.upload_points(b"".join(set_enc))
    st, dy, dy_enc, sizes = bytearray(), bytearray(), bytearray(), []
    n_mixed = 0
    for scalars, encs, _ in calls:
        row = [0] * n_static
        n_dyn = 0
        for s, e in zip(scalars, encs):
            if e in where:
                row[where[e]] = (row[where[e]] + s) % L
            else:
                dy += s.to_bytes(32, "little")
                dy_enc += e
                n_dyn += 1
        n_mixed += 0 < n_dyn < len(encs)
        st += b"".join(s.to_bytes(32, "little") for s in row)
        sizes.append(n_dyn)
    assert n_mixed >= 4   # the verifier's sites carry both kinds
    got, ok = backend.msm_mixed(bytes(st), pts, n_static, bytes(dy), bytes(dy_enc), sizes)
    assert all(ok)
    assert got == [o for _, _, o in calls]


def test_dev_form_on_a_torch_stream(backend):
    """Device pointers on the context's (torch) stream, with work queued ahead of the call: the results equal the host
    form's, the ok bytes land in device memory, and bit 255 of a device scalar is read as zero in both parts."""
    import torch
    import bpperm_b200
    sizes = [0, 2, 31, 33, 105, 209, 700, 3000, 1]
    count, n_static, off = len(sizes), 24, 3
    rng = random.Random(12)
    st = _scalars(count * n_static, rng)
    dy, _, dy_enc = _dynamic(sizes, 13)
    be = bpperm_b200.Backend(0)   # a context of its own: set_stream is for the life of a context
    try:
        _, enc = _points(off + n_static, 14)
        pts = be.upload_points(enc)
        want, _ = be.msm_mixed(st, pts, n_static, dy, dy_enc, sizes, off)   # builds the c = 8 table on first use
        st_hi, dy_hi = bytearray(st), bytearray(dy)
        for buf in (st_hi, dy_hi):
            for t in range(0, len(buf) // 32, 5):
                buf[32 * t + 31] |= 0x80
        stream = torch.cuda.Stream()
        be.set_stream(stream.cuda_stream)
        blob = bytes(st_hi) + bytes(dy_hi) + dy_enc
        host = torch.frombuffer(bytearray(blob), dtype=torch.uint8).pin_memory()
        with torch.cuda.stream(stream):
            d_in = torch.zeros(len(blob), dtype=torch.uint8, device="cuda")
            torch.cuda._sleep(1 << 22)                      # queued work ahead of the inputs and the call
            d_in.copy_(host, non_blocking=True)
            d_out = torch.full((32 * count,), 0xa5, dtype=torch.uint8, device="cuda")
            d_ok = torch.zeros(count, dtype=torch.uint8, device="cuda")
            base = d_in.data_ptr()
            be.msm_mixed_dev(pts, n_static, base, sizes, base + len(st), base + len(st) + len(dy), d_out.data_ptr(),
                             d_ok.data_ptr(), off)
        stream.synchronize()
        assert d_ok.device.type == "cuda" and d_ok.cpu().tolist() == [1] * count
        got = bytes(d_out.cpu().numpy())
        assert [got[32 * j:32 * j + 32] for j in range(count)] == want
    finally:
        be.close()
