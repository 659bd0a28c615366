"""GPU parity of the batched variable-base MSM (bpp_msm_multi*): `count` independent MSMs with ragged sizes, each over its
own points, against the oracle - the C restatement (oracle.cref.msm) for batches and large MSMs, R.vartime_multiscalar_mul
for the edge values - and against the table path (bpp_msm_vartime_batch) over the same points."""
import ctypes
import random

import pytest

from oracle import acproof as A, cref, ristretto255 as R
from oracle.chacha import ChaChaRng

pytestmark = pytest.mark.gpu
L = R.L

# size-class boundaries of csrc/msm_multi_kernels.cuh: Straus up to 32 terms, Pippenger above, split into chunks of 1024
STRAUS_MAX, CHUNK = 32, 1024


def _points(n, seed):
    """n random points: (raw points of the C oracle, their encodings)."""
    rng = ChaChaRng(bytes([seed]) * 32)
    raw = cref.from_uniform(rng.fill_bytes(64 * n))
    return raw, cref.compress(raw)


def _scalars(n, rng):
    return b"".join(rng.randrange(0, 2 ** 255).to_bytes(32, "little") if rng.random() < 0.1 else
                    rng.randrange(0, L).to_bytes(32, "little") for _ in range(n))


def _oracle_batch(sizes, sc, raw):
    out, t = [], 0
    for n in sizes:
        out.append(cref.msm(sc[32 * t:32 * (t + n)], raw[160 * t:160 * (t + n)]) if n else bytes(32))
        t += n
    return out


def _batch(sizes, seed):
    rng = random.Random(seed)
    T = sum(sizes)
    raw, enc = _points(max(T, 1), seed & 0xff)
    return _scalars(T, rng), raw[:160 * T], enc[:32 * T]


def test_ragged_batch_both_forms_and_permutation(backend):
    rng = random.Random(1)
    sizes = [0, 1, 2, 3, 17, 104, 105, 110, 111, 209, 600, 4096] * 3
    rng.shuffle(sizes)
    sc, raw, enc = _batch(sizes, 11)
    want = _oracle_batch(sizes, sc, raw)
    got, ok = backend.msm_multi(sc, enc, sizes)
    assert ok == [True] * len(sizes)
    assert got == want
    pts = backend.upload_points(enc)
    assert backend.msm_multi_indexed(sc, pts, list(range(sum(sizes))), sizes) == want
    # the same MSMs in another order: the results follow them
    starts = [sum(sizes[:j]) for j in range(len(sizes))]
    perm = list(range(len(sizes)))
    rng.shuffle(perm)
    sizes_p = [sizes[j] for j in perm]
    sc_p = b"".join(sc[32 * starts[j]:32 * (starts[j] + sizes[j])] for j in perm)
    enc_p = b"".join(enc[32 * starts[j]:32 * (starts[j] + sizes[j])] for j in perm)
    got_p, ok_p = backend.msm_multi(sc_p, enc_p, sizes_p)
    assert all(ok_p) and got_p == [want[j] for j in perm]


@pytest.mark.parametrize("n", [b + d for b in (STRAUS_MAX, CHUNK, 2 * CHUNK) for d in (-1, 0, 1)])
def test_size_class_boundaries(backend, n):
    sizes = [n, 2, n, 1]
    sc, raw, enc = _batch(sizes, n)
    want = _oracle_batch(sizes, sc, raw)
    got, ok = backend.msm_multi(sc, enc, sizes)
    assert all(ok) and got == want
    pts = backend.upload_points(enc)
    assert backend.msm_multi_indexed(sc, pts, list(range(sum(sizes))), sizes) == want


def test_large_msm_among_many_two_term_msms(backend):
    sizes = [2] * 2048 + [8192] + [2] * 2048
    sc, raw, enc = _batch(sizes, 81)
    want = _oracle_batch(sizes, sc, raw)
    got, ok = backend.msm_multi(sc, enc, sizes)
    assert all(ok) and got == want


def test_edge_values(backend):
    G = R.BASEPOINT
    P1, P2 = R.pt_mul(7, G), R.from_uniform_bytes(bytes(range(64)))
    special = [0, 1, L - 1, 2 ** 252, L - 2 ** 128, 2 ** 255 - 1 - 2 ** 254]
    calls = [
        (special, [P1, P2, G, P1, P2, G]),                          # every special scalar, repeated points
        ([5, 9], [R.IDENTITY, P1]),                                 # the identity point
        ([3, 3, 3], [P2, P2, P2]),                                  # one point three times
        ([12345, L - 12345], [P1, P1]),                             # s P + (-s) P = identity
        ([0] * 40, [P1] * 20 + [P2] * 20),                          # all-zero scalars (Straus and Pippenger)
        ([0] * 200, [P2] * 200),
        ([2 ** 255 - 1 - 2 ** 254] * 40, [P1, P2] * 20),            # non-canonical scalars, Pippenger
        ([L - 1] * 1100, [P2] * 1100),                              # two chunks
    ]
    sizes = [len(s) for s, _ in calls]
    sc = b"".join(s.to_bytes(32, "little") for ss, _ in calls for s in ss)
    enc = b"".join(R.compress(p) for _, pp in calls for p in pp)
    want = [R.compress(R.vartime_multiscalar_mul([s % L for s in ss], pp)) if len(ss) <= 6 else
            cref.msm(b"".join(s.to_bytes(32, "little") for s in ss), cref.decompress(b"".join(R.compress(p) for p in pp)))
            for ss, pp in calls]
    got, ok = backend.msm_multi(sc, enc, sizes)
    assert all(ok) and got == want
    assert got[3] == bytes(32) and got[4] == bytes(32) and got[5] == bytes(32)


def test_decode_failure_zeroes_only_its_own_msm(backend):
    from test_gpu_decode import _invalid_encodings
    bad = [e for v in _invalid_encodings().values() for e in v]
    rng = random.Random(5)
    sizes = [3, 40, 2, 200, 700, 1, 2500, 5] * 4
    sc, raw, enc = _batch(sizes, 77)
    want = _oracle_batch(sizes, sc, raw)
    starts = [sum(sizes[:j]) for j in range(len(sizes))]
    encl = bytearray(enc)
    spoiled = {}
    for i, e in enumerate(bad):   # every invalid class into a different MSM, at a random term
        j = (3 * i + 1) % len(sizes)
        t = starts[j] + rng.randrange(sizes[j])
        encl[32 * t:32 * t + 32] = e
        spoiled[j] = True
    got, ok = backend.msm_multi(sc, bytes(encl), sizes)
    for j in range(len(sizes)):
        if j in spoiled:
            assert not ok[j] and got[j] == bytes(32), j
        else:
            assert ok[j] and got[j] == want[j], j


def test_errors_leave_the_outputs_untouched(backend):
    lib, ctx = backend._lib, backend._ctx
    sizes = [2, 3]
    arr = (ctypes.c_uint32 * 2)(*sizes)
    sc, raw, enc = _batch(sizes, 3)
    pts = backend.upload_points(enc)
    out, ok = ctypes.create_string_buffer(b"\xa5" * 64, 64), ctypes.create_string_buffer(b"\x5a" * 2, 2)

    def untouched():
        return out.raw == b"\xa5" * 64 and ok.raw == b"\x5a" * 2

    high = bytearray(sc)
    high[32 * 4 + 31] |= 0x80
    assert lib.bpp_msm_multi(ctx, 2, arr, bytes(high), enc, out, ok) == -6
    assert lib.bpp_msm_multi_indexed(ctx, 2, arr, bytes(high), pts._h, (ctypes.c_uint32 * 5)(0, 1, 2, 3, 4), out) == -6
    assert lib.bpp_msm_multi_indexed(ctx, 2, arr, sc, pts._h, (ctypes.c_uint32 * 5)(0, 1, 2, 5, 4), out) == -4
    assert lib.bpp_msm_multi(ctx, 0, arr, sc, enc, out, ok) == -3
    assert lib.bpp_msm_multi(ctx, 2, None, sc, enc, out, ok) == -3
    assert lib.bpp_msm_multi(ctx, 2, arr, None, enc, out, ok) == -3
    assert lib.bpp_msm_multi(ctx, 2, arr, sc, None, out, ok) == -3
    assert lib.bpp_msm_multi(ctx, 2, arr, sc, enc, out, None) == -3
    assert lib.bpp_msm_multi_indexed(ctx, 2, arr, sc, None, (ctypes.c_uint32 * 5)(0, 1, 2, 3, 4), out) == -3
    assert lib.bpp_msm_multi_indexed(ctx, 2, arr, sc, pts._h, None, out) == -3
    assert lib.bpp_msm_multi_dev(ctx, 0, arr, 1, 1, 1, 1) == -3
    assert lib.bpp_msm_multi_dev(ctx, 2, arr, None, 1, 1, 1) == -3
    assert lib.bpp_msm_multi_indexed_dev(ctx, 2, arr, 1, pts._h, None, 1) == -3
    huge = (ctypes.c_uint32 * 2)(2 ** 31 - 1, 1)
    assert lib.bpp_msm_multi_dev(ctx, 2, huge, 1, 1, 1, 1) == -3
    assert untouched()


@pytest.mark.parametrize("n", [105, 209])
def test_indexed_form_equals_the_table_path(backend, n):
    count, off = 4096, 3
    rng = random.Random(n)
    _, enc = _points(off + n, 40)
    pts = backend.upload_points(enc)
    backend.precompute(pts)
    sc = _scalars(count * n, rng)
    want = backend.msm_batch(sc, pts, n, count, off)
    got = backend.msm_multi_indexed(sc, pts, [off + i for _ in range(count) for i in range(n)], [n] * count)
    assert got == [want[32 * j:32 * j + 32] for j in range(count)]


def test_reference_call_sites_in_one_call(backend):
    """Every vartime_multiscalar_mul of the reference's prover and verifier (all 15 sites, h_, T_i and V included) for
    3-, 5- and 52-card proofs, recorded from the oracle's flow and replayed as one bpp_msm_multi."""
    calls = []

    def recording_msm(scalars, points):
        scalars, points = list(scalars), list(points)
        enc = b"".join(R.compress(p) for p in points)
        sb = b"".join(R.sc_bytes(s % L) for s in scalars)
        out = cref.msm(sb, cref.decompress(enc))
        calls.append((sb, enc, out))
        return R.decompress(out) if out != bytes(32) else R.IDENTITY

    for k, seed in ((3, 1), (3, 2), (5, 3), (52, 4)):
        rng = ChaChaRng(bytes([60 + seed]) * 32)
        core, prover, V = A.make_instance(k, rng)
        _, ok, _, _ = A.run_flow(core, prover, V, ChaChaRng(bytes([seed]) * 32), "reference-fixed", b"test", recording_msm)
        assert ok
    assert len(calls) == 4 * 15
    sizes = [len(e) // 32 for _, e, _ in calls]
    got, ok = backend.msm_multi(b"".join(s for s, _, _ in calls), b"".join(e for _, e, _ in calls), sizes)
    assert all(ok)
    assert got == [o for _, _, o in calls]


def test_dev_forms_on_torch_tensors(backend):
    """Device pointers on the context's (torch) stream, with work queued ahead of the call: the results equal the host
    forms', and the ok bytes land in device memory."""
    import torch
    import bpperm_b200
    sizes = [0, 2, 31, 33, 105, 209, 700, 3000, 1]
    sc, raw, enc = _batch(sizes, 9)
    want, _ = backend.msm_multi(sc, enc, sizes)
    be = bpperm_b200.Backend(0)   # a context of its own: set_stream is for the life of a context
    try:
        pts = be.upload_points(enc)
        assert be.msm_multi_indexed(sc, pts, list(range(sum(sizes))), sizes) == want
        stream = torch.cuda.Stream()
        be.set_stream(stream.cuda_stream)
        host = torch.frombuffer(bytearray(sc + enc), dtype=torch.uint8).pin_memory()
        with torch.cuda.stream(stream):
            d_in = torch.zeros(len(sc) + len(enc), dtype=torch.uint8, device="cuda")
            torch.cuda._sleep(1 << 22)                      # queued work ahead of the inputs and the call
            d_in.copy_(host, non_blocking=True)
            d_out = torch.full((32 * len(sizes),), 0xa5, dtype=torch.uint8, device="cuda")
            d_ok = torch.zeros(len(sizes), dtype=torch.uint8, device="cuda")
            be.msm_multi_dev(sizes, d_in.data_ptr(), d_in.data_ptr() + len(sc), d_out.data_ptr(), d_ok.data_ptr())
            d_ix = torch.arange(sum(sizes), dtype=torch.int32, device="cuda")
            d_out2 = torch.zeros(32 * len(sizes), dtype=torch.uint8, device="cuda")
            be.msm_multi_indexed_dev(sizes, d_in.data_ptr(), pts, d_ix.data_ptr(), d_out2.data_ptr())
        stream.synchronize()
        assert d_ok.device.type == "cuda" and d_ok.cpu().tolist() == [1] * len(sizes)
        got = bytes(d_out.cpu().numpy())
        assert [got[32 * j:32 * j + 32] for j in range(len(sizes))] == want
        got2 = bytes(d_out2.cpu().numpy())
        assert [got2[32 * j:32 * j + 32] for j in range(len(sizes))] == want
    finally:
        be.close()
