"""Host-side handle on the CUDA backend: the Python mirror of the reference's operator boundary.

`Backend.vartime_multiscalar_mul(scalars, points)` has the argument meaning and error behaviour of
`RistrettoPoint::vartime_multiscalar_mul` (dalek-ng 4.1.1 traits.rs; called at
/root/reference/bp-perm/src/circuit_lib.rs:187-568): equal-length iterables of scalars and points,
a length mismatch is an error (dalek asserts), an undecodable point is an error (dalek:
`decompress().unwrap()` panics, circuit_lib.rs:532), the result is one Ristretto point - returned
here in its canonical 32-byte encoding.
"""
from __future__ import annotations

import array
import ctypes
import weakref
from typing import Iterable, Sequence, Union

from . import _lib

FMT_COMPRESSED, FMT_AFFINE, FMT_DALEK_XYZT = 0, 1, 2
_FMT_BYTES = {FMT_COMPRESSED: 32, FMT_AFFINE: 64, FMT_DALEK_XYZT: 160}
PHASES = ["recode", "scan", "scatter", "accumulate", "reduce", "finish"]

ScalarLike = Union[int, bytes]


def scalars_to_bytes(scalars: Iterable[ScalarLike]) -> bytes:
    out = bytearray()
    for s in scalars:
        if isinstance(s, int):
            out += s.to_bytes(32, "little")
        else:
            if len(s) != 32:
                raise ValueError("scalar must be 32 bytes")
            out += s
    return bytes(out)


class Points:
    """Device-resident point table (affine Niels); upload once, reuse across MSMs."""

    def __init__(self, backend: "Backend", handle: int, n: int):
        self._backend, self._h, self.n = backend, handle, n
        backend._adopt(self)

    def __len__(self):
        return self.n

    def free(self):
        if self._h and self._backend._ctx:
            self._backend._lib.bpp_points_free(self._backend._ctx, self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Backend:
    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        ctx = ctypes.c_void_p()
        rc = self._lib.bpp_init(device, ctypes.byref(ctx))
        if rc != 0:
            raise _lib.BppError(rc, self._lib.bpp_strerror(rc).decode())
        self._ctx = ctx
        self.device = device
        self._children = weakref.WeakSet()   # device objects created on this context: freed before it

    def _adopt(self, child):
        self._children.add(child)

    # -- plumbing -------------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            detail = self._lib.bpp_last_error(self._ctx).decode() if rc == -2 else ""
            raise _lib.BppError(rc, self._lib.bpp_strerror(rc).decode() + (": " + detail if detail else ""))

    def close(self):
        if self._ctx:
            for child in list(self._children):
                try:
                    child.free()
                except Exception:
                    pass
            self._lib.bpp_free(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int):
        self._check(self._lib.bpp_set_stream(self._ctx, ctypes.c_void_p(cuda_stream)))

    def synchronize(self):
        self._check(self._lib.bpp_synchronize(self._ctx))

    @property
    def launch_count(self) -> int:
        return int(self._lib.bpp_launch_count(self._ctx))

    def device_info(self):
        sm, ma, mi, mem = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_size_t()
        self._check(self._lib.bpp_device_info(self._ctx, ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi),
                                              ctypes.byref(mem)))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "total_mem": mem.value,
                "clock_khz": int(self._lib.bpp_device_clock_khz(self._ctx))}

    def imad_pipe_limit(self) -> float:
        """IMAD.WIDE.U32 issue limit in ops/s: one warp instruction per 4 clocks per SM sub-partition
        (= 32 lanes/clk/SM; ncu: fmaheavy cycles per IMAD.WIDE = 4.0, profiles/r1_imad_rate.md) at the
        maximum SM clock.  The roofline denominator for every IMAD-bound kernel."""
        info = self.device_info()
        return info["sm_count"] * 32.0 * info["clock_khz"] * 1e3

    def set_window_bits(self, c: int):
        self._check(self._lib.bpp_set_window_bits(self._ctx, c))

    def set_msm_groups(self, groups: int):
        """Window groups of the pipelined MSM (0 = automatic, 1 = in order on one stream)."""
        self._check(self._lib.bpp_set_msm_groups(self._ctx, groups))

    def set_msm_tile(self, tile_len: int):
        """Entries per accumulate tile (0 = by input size)."""
        self._check(self._lib.bpp_set_msm_tile(self._ctx, tile_len))

    def set_msm_partition(self, sizes):
        """Explicit window-group sizes, top group first (empty = clear)."""
        arr = (ctypes.c_int * max(1, len(sizes)))(*sizes)
        self._check(self._lib.bpp_set_msm_partition(self._ctx, arr, len(sizes)))

    def set_msm_trace(self, on: bool):
        self._check(self._lib.bpp_set_msm_trace(self._ctx, int(on)))

    def msm_trace(self) -> str:
        """Stage timeline of the last MSM (see bpp_msm_trace_dump)."""
        buf = ctypes.create_string_buffer(1 << 16)
        self._check(self._lib.bpp_msm_trace_dump(self._ctx, buf, len(buf)))
        return buf.value.decode()

    def set_profiling(self, on: bool):
        self._check(self._lib.bpp_set_profiling(self._ctx, int(on)))

    def last_phase_ms(self):
        arr = (ctypes.c_float * len(PHASES))()
        self._check(self._lib.bpp_last_phase_ms(self._ctx, arr))
        return dict(zip(PHASES, [float(x) for x in arr]))

    def last_op_counts(self):
        m, a, d = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        self._check(self._lib.bpp_last_op_counts(self._ctx, ctypes.byref(m), ctypes.byref(a), ctypes.byref(d)))
        return {"mixed_adds": m.value, "full_adds": a.value, "doublings": d.value}

    def imad_peak(self, iters: int = 4096):
        ops, ms = ctypes.c_double(), ctypes.c_double()
        self._check(self._lib.bpp_bench_imad_peak(self._ctx, iters, ctypes.byref(ops), ctypes.byref(ms)))
        return ops.value, ms.value

    def pipe_probe(self, mode: int, iters: int = 2048) -> float:
        ops = ctypes.c_double()
        self._check(self._lib.bpp_bench_pipe_probe(self._ctx, mode, iters, ctypes.byref(ops)))
        return ops.value

    # -- points ---------------------------------------------------------------------------------
    def upload_points(self, pts: Union[bytes, Sequence[bytes]], fmt: int = FMT_COMPRESSED) -> Points:
        if not isinstance(pts, (bytes, bytearray)):
            pts = b"".join(pts)
        eb = _FMT_BYTES[fmt]
        if len(pts) % eb:
            raise ValueError("point buffer length is not a multiple of the format size")
        n = len(pts) // eb
        h = ctypes.c_void_p()
        self._check(self._lib.bpp_points_upload(self._ctx, fmt, bytes(pts), n, ctypes.byref(h)))
        return Points(self, h, n)

    def points_from_uniform(self, bytes64: bytes) -> Points:
        """RistrettoPoint::from_uniform_bytes over n x 64 bytes (RistrettoPoint::random with an RNG stream)."""
        n = len(bytes64) // 64
        h = ctypes.c_void_p()
        self._check(self._lib.bpp_points_from_uniform(self._ctx, bytes(bytes64), n, ctypes.byref(h)))
        return Points(self, h, n)

    def compress_points(self, points: Points, off: int = 0, n: int = None) -> bytes:
        if n is None:
            n = len(points) - off
        out = ctypes.create_string_buffer(32 * n)
        self._check(self._lib.bpp_points_compress(self._ctx, points._h, off, n, out))
        return out.raw

    # -- the operator ------------------------------------------------------------------------------
    def vartime_multiscalar_mul(self, scalars, points, off: int = 0, n: int = None, want_ext: bool = False):
        """sum_i scalars[i] * points[i] -> 32-byte compressed Ristretto point."""
        sb = scalars if isinstance(scalars, (bytes, bytearray)) else scalars_to_bytes(scalars)
        ns = len(sb) // 32
        out = ctypes.create_string_buffer(32)
        if isinstance(points, Points):
            if n is None:
                n = len(points) - off
            ext = ctypes.create_string_buffer(128) if want_ext else None
            self._check(self._lib.bpp_msm_vartime(self._ctx, bytes(sb), ns, points._h, off, n, out, ext))
            return (out.raw, ext.raw) if want_ext else out.raw
        pb = points if isinstance(points, (bytes, bytearray)) else b"".join(points)
        self._check(self._lib.bpp_msm_vartime_host(self._ctx, bytes(sb), ns, FMT_COMPRESSED, bytes(pb), len(pb) // 32,
                                                   out))
        return out.raw

    def msm_host(self, scalars: bytes, points_enc: bytes) -> bytes:
        """The trait-level call: scalars and compressed points in host memory -> compressed result
        (bpp_msm_vartime_host: decompress, multiply, compress; one call, nothing stays resident)."""
        return self.vartime_multiscalar_mul(scalars, bytes(points_enc))

    def precompute(self, points: Points, window_bits: int = 0):
        """Attach a fixed-base window table to a long-lived point set (bpp_points_precompute)."""
        self._check(self._lib.bpp_points_precompute(self._ctx, points._h, window_bits))

    def msm_batch(self, scalars: bytes, points: Points, n: int, count: int, off: int = 0) -> bytes:
        """`count` MSMs over the same points[off:off+n] with count x n scalars, one launch -> count x 32 bytes."""
        if len(scalars) != 32 * n * count:
            raise ValueError("scalars: count x n x 32 bytes")
        out = ctypes.create_string_buffer(32 * count)
        self._check(self._lib.bpp_msm_vartime_batch(self._ctx, bytes(scalars), count, points._h, off, n, out))
        return out.raw

    # -- many independent MSMs over caller points (bpp_msm_multi*): MSM j takes the next sizes[j] terms ----------
    @staticmethod
    def _sizes(sizes):
        sizes = [int(x) for x in sizes]
        return (ctypes.c_uint32 * max(1, len(sizes)))(*sizes), len(sizes), sum(sizes)

    def msm_multi(self, scalars: bytes, points_enc: bytes, sizes):
        """`len(sizes)` MSMs over T x 32 scalars and T x 32 encodings -> (encodings, ok flags).  An undecodable point
        fails only its own MSM (ok False, 32 zero bytes)."""
        arr, count, T = self._sizes(sizes)
        if len(scalars) != 32 * T or len(points_enc) != 32 * T:
            raise ValueError("scalars and points: sum(sizes) x 32 bytes each")
        out, ok = ctypes.create_string_buffer(32 * count), ctypes.create_string_buffer(count)
        self._check(self._lib.bpp_msm_multi(self._ctx, count, arr, bytes(scalars), bytes(points_enc), out, ok))
        return [out.raw[32 * j:32 * j + 32] for j in range(count)], [b != 0 for b in ok.raw]

    def msm_multi_indexed(self, scalars: bytes, points: Points, index, sizes):
        """`len(sizes)` MSMs with P_t = points[index[t]] -> list of encodings."""
        arr, count, T = self._sizes(sizes)
        raw = index.tobytes() if hasattr(index, "tobytes") else array.array("I", index).tobytes()   # uint32 each
        if len(scalars) != 32 * T or len(raw) != 4 * T:
            raise ValueError("scalars: sum(sizes) x 32 bytes, index: sum(sizes) uint32 entries")
        ix = (ctypes.c_uint32 * max(1, T)).from_buffer_copy(raw or bytes(4))
        out = ctypes.create_string_buffer(32 * count)
        self._check(self._lib.bpp_msm_multi_indexed(self._ctx, count, arr, bytes(scalars), points._h, ix, out))
        return [out.raw[32 * j:32 * j + 32] for j in range(count)]

    def msm_multi_dev(self, sizes, d_scalars: int, d_points_enc: int, d_out32: int, d_ok: int):
        arr, count, _ = self._sizes(sizes)
        self._check(self._lib.bpp_msm_multi_dev(self._ctx, count, arr, ctypes.c_void_p(d_scalars), ctypes.c_void_p(d_points_enc),
                                                ctypes.c_void_p(d_out32), ctypes.c_void_p(d_ok)))

    def msm_multi_indexed_dev(self, sizes, d_scalars: int, points: Points, d_index: int, d_out32: int):
        arr, count, _ = self._sizes(sizes)
        self._check(self._lib.bpp_msm_multi_indexed_dev(self._ctx, count, arr, ctypes.c_void_p(d_scalars), points._h,
                                                        ctypes.c_void_p(d_index), ctypes.c_void_p(d_out32)))

    # -- mixed MSMs (bpp_msm_mixed*): a static part over points[off:off+n_static] plus the next sizes[j] caller terms ----
    def msm_mixed(self, static_scalars: bytes, points: Points, n_static: int, dyn_scalars: bytes, dyn_points_enc: bytes, sizes,
                  off: int = 0):
        """`len(sizes)` MSMs, MSM j = sum_i static_scalars[j][i] points[off + i] + its sizes[j] dynamic terms (T x 32
        scalars, T x 32 encodings) -> (encodings, ok flags).  An undecodable dynamic point fails only its own MSM (ok False,
        32 zero bytes)."""
        arr, count, T = self._sizes(sizes)
        if len(static_scalars) != 32 * n_static * count:
            raise ValueError("static scalars: len(sizes) x n_static x 32 bytes")
        if len(dyn_scalars) != 32 * T or len(dyn_points_enc) != 32 * T:
            raise ValueError("dynamic scalars and points: sum(sizes) x 32 bytes each")
        out, ok = ctypes.create_string_buffer(32 * count), ctypes.create_string_buffer(count)
        self._check(self._lib.bpp_msm_mixed(self._ctx, count, points._h, off, n_static, bytes(static_scalars), arr,
                                            bytes(dyn_scalars), bytes(dyn_points_enc), out, ok))
        return [out.raw[32 * j:32 * j + 32] for j in range(count)], [b != 0 for b in ok.raw]

    def msm_mixed_dev(self, points: Points, n_static: int, d_static_scalars: int, sizes, d_dyn_scalars: int, d_dyn_points_enc: int,
                      d_out32: int, d_ok: int, off: int = 0):
        arr, count, _ = self._sizes(sizes)
        self._check(self._lib.bpp_msm_mixed_dev(self._ctx, count, points._h, off, n_static, ctypes.c_void_p(d_static_scalars), arr,
                                                ctypes.c_void_p(d_dyn_scalars), ctypes.c_void_p(d_dyn_points_enc),
                                                ctypes.c_void_p(d_out32), ctypes.c_void_p(d_ok)))

    # device-pointer forms (pointers are ints, e.g. torch.Tensor.data_ptr())
    def msm_dev(self, d_scalars: int, points: Points, off: int, n: int, d_out: int):
        self._check(self._lib.bpp_msm_vartime_dev(self._ctx, ctypes.c_void_p(d_scalars), points._h, off, n,
                                                  ctypes.c_void_p(d_out)))

    def msm_submit_dev(self, d_scalars: int, points: Points, off: int, n: int, d_out: int):
        """Throughput form: enqueue without making the caller's stream wait; the result is valid after msm_wait()."""
        self._check(self._lib.bpp_msm_submit_dev(self._ctx, ctypes.c_void_p(d_scalars), points._h, off, n,
                                                 ctypes.c_void_p(d_out)))

    def msm_submit_partial_dev(self, d_scalars: int, points: Points, off: int, n: int, d_partial: int):
        self._check(self._lib.bpp_msm_submit_partial_dev(self._ctx, ctypes.c_void_p(d_scalars), points._h, off, n,
                                                         ctypes.c_void_p(d_partial)))

    def msm_wait(self):
        self._check(self._lib.bpp_msm_wait(self._ctx))

    def msm_wait_previous(self):
        """Wait for every submitted MSM except the one submitted last."""
        self._check(self._lib.bpp_msm_wait_previous(self._ctx))

    def msm_partial_dev(self, d_scalars: int, points: Points, off: int, n: int, d_partial: int):
        self._check(self._lib.bpp_msm_partial_dev(self._ctx, ctypes.c_void_p(d_scalars), points._h, off, n,
                                                  ctypes.c_void_p(d_partial)))

    def points_sum_compress_dev(self, d_partials: int, g: int, d_out32: int):
        self._check(self._lib.bpp_points_sum_compress_dev(self._ctx, ctypes.c_void_p(d_partials), g,
                                                          ctypes.c_void_p(d_out32)))

    def ipa_fold_generators(self, points: Points, n: int, u: bytes, uinv: bytes, off: int = 0, want: bool = True):
        """K7: `folds` foldings G'_i = u^-1 P_i + u P_{i+n/2} of points[off:off+n]; returns (encodings or b"", kernel ms)."""
        folds = len(u) // 32
        out = ctypes.create_string_buffer(32 * folds * (n // 2)) if want else None
        ms = ctypes.c_float()
        self._check(self._lib.bpp_ipa_fold_generators(self._ctx, points._h, off, n, bytes(u), bytes(uinv), folds, out, ctypes.byref(ms)))
        return (out.raw if want else b""), ms.value

    # -- multi-GPU: the library's own NCCL communicator (one process per GPU) -----------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        """128-byte id made on rank 0; the host program hands it to every rank (bpp_comm_unique_id)."""
        from . import _lib
        out = ctypes.create_string_buffer(128)
        rc = _lib.load().bpp_comm_unique_id(out)
        if rc:
            raise _lib.BppError(rc, "bpp_comm_unique_id")
        return out.raw

    def comm_init(self, nranks: int, rank: int, uid: bytes):
        self._check(self._lib.bpp_comm_init(self._ctx, nranks, rank, bytes(uid)))

    def comm_free(self):
        self._check(self._lib.bpp_comm_free(self._ctx))

    def comm_info(self):
        nr, r = ctypes.c_int(), ctypes.c_int()
        self._check(self._lib.bpp_comm_info(self._ctx, ctypes.byref(nr), ctypes.byref(r)))
        return nr.value, r.value

    def all_gather_dev(self, d_send: int, bytes_per_rank: int, d_recv: int):
        self._check(self._lib.bpp_comm_all_gather_dev(self._ctx, ctypes.c_void_p(d_send), bytes_per_rank, ctypes.c_void_p(d_recv)))

    def msm_sharded_dev(self, d_scalars: int, points: Points, off: int, n: int, d_out32: int):
        """This rank's slice -> the full MSM's encoding on every rank (partial, 128-byte all-gather, sum, compress)."""
        self._check(self._lib.bpp_msm_sharded_dev(self._ctx, ctypes.c_void_p(d_scalars), points._h, off, n, ctypes.c_void_p(d_out32)))

    def msm_sharded_submit_dev(self, d_scalars: int, points: Points, off: int, n: int, d_out32: int):
        self._check(self._lib.bpp_msm_sharded_submit_dev(self._ctx, ctypes.c_void_p(d_scalars), points._h, off, n,
                                                         ctypes.c_void_p(d_out32)))

    def msm_sharded_wait(self):
        self._check(self._lib.bpp_msm_sharded_wait(self._ctx))

    # -- element-wise self-test hook ------------------------------------------------------------------
    def test_op(self, op: int, a: bytes, b: bytes) -> bytes:
        n = len(a) // 32
        out = ctypes.create_string_buffer(32 * n)
        self._check(self._lib.bpp_test_op(self._ctx, op, a, b, out, n))
        return out.raw
