"""ctypes wrapper for oracle/c/dalek_ref.c (C restatement of the dalek-ng 4.1.1 serial backend).

TEST INFRASTRUCTURE (see oracle/__init__.py): fast checker for sizes the Python oracle cannot
reach, and the timed CPU baseline.  Points cross this API as opaque 160-byte blobs
(the in-memory layout of dalek's RistrettoPoint: 4 x FieldElement51).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libbpperm_oracle.so")
_lib = None
PT = 160


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, "c", f) for f in ("dalek_ref.c", "acproof_ref.c")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(x) for x in srcs):
        subprocess.check_call(["make", "-C", os.path.join(_HERE, "c"), "-B"], stdout=subprocess.DEVNULL)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        l = ctypes.CDLL(_SO)
        c = ctypes
        l.orc_point_size.restype = c.c_int
        l.orc_decompress.argtypes = [c.c_char_p, c.c_size_t, c.c_char_p]
        l.orc_compress.argtypes = [c.c_char_p, c.c_size_t, c.c_char_p]
        l.orc_compress.restype = None
        l.orc_from_uniform.argtypes = [c.c_char_p, c.c_size_t, c.c_char_p]
        l.orc_from_uniform.restype = None
        l.orc_point_add.argtypes = [c.c_char_p, c.c_char_p, c.c_char_p]
        l.orc_point_add.restype = None
        l.orc_msm_vartime.argtypes = [c.c_char_p, c.c_char_p, c.c_size_t, c.c_char_p]
        l.orc_msm_vartime.restype = None
        l.orc_msm_forced.argtypes = [c.c_int, c.c_char_p, c.c_char_p, c.c_size_t, c.c_char_p]
        l.orc_msm_forced.restype = None
        l.orc_scalar_mul.argtypes = [c.c_char_p, c.c_char_p, c.c_char_p]
        l.orc_scalar_mul.restype = None
        l.orc_msm_vartime_mt.argtypes = [c.c_char_p, c.c_char_p, c.c_size_t, c.c_int, c.c_char_p]
        l.orc_msm_vartime_mt.restype = None
        l.orc_acp_prove_verify.argtypes = [c.c_int, c.c_size_t, c.c_size_t, c.c_size_t] + [c.c_char_p] * 17 + [
            c.c_size_t, c.c_char_p, c.c_int]
        l.orc_acp_verify.argtypes = [c.c_int, c.c_size_t, c.c_size_t, c.c_size_t] + [c.c_char_p] * 13 + [c.c_size_t]
        l.orc_acp_fixed_proof_len.argtypes = [c.c_size_t]
        l.orc_acp_fixed_proof_len.restype = c.c_size_t
        l.orc_acp_fixed_prove_verify.argtypes = [c.c_size_t, c.c_size_t, c.c_size_t, c.c_char_p, c.c_char_p, c.c_char_p] + [
            c.c_char_p] * 13 + [c.c_char_p, c.c_size_t, c.c_char_p, c.c_int, c.c_int]
        l.orc_commit_variables.argtypes = [c.c_char_p] * 4 + [c.c_size_t, c.c_char_p]
        l.orc_commit_variables.restype = None
        l.orc_scalar_ops_selftest.argtypes = [c.c_char_p] * 4
        l.orc_scalar_ops_selftest.restype = None
        assert l.orc_point_size() == PT
        _lib = l
    return _lib


def decompress(enc: bytes) -> bytes:
    n = len(enc) // 32
    out = ctypes.create_string_buffer(PT * n)
    rc = lib().orc_decompress(enc, n, out)
    if rc != 0:
        raise ValueError("invalid ristretto255 encoding")
    return out.raw


def compress(pts: bytes) -> bytes:
    n = len(pts) // PT
    out = ctypes.create_string_buffer(32 * n)
    lib().orc_compress(pts, n, out)
    return out.raw


def from_uniform(b64: bytes) -> bytes:
    n = len(b64) // 64
    out = ctypes.create_string_buffer(PT * n)
    lib().orc_from_uniform(b64, n, out)
    return out.raw


def msm(scalars: bytes, pts: bytes, threads: int = 1, forced: int = -1) -> bytes:
    """vartime_multiscalar_mul with dalek's dispatch -> 32-byte compressed result."""
    n = len(pts) // PT
    assert len(scalars) == 32 * n
    out = ctypes.create_string_buffer(PT)
    if forced >= 0:
        lib().orc_msm_forced(forced, scalars, pts, n, out)
    elif threads > 1:
        lib().orc_msm_vartime_mt(scalars, pts, n, threads, out)
    else:
        lib().orc_msm_vartime(scalars, pts, n, out)
    return compress(out.raw)


def msm_raw(scalars: bytes, pts: bytes, threads: int = 1) -> bytes:
    n = len(pts) // PT
    out = ctypes.create_string_buffer(PT)
    if threads > 1:
        lib().orc_msm_vartime_mt(scalars, pts, n, threads, out)
    else:
        lib().orc_msm_vartime(scalars, pts, n, out)
    return out.raw


class AcpInstance:
    """Dense-matrix instance for orc_acp_prove_verify (the reference's ACEssentials + ACProver shapes)."""

    def __init__(self, n, Q, m, W_L, W_R, W_O, W_V, c_vec, g, h, G, H):
        """W_* and c_vec: bytes of dense row-major scalar matrices; g, h, G, H: compressed encodings."""
        self.n, self.Q, self.m = n, Q, m
        self.W = (W_L, W_R, W_O, W_V)
        self.c = c_vec
        self.g, self.h = decompress(g), decompress(h)
        self.G, self.H = decompress(G), decompress(H)

    def commit(self, v: bytes, gamma: bytes) -> bytes:
        out = ctypes.create_string_buffer(PT * self.m)
        lib().orc_commit_variables(self.g, self.h, v, gamma, self.m, out)
        return out.raw

    def prove_verify(self, aL, aR, aO, gamma, V_pts, seed, mode=1, label=b"test", do_verify=True, V_enc=None):
        """-> (proof_bytes, result) with result 1 = Ok(()), 0 = Err(VerificationError).  V_pts: the commitments as
        points (orc layout); V_enc: their 32-byte encodings when the caller has them (else compressed inside)."""
        out = ctypes.create_string_buffer(32 * (11 + 2 * self.n))
        rc = lib().orc_acp_prove_verify(mode, self.n, self.Q, self.m, self.W[0], self.W[1], self.W[2], self.W[3], self.c,
                                        self.g, self.h, self.G, self.H, aL, aR, aO, gamma, V_pts, V_enc, seed, label,
                                        len(label), out, 1 if do_verify else 0)
        return out.raw, rc

    def verify(self, proof: bytes, V_pts, mode=1, V_enc=None, label=b"test") -> bool:
        """The verifier of modes 0 and 1 from the proof bytes alone (orc_acp_verify): the transcript is replayed from
        them, a scalar >= l is taken mod l, an undecodable point is a reject and the all-zero encoding is the identity.
        V_pts: the commitments as points (orc layout), or None to decode them from V_enc (an undecodable commitment is
        a reject); V_enc: the encodings the transcript binds (default: V_pts compressed)."""
        if len(proof) != 32 * (11 + 2 * self.n):
            raise ValueError("proof: 32 (11 + 2 n) bytes")
        if V_pts is None and V_enc is None:
            raise ValueError("verify: V_pts or V_enc")
        mode = {"reference": 0, "reference-fixed": 1}.get(mode, mode)
        rc = lib().orc_acp_verify(mode, self.n, self.Q, self.m, self.W[0], self.W[1], self.W[2], self.W[3], self.c,
                                  self.g, self.h, self.G, self.H, proof, V_pts, V_enc, label, len(label))
        return rc == 1


class AcpFixedInstance:
    """Sparse-weight instance for orc_acp_fixed_prove_verify (`fixed` mode: standard powers + IPA,
    oracle/ipa.py).  W_* are lists of (wire, constraint, coeff) triples; G, H hold next_pow2(n) generators."""

    def __init__(self, n, Q, m, WL, WR, WO, WV, c_vec: bytes, g, h, G, H):
        import struct
        self.n, self.Q, self.m = n, Q, m
        mats = (WL, WR, WO, WV)
        self.nnz = struct.pack("<4I", *[len(x) for x in mats])
        self.wire = b"".join(struct.pack("<I", t[0]) for M in mats for t in M)
        self.cons = b"".join(struct.pack("<I", t[1]) for M in mats for t in M)
        self.coeff = b"".join(int(t[2]).to_bytes(32, "little") for M in mats for t in M)
        self.c = c_vec
        self.g, self.h = decompress(g), decompress(h)
        self.G, self.H = decompress(G), decompress(H)
        self.proof_len = lib().orc_acp_fixed_proof_len(n)

    @classmethod
    def from_core(cls, core):
        """From an oracle.ipa.make_instance() core dict (points as oracle.ristretto255 tuples)."""
        from . import ristretto255 as R
        WL, WR, WO, WV = core["sparse"]
        return cls(core["n"], core["Q"], core["m"], WL, WR, WO, WV, b"".join(R.sc_bytes(s) for s in core["c_vec"]),
                   R.compress(core["g_base"]), R.compress(core["h_base"]),
                   b"".join(R.compress(p) for p in core["G_vec"]), b"".join(R.compress(p) for p in core["H_vec"]))

    def commit(self, v: bytes, gamma: bytes) -> bytes:
        out = ctypes.create_string_buffer(PT * self.m)
        lib().orc_commit_variables(self.g, self.h, v, gamma, self.m, out)
        return out.raw

    def _call(self, aL, aR, aO, gamma, V_pts, V_enc, seed, label, buf, do_prove, do_verify):
        return lib().orc_acp_fixed_prove_verify(self.n, self.Q, self.m, self.nnz, self.wire, self.cons, self.coeff, self.c,
                                                self.g, self.h, self.G, self.H, aL, aR, aO, gamma, V_pts, V_enc, seed, label,
                                                len(label), buf, do_prove, do_verify)

    def prove(self, aL, aR, aO, gamma, V_pts, seed, label=b"test", V_enc=None) -> bytes:
        """V_pts: the value commitments as points (bound to the transcript); V_enc: their encodings, if at hand."""
        buf = ctypes.create_string_buffer(self.proof_len)
        self._call(aL, aR, aO, gamma, V_pts, V_enc, seed, label, buf, 1, 0)
        return buf.raw

    def verify(self, proof: bytes, V_pts: bytes, label=b"test", V_enc=None) -> bool:
        buf = ctypes.create_string_buffer(proof, len(proof))
        return self._call(None, None, None, None, V_pts, V_enc, None, label, buf, 0, 1) == 1
