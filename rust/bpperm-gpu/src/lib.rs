//! Drop-in host layer for ercembu/bulletproof-perm over libbpperm_cuda.so.  NOT compiled in the build image
//! (no Rust toolchain there); kept mechanical so that it can be checked by reading it against include/bpperm.h.
use bpperm_sys as sys;
use bulletproofs::ProofError;
use curve25519_dalek_ng::ristretto::{CompressedRistretto, RistrettoPoint};
use curve25519_dalek_ng::scalar::Scalar;
use curve25519_dalek_ng::traits::{VartimeMultiscalarMul, VartimePrecomputedMultiscalarMul};
use once_cell::sync::Lazy;
use std::borrow::Borrow;
use std::sync::Mutex;

struct Ctx(*mut sys::bpp_ctx);
unsafe impl Send for Ctx {}
/// The trait is stateless (associated functions), so the GPU context is a lazily created process global.
static CTX: Lazy<Mutex<Ctx>> = Lazy::new(|| {
    let mut c = std::ptr::null_mut();
    let rc = unsafe { sys::bpp_init(0, &mut c) };
    assert_eq!(rc, 0, "bpp_init failed: no sm_100 GPU (this backend has no CPU fallback)");
    Mutex::new(Ctx(c))
});
fn with_ctx<T>(f: impl FnOnce(*mut sys::bpp_ctx) -> T) -> T { f(CTX.lock().unwrap().0) }

/// `RistrettoPoint::vartime_multiscalar_mul(..)` -> `GpuRistretto::vartime_multiscalar_mul(..)`
/// (circuit_lib.rs:187,202,216,363,374,385,396,407,498,504,509,525,535,552,568).
pub struct GpuRistretto;
impl VartimeMultiscalarMul for GpuRistretto {
    type Point = RistrettoPoint;
    fn optional_multiscalar_mul<I, J>(scalars: I, points: J) -> Option<RistrettoPoint>
    where I: IntoIterator, I::Item: Borrow<Scalar>, J: IntoIterator<Item = Option<RistrettoPoint>> {
        let s: Vec<u8> = scalars.into_iter().flat_map(|s| s.borrow().to_bytes().to_vec()).collect();
        let p: Vec<RistrettoPoint> = points.into_iter().collect::<Option<Vec<_>>>()?;
        assert_eq!(s.len() / 32, p.len()); // dalek asserts on the iterators' size hints
        // Points cross the boundary as their 32-byte encodings: dalek gives no layout guarantee for RistrettoPoint
        // (BPP_FMT_DALEK_XYZT exists for builds that pin curve25519-dalek-ng 4.1.1's u64 backend and accept that).
        // Long-lived generator sets should not come through here at all: see `GeneratorSet` below.
        let enc: Vec<u8> = p.iter().flat_map(|q| q.compress().to_bytes().to_vec()).collect();
        let mut out = [0u8; 32];
        let rc = with_ctx(|c| unsafe {
            sys::bpp_msm_vartime_host(c, s.as_ptr(), p.len(), sys::BPP_FMT_COMPRESSED, enc.as_ptr(), p.len(), out.as_mut_ptr())
        });
        assert_eq!(rc, 0);
        CompressedRistretto(out).decompress()
    }
}
impl GpuRistretto {
    /// Many independent `optional_multiscalar_mul` calls in one `bpp_msm_multi`: call k is (scalars, points), the
    /// results come back in call order.  A call whose points do not all decode gives `None`, as a single call does;
    /// the other calls are unaffected.
    pub fn optional_multiscalar_mul_many(calls: &[(Vec<Scalar>, Vec<CompressedRistretto>)]) -> Vec<Option<RistrettoPoint>> {
        if calls.is_empty() { return Vec::new(); }
        let sizes: Vec<u32> = calls.iter().map(|(s, p)| { assert_eq!(s.len(), p.len()); s.len() as u32 }).collect();
        let s: Vec<u8> = calls.iter().flat_map(|(s, _)| s.iter().flat_map(|x| x.to_bytes().to_vec())).collect();
        let enc: Vec<u8> = calls.iter().flat_map(|(_, p)| p.iter().flat_map(|q| q.to_bytes().to_vec())).collect();
        let mut out = vec![0u8; 32 * calls.len()];
        let mut ok = vec![0u8; calls.len()];
        let rc = with_ctx(|c| unsafe {
            sys::bpp_msm_multi(c, calls.len(), sizes.as_ptr(), s.as_ptr(), enc.as_ptr(), out.as_mut_ptr(), ok.as_mut_ptr())
        });
        assert_eq!(rc, 0);
        out.chunks_exact(32).zip(ok.iter())
            .map(|(o, &k)| if k == 1 { CompressedRistretto(<[u8; 32]>::try_from(o).unwrap()).decompress() } else { None })
            .collect()
    }
}

/// The reference's 15 call sites always multiply sub-ranges of the same generators (g, h, G_vec, H_vec: lib.rs:164-180).
/// Upload them once, attach the window table once; every later MSM is table look-ups + mixed adds, and
/// `msm_batch` runs `count` of them (one per proof) in a single launch.
pub struct GeneratorSet { pts: *mut sys::bpp_points, n: usize }
unsafe impl Send for GeneratorSet {}
impl GeneratorSet {
    pub fn new(points: &[RistrettoPoint], window_bits: i32) -> Self {
        let enc: Vec<u8> = points.iter().flat_map(|q| q.compress().to_bytes().to_vec()).collect();
        let mut pts = std::ptr::null_mut();
        with_ctx(|c| unsafe {
            assert_eq!(sys::bpp_points_upload(c, sys::BPP_FMT_COMPRESSED, enc.as_ptr(), points.len(), &mut pts), 0);
            assert_eq!(sys::bpp_points_precompute(c, pts, window_bits), 0);
        });
        GeneratorSet { pts, n: points.len() }
    }
    /// sum_i scalars[i] * points[off + i]
    pub fn msm(&self, scalars: &[Scalar], off: usize) -> RistrettoPoint {
        assert!(off + scalars.len() <= self.n);
        let mut out = [0u8; 32];
        let rc = with_ctx(|c| unsafe {
            sys::bpp_msm_vartime(c, bytes_of(scalars).as_ptr(), scalars.len(), self.pts, off, scalars.len(), out.as_mut_ptr(), std::ptr::null_mut())
        });
        assert_eq!(rc, 0);
        CompressedRistretto(out).decompress().expect("library returns valid encodings")
    }
    /// `count` MSMs over points[off..off + n) with count x n scalars (row-major), one launch
    pub fn msm_batch(&self, scalars: &[Scalar], count: usize, off: usize, n: usize) -> Vec<CompressedRistretto> {
        assert_eq!(scalars.len(), count * n);
        let mut out = vec![0u8; 32 * count];
        let rc = with_ctx(|c| unsafe { sys::bpp_msm_vartime_batch(c, bytes_of(scalars).as_ptr(), count, self.pts, off, n, out.as_mut_ptr()) });
        assert_eq!(rc, 0);
        out.chunks_exact(32).map(|c| CompressedRistretto(<[u8; 32]>::try_from(c).unwrap())).collect()
    }
    /// Independent MSMs over points of this set chosen per term: MSM j = sum scalars[t] * points[index[t]] over its
    /// sizes[j] terms (terms of all MSMs one after another).  No table: any mix of sub-ranges and sizes, one call.
    pub fn msm_many_indexed(&self, sizes: &[u32], scalars: &[Scalar], index: &[u32]) -> Vec<CompressedRistretto> {
        let total: usize = sizes.iter().map(|&n| n as usize).sum();
        assert!(scalars.len() == total && index.len() == total && !sizes.is_empty());
        let mut out = vec![0u8; 32 * sizes.len()];
        let rc = with_ctx(|c| unsafe {
            sys::bpp_msm_multi_indexed(c, sizes.len(), sizes.as_ptr(), bytes_of(scalars).as_ptr(), self.pts, index.as_ptr(), out.as_mut_ptr())
        });
        assert_eq!(rc, 0);
        out.chunks_exact(32).map(|c| CompressedRistretto(<[u8; 32]>::try_from(c).unwrap())).collect()
    }
    /// Mixed MSMs in one `bpp_msm_mixed`: call j = sum_i static_scalars[j n + i] * points[off + i] + sum of the call's own
    /// (scalars, points).  `static_scalars` holds calls.len() rows of n scalars (zeros where a call has fewer static
    /// terms).  A call whose points do not all decode gives `None`; the other calls are unaffected.
    pub fn mixed_msm_many(&self, static_scalars: &[Scalar], off: usize, n: usize, calls: &[(Vec<Scalar>, Vec<CompressedRistretto>)])
                          -> Vec<Option<RistrettoPoint>> {
        if calls.is_empty() { return Vec::new(); }
        assert!(n > 0 && off + n <= self.n && static_scalars.len() == calls.len() * n);
        let sizes: Vec<u32> = calls.iter().map(|(s, p)| { assert_eq!(s.len(), p.len()); s.len() as u32 }).collect();
        let s: Vec<u8> = calls.iter().flat_map(|(s, _)| s.iter().flat_map(|x| x.to_bytes().to_vec())).collect();
        let enc: Vec<u8> = calls.iter().flat_map(|(_, p)| p.iter().flat_map(|q| q.to_bytes().to_vec())).collect();
        let mut out = vec![0u8; 32 * calls.len()];
        let mut ok = vec![0u8; calls.len()];
        let rc = with_ctx(|c| unsafe {
            sys::bpp_msm_mixed(c, calls.len(), self.pts, off, n, bytes_of(static_scalars).as_ptr(), sizes.as_ptr(), s.as_ptr(),
                               enc.as_ptr(), out.as_mut_ptr(), ok.as_mut_ptr())
        });
        assert_eq!(rc, 0);
        out.chunks_exact(32).zip(ok.iter())
            .map(|(o, &k)| if k == 1 { CompressedRistretto(<[u8; 32]>::try_from(o).unwrap()).decompress() } else { None })
            .collect()
    }
}
impl Drop for GeneratorSet { fn drop(&mut self) { with_ctx(|c| unsafe { sys::bpp_points_free(c, self.pts) }) } }

/// `ristretto::VartimeRistrettoPrecomputation` -> `GpuRistrettoPrecomputation`: dalek's `VartimePrecomputedMultiscalarMul`
/// (the verifier's MSM: static generators plus points from the proof).  `new` uploads the static points and builds their
/// window table (c = 8) once; each call is a one-MSM `bpp_msm_mixed`.  For many such MSMs at once use
/// `GeneratorSet::mixed_msm_many`.
pub struct GpuRistrettoPrecomputation { set: Option<GeneratorSet> }   // None: no static points
impl VartimePrecomputedMultiscalarMul for GpuRistrettoPrecomputation {
    type Point = RistrettoPoint;
    fn new<I>(static_points: I) -> Self where I: IntoIterator, I::Item: Borrow<RistrettoPoint> {
        let pts: Vec<RistrettoPoint> = static_points.into_iter().map(|p| *p.borrow()).collect();
        GpuRistrettoPrecomputation { set: if pts.is_empty() { None } else { Some(GeneratorSet::new(&pts, 8)) } }
    }
    fn optional_mixed_multiscalar_mul<I, J, K>(&self, static_scalars: I, dynamic_scalars: J, dynamic_points: K) -> Option<RistrettoPoint>
    where I: IntoIterator, I::Item: Borrow<Scalar>, J: IntoIterator, J::Item: Borrow<Scalar>, K: IntoIterator<Item = Option<RistrettoPoint>> {
        let st: Vec<Scalar> = static_scalars.into_iter().map(|s| *s.borrow()).collect();
        let ds: Vec<Scalar> = dynamic_scalars.into_iter().map(|s| *s.borrow()).collect();
        let dp: Vec<RistrettoPoint> = dynamic_points.into_iter().collect::<Option<Vec<_>>>()?;
        assert_eq!(ds.len(), dp.len());
        let enc: Vec<CompressedRistretto> = dp.iter().map(|p| p.compress()).collect();
        match &self.set {
            Some(set) => {
                assert_eq!(st.len(), set.n, "one static scalar per static point");
                set.mixed_msm_many(&st, 0, set.n, &[(ds, enc)]).pop().unwrap()
            }
            None => {
                assert!(st.is_empty(), "one static scalar per static point");
                GpuRistretto::optional_multiscalar_mul_many(&[(ds, enc)]).pop().unwrap()
            }
        }
    }
}

/// A merlin `Transcript` held as the library's state (bpperm.h: bpp_transcript_*).  merlin::Transcript cannot be
/// exported, so a caller that hands its protocol's inner-product argument to `InnerProductBatch` runs the transcript
/// here: every append it makes to its own `Transcript` before the argument must be mirrored into this one.
#[derive(Clone)]
pub struct GpuTranscript { state: [u8; sys::BPP_TRANSCRIPT_BYTES] }
impl GpuTranscript {
    pub fn new(label: &'static [u8]) -> Self {
        let mut state = [0u8; sys::BPP_TRANSCRIPT_BYTES];
        assert_eq!(unsafe { sys::bpp_transcript_new(label.as_ptr(), label.len(), state.as_mut_ptr()) }, 0);
        GpuTranscript { state }
    }
    pub fn append_message(&mut self, label: &'static [u8], message: &[u8]) {
        assert_eq!(unsafe { sys::bpp_transcript_append_message(self.state.as_mut_ptr(), label.as_ptr(), label.len(), message.as_ptr(),
                                                               message.len()) }, 0);
    }
    pub fn append_u64(&mut self, label: &'static [u8], x: u64) { self.append_message(label, &x.to_le_bytes()) }
    pub fn challenge_bytes(&mut self, label: &'static [u8], dest: &mut [u8]) {
        assert_eq!(unsafe { sys::bpp_transcript_challenge_bytes(self.state.as_mut_ptr(), label.as_ptr(), label.len(), dest.as_mut_ptr(),
                                                                dest.len()) }, 0);
    }
}

/// `count` inner-product proofs of length n (bulletproofs 4.0.0 `InnerProductProof::create` / `verify`) over a
/// `GeneratorSet`: G = set[g_off..g_off + n), H = set[h_off..h_off + n), Q_p = q_p * set[q_off].
pub struct InnerProductBatch { b: *mut sys::bpp_ipa_batch, count: usize, n: usize, proof_len: usize }
impl InnerProductBatch {
    pub fn new(gens: &GeneratorSet, g_off: usize, h_off: usize, q_off: usize, n: usize, count: usize) -> Self {
        let mut b = std::ptr::null_mut();
        let rc = with_ctx(|c| unsafe { sys::bpp_ipa_batch_create(c, gens.pts, g_off, h_off, q_off, n, count, &mut b) });
        assert_eq!(rc, 0);
        InnerProductBatch { b, count, n, proof_len: unsafe { sys::bpp_ipa_proof_len(n) } }
    }
    fn states(ts: &[GpuTranscript]) -> Vec<u8> { ts.iter().flat_map(|t| t.state.to_vec()).collect() }
    fn opt(v: Option<&[Scalar]>) -> *const u8 { v.map_or(std::ptr::null(), |s| bytes_of(s).as_ptr()) }
    /// create for every proof; a, b, factors: count x n (row-major), q: count; None = ones.  The transcripts advance as
    /// create advances them.  Returns count proofs of `proof_len` bytes (InnerProductProof::to_bytes).
    pub fn prove(&mut self, transcripts: &mut [GpuTranscript], q: Option<&[Scalar]>, g_factors: Option<&[Scalar]>,
                 h_factors: Option<&[Scalar]>, a: &[Scalar], b: &[Scalar]) -> Vec<u8> {
        assert!(transcripts.len() == self.count && a.len() == self.count * self.n && b.len() == self.count * self.n);
        let mut st = Self::states(transcripts);
        let mut proofs = vec![0u8; self.count * self.proof_len];
        assert_eq!(unsafe { sys::bpp_ipa_batch_prove(self.b, Self::opt(q), Self::opt(g_factors), Self::opt(h_factors), bytes_of(a).as_ptr(),
                                                     bytes_of(b).as_ptr(), st.as_mut_ptr(), proofs.as_mut_ptr()) }, 0);
        for (t, s) in transcripts.iter_mut().zip(st.chunks_exact(sys::BPP_TRANSCRIPT_BYTES)) { t.state.copy_from_slice(s) }
        proofs
    }
    /// verify for every proof; one Result per proof.  The transcripts of accepted proofs advance as verify advances them.
    pub fn verify(&mut self, transcripts: &mut [GpuTranscript], q: Option<&[Scalar]>, g_factors: Option<&[Scalar]>,
                  h_factors: Option<&[Scalar]>, p: &[CompressedRistretto], proofs: &[u8]) -> Vec<Result<(), ProofError>> {
        assert!(transcripts.len() == self.count && p.len() == self.count && proofs.len() == self.count * self.proof_len);
        let mut st = Self::states(transcripts);
        let mut acc = vec![0u8; self.count];
        assert_eq!(unsafe { sys::bpp_ipa_batch_verify(self.b, Self::opt(q), Self::opt(g_factors), Self::opt(h_factors),
                                                      p.as_ptr() as *const u8, proofs.as_ptr(), st.as_mut_ptr(), acc.as_mut_ptr()) }, 0);
        for ((t, s), a) in transcripts.iter_mut().zip(st.chunks_exact(sys::BPP_TRANSCRIPT_BYTES)).zip(&acc) {
            if *a == 1 { t.state.copy_from_slice(s) }
        }
        acc.into_iter().map(|a| if a == 1 { Ok(()) } else { Err(ProofError::VerificationError) }).collect()
    }
    /// `verify`'s results and transcripts through one random-linear-combination MSM over the batch (every proof on its
    /// own only when the combination is not the identity).  verifier_seed: 32 bytes of SECRET, FRESH randomness, or
    /// None to have the library draw them from the OS.
    pub fn verify_combined(&mut self, transcripts: &mut [GpuTranscript], q: Option<&[Scalar]>, g_factors: Option<&[Scalar]>,
                           h_factors: Option<&[Scalar]>, p: &[CompressedRistretto], proofs: &[u8],
                           verifier_seed: Option<&[u8; 32]>) -> Vec<Result<(), ProofError>> {
        assert!(transcripts.len() == self.count && p.len() == self.count && proofs.len() == self.count * self.proof_len);
        let mut st = Self::states(transcripts);
        let mut acc = vec![0u8; self.count];
        assert_eq!(unsafe { sys::bpp_ipa_batch_verify_combined(self.b, Self::opt(q), Self::opt(g_factors), Self::opt(h_factors),
                                                               p.as_ptr() as *const u8, proofs.as_ptr(),
                                                               verifier_seed.map_or(std::ptr::null(), |s| s.as_ptr()),
                                                               st.as_mut_ptr(), acc.as_mut_ptr()) }, 0);
        for ((t, s), a) in transcripts.iter_mut().zip(st.chunks_exact(sys::BPP_TRANSCRIPT_BYTES)).zip(&acc) {
            if *a == 1 { t.state.copy_from_slice(s) }
        }
        acc.into_iter().map(|a| if a == 1 { Ok(()) } else { Err(ProofError::VerificationError) }).collect()
    }
    /// Sharded verification: every rank's accept bytes of its last verify (nranks x per, rank r's at r * per) through
    /// the library's communicator; this rank's own bytes without one.
    pub fn gather_accept(&mut self, per: usize) -> Vec<u8> {
        let (mut nranks, mut rank) = (0, 0);
        assert_eq!(with_ctx(|c| unsafe { sys::bpp_comm_info(c, &mut nranks, &mut rank) }), 0);
        let mut out = vec![0u8; per * nranks as usize];
        assert_eq!(unsafe { sys::bpp_ipa_batch_gather_accept(self.b, per, out.as_mut_ptr()) }, 0);
        out
    }
}
impl Drop for InnerProductBatch { fn drop(&mut self) { unsafe { sys::bpp_ipa_batch_free(self.b) } } }

fn bytes_of(v: &[Scalar]) -> &[u8] { unsafe { std::slice::from_raw_parts(v.as_ptr() as *const u8, v.len() * 32) } }

/// util.rs:84-94 (same panic text on a length mismatch)
pub fn inner_product(a: &Vec<Scalar>, b: &Vec<Scalar>) -> Scalar {
    let mut out = [0u8; 32];
    let rc = with_ctx(|c| unsafe { sys::bpp_inner_product(c, bytes_of(a).as_ptr(), a.len(), bytes_of(b).as_ptr(), b.len(), out.as_mut_ptr()) });
    if rc == sys::BPP_ERR_LENGTH_MISMATCH { panic!("inner_product(a,b): lengths dont match, {}, {}", a.len(), b.len()); }
    assert_eq!(rc, 0);
    Scalar::from_canonical_bytes(out).unwrap()
}
/// util.rs:6-20
pub fn hadamard_V(a: &Vec<Scalar>, b: &Vec<Scalar>) -> Vec<Scalar> {
    let mut out = vec![Scalar::zero(); a.len()];
    let rc = with_ctx(|c| unsafe { sys::bpp_hadamard_V(c, bytes_of(a).as_ptr(), a.len(), bytes_of(b).as_ptr(), b.len(), out.as_mut_ptr() as *mut u8) });
    if rc == sys::BPP_ERR_LENGTH_MISMATCH { panic!("hadamard_V(a,b): lengths dont match, {}, {}", a.len(), b.len()); }
    assert_eq!(rc, 0);
    out
}
/// util.rs:63-65,139-157: exp_iter(x).take(n) with the reference iterator's (Fibonacci) exponents
pub fn exp_iter_take(x: Scalar, n: usize) -> Vec<Scalar> {
    let mut out = vec![Scalar::zero(); n];
    let rc = with_ctx(|c| unsafe { sys::bpp_exp_iter(c, x.as_bytes().as_ptr(), n, out.as_mut_ptr() as *mut u8) });
    assert_eq!(rc, 0);
    out
}

fn flatten(m: &Vec<Vec<Scalar>>) -> Vec<u8> { m.iter().flat_map(|r| bytes_of(r).to_vec()).collect() }
/// util.rs:22-38: out[i] = <a, b[i]> (b: rows of length a.len())
pub fn vm_mult(a: &Vec<Scalar>, b: &Vec<Vec<Scalar>>) -> Vec<Scalar> {
    if a.len() != b[0].len() { panic!("vm_mult(a,b): a -> 1x{}, b -> {}x{} needs to be", a.len(), b[0].len(), b.len()); }
    let mut out = vec![Scalar::zero(); b.len()];
    let flat = flatten(b);
    let rc = with_ctx(|c| unsafe { sys::bpp_vm_mult(c, bytes_of(a).as_ptr(), a.len(), flat.as_ptr(), b.len(), b[0].len(), out.as_mut_ptr() as *mut u8) });
    assert_eq!(rc, 0);
    out
}
/// util.rs:58-61
pub fn lm_mult(a: &[Scalar], b: &Vec<Vec<Scalar>>) -> Vec<Scalar> { vm_mult(&Vec::from(a), b) }
/// util.rs:40-56: out[i] = sum_j a[j][i] * b[j]
pub fn mv_mult(a: &Vec<Vec<Scalar>>, b: &Vec<Scalar>) -> Vec<Scalar> {
    if a.len() != b.len() { panic!("mv_mult(a,b): a->{}x{}, b->{}x1 needs to be", a.len(), a[0].len(), b.len()); }
    let mut out = vec![Scalar::zero(); a[0].len()];
    let flat = flatten(a);
    let rc = with_ctx(|c| unsafe { sys::bpp_mv_mult(c, flat.as_ptr(), a.len(), a[0].len(), bytes_of(b).as_ptr(), b.len(), out.as_mut_ptr() as *mut u8) });
    assert_eq!(rc, 0);
    out
}
/// util.rs:67-82 (scalar_exp and scalar_exp_u): x^pow by repeated multiplication; pow <= 0 gives one
pub fn scalar_exp(x: &Scalar, pow: i32) -> Scalar {
    let mut out = [0u8; 32];
    let rc = with_ctx(|c| unsafe { sys::bpp_scalar_exp(c, x.as_bytes().as_ptr(), pow.max(0) as u32, out.as_mut_ptr()) });
    assert_eq!(rc, 0);
    Scalar::from_canonical_bytes(out).unwrap()
}
pub fn scalar_exp_u(x: &Scalar, pow: usize) -> Scalar { scalar_exp(x, pow as i32) }
/// circuit_lib.rs:273-275: y_n.iter().map(|k| k.invert()) - all inversions in one launch (0 -> 0 like Scalar::invert)
pub fn invert_all(v: &[Scalar]) -> Vec<Scalar> {
    let mut out = vec![Scalar::zero(); v.len()];
    let rc = with_ctx(|c| unsafe { sys::bpp_scalar_invert(c, bytes_of(v).as_ptr(), v.len(), out.as_mut_ptr() as *mut u8) });
    assert_eq!(rc, 0);
    out
}
/// poly.rs:5-18
pub struct Poly6 { pub t1: Scalar, pub t2: Scalar, pub t3: Scalar, pub t4: Scalar, pub t5: Scalar, pub t6: Scalar }
impl Poly6 {
    pub fn eval(&self, x: Scalar) -> Scalar {
        let t = [self.t1, self.t2, self.t3, self.t4, self.t5, self.t6];
        let mut out = [0u8; 32];
        let rc = with_ctx(|c| unsafe { sys::bpp_poly6_eval(c, bytes_of(&t).as_ptr(), x.as_bytes().as_ptr(), out.as_mut_ptr()) });
        assert_eq!(rc, 0);
        Scalar::from_canonical_bytes(out).unwrap()
    }
}
/// poly.rs:21-76
#[derive(Clone, Debug, Default)]
pub struct VecPoly3(pub Vec<Scalar>, pub Vec<Scalar>, pub Vec<Scalar>, pub Vec<Scalar>);
impl VecPoly3 {
    pub fn zero(n: usize) -> Self { VecPoly3(vec![Scalar::zero(); n], vec![Scalar::zero(); n], vec![Scalar::zero(); n], vec![Scalar::zero(); n]) }
    fn flat(&self) -> Vec<u8> { [&self.0, &self.1, &self.2, &self.3].iter().flat_map(|v| bytes_of(v).to_vec()).collect() }
    /// poly.rs:39-55 (the six sums as the reference codes them)
    pub fn special_inner_product(lhs: &Self, rhs: &Self) -> Poly6 {
        let (l, r) = (lhs.flat(), rhs.flat());
        let mut t = [Scalar::zero(); 6];
        let rc = with_ctx(|c| unsafe { sys::bpp_vecpoly3_special_inner_product(c, l.as_ptr(), r.as_ptr(), lhs.0.len(), t.as_mut_ptr() as *mut u8) });
        assert_eq!(rc, 0);
        Poly6 { t1: t[0], t2: t[1], t3: t[2], t4: t[3], t5: t[4], t6: t[5] }
    }
    /// poly.rs:57-76 (eval and eval_ref)
    pub fn eval(&self, x: Scalar) -> Vec<Scalar> { self.eval_ref(&x) }
    pub fn eval_ref(&self, x: &Scalar) -> Vec<Scalar> {
        let mut out = vec![Scalar::zero(); self.0.len()];
        let f = self.flat();
        let rc = with_ctx(|c| unsafe { sys::bpp_vecpoly3_eval(c, f.as_ptr(), self.0.len(), x.as_bytes().as_ptr(), out.as_mut_ptr() as *mut u8) });
        assert_eq!(rc, 0);
        out
    }
}

/// `count` ACProvers sharing one ACEssentials (circuit_lib.rs:58-88), proved and verified in lock-step.
pub struct ShuffleBatch { b: *mut sys::bpp_acp_batch, count: usize, proof_len: usize }
impl ShuffleBatch {
    pub fn new(cir: *const sys::bpp_circuit, gens: *const sys::bpp_gens, n: usize, mode: i32, count: usize, label: &[u8]) -> Self {
        let mut b = std::ptr::null_mut();
        let rc = with_ctx(|c| unsafe { sys::bpp_acp_batch_create(c, cir, gens, mode, count, label.as_ptr(), label.len(), &mut b) });
        assert_eq!(rc, 0);
        ShuffleBatch { b, count, proof_len: unsafe { sys::bpp_acproof_proof_len_mode(n, mode) } }
    }
    /// weights.rs:38-113 on the device: the witness of `count` shuffles from the deck, one permutation and one challenge
    /// value per proof; returns the value commitments V (commit_variables, weights.rs:58-61), which stay resident.
    pub fn witness_from_shuffles(&mut self, deck: &[Scalar], perm: &[u32], x: &[Scalar], gamma: &[Scalar], seeds: &[[u8; 32]],
                                 m: usize) -> Vec<CompressedRistretto> {
        let mut v = vec![0u8; 32 * m * self.count];
        unsafe {
            assert_eq!(sys::bpp_acp_batch_gen_shuffle_witness(self.b, bytes_of(deck).as_ptr(), perm.as_ptr(), bytes_of(x).as_ptr(),
                                                              bytes_of(gamma).as_ptr(), seeds.as_ptr() as *const u8), 0);
            assert_eq!(sys::bpp_acp_batch_commit(self.b, std::ptr::null(), v.as_mut_ptr()), 0);
        }
        v.chunks_exact(32).map(|c| CompressedRistretto(<[u8; 32]>::try_from(c).unwrap())).collect()
    }
    /// prove the witness left by `witness_from_shuffles`
    pub fn prove_resident(&mut self) -> Vec<u8> {
        let mut proofs = vec![0u8; self.count * self.proof_len];
        unsafe {
            assert_eq!(sys::bpp_acp_batch_prove(self.b), 0);
            assert_eq!(sys::bpp_acp_batch_download_proofs(self.b, proofs.as_mut_ptr()), 0);
        }
        proofs
    }
    /// create .. blinding_values (lib.rs:219-228); seeds: ChaCha20Rng::from_seed per proof instead of thread_rng();
    /// v: the value commitments (count x m), bound to every transcript in modes 1 and 2
    pub fn prove(&mut self, a_l: &[Scalar], a_r: &[Scalar], a_o: &[Scalar], gamma: &[Scalar], seeds: &[[u8; 32]],
                 v: &[CompressedRistretto]) -> Vec<u8> {
        let mut proofs = vec![0u8; self.count * self.proof_len];
        unsafe {
            assert_eq!(sys::bpp_acp_batch_upload_witness(self.b, bytes_of(a_l).as_ptr(), bytes_of(a_r).as_ptr(), bytes_of(a_o).as_ptr(),
                                                         bytes_of(gamma).as_ptr(), seeds.as_ptr() as *const u8), 0);
            assert_eq!(sys::bpp_acp_batch_upload_commitments(self.b, v.as_ptr() as *const u8), 0);
            assert_eq!(sys::bpp_acp_batch_prove(self.b), 0);
            assert_eq!(sys::bpp_acp_batch_download_proofs(self.b, proofs.as_mut_ptr()), 0);
        }
        proofs
    }
    /// verify (lib.rs:230): one Result per proof.  verifier_seed: 32 bytes of SECRET, FRESH randomness (e.g. from
    /// `thread_rng()`), or None to have the library draw them from the operating system; never a constant.
    pub fn verify(&mut self, proofs: &[u8], v: &[CompressedRistretto], verifier_seed: Option<&[u8; 32]>) -> Vec<Result<(), ProofError>> {
        let mut acc = vec![0u8; self.count];
        unsafe {
            assert_eq!(sys::bpp_acp_batch_upload_proofs(self.b, proofs.as_ptr(), v.as_ptr() as *const u8), 0);
            assert_eq!(sys::bpp_acp_batch_verify(self.b, verifier_seed.map_or(std::ptr::null(), |s| s.as_ptr())), 0);
            assert_eq!(sys::bpp_acp_batch_download_accept(self.b, acc.as_mut_ptr()), 0);
        }
        acc.into_iter().map(|a| if a == 1 { Ok(()) } else { Err(ProofError::VerificationError) }).collect()
    }
}
impl Drop for ShuffleBatch { fn drop(&mut self) { unsafe { sys::bpp_acp_batch_free(self.b) } } }

// ---- proof records on the wire (bpperm.h: bpp_acproof_to_wire / bpp_acproof_from_wire) ------------------------
// mode 2 records are bulletproofs 4.0.0 `R1CSProof::to_bytes` of a one-phase proof (version byte 0).
pub fn proofs_to_wire(n: usize, mode: i32, count: usize, proofs: &[u8]) -> Vec<u8> {
    let wlen = unsafe { sys::bpp_acproof_wire_len(n, mode) };
    let mut out = vec![0u8; count * wlen];
    assert_eq!(unsafe { sys::bpp_acproof_to_wire(n, mode, count, proofs.as_ptr(), out.as_mut_ptr()) }, 0);
    out
}
/// One `Result` per record: `Err(ProofError::FormatError)` for a wrong version byte or a non-canonical scalar
/// (what `R1CSProof::from_bytes` rejects); the proof bytes of a rejected record are zeroed.
pub fn proofs_from_wire(n: usize, mode: i32, count: usize, wire: &[u8]) -> Result<(Vec<u8>, Vec<Result<(), ProofError>>), ProofError> {
    let plen = unsafe { sys::bpp_acproof_proof_len_mode(n, mode) };
    let mut proofs = vec![0u8; count * plen];
    let mut status = vec![0u8; count];
    if count == 0 || wire.len() % count != 0 { return Err(ProofError::FormatError); }
    let rc = unsafe { sys::bpp_acproof_from_wire(n, mode, count, wire.as_ptr(), wire.len() / count, proofs.as_mut_ptr(), status.as_mut_ptr()) };
    if rc != 0 { return Err(ProofError::FormatError); }          // record length does not match the circuit
    Ok((proofs, status.into_iter().map(|s| if s == 0 { Ok(()) } else { Err(ProofError::FormatError) }).collect()))
}

// ---- many independent large MSMs: two in flight (bpp_msm_submit_dev / bpp_msm_wait_previous / bpp_msm_wait) ---
// `d_scalars[i]` / `d_out[i & 1]` are device pointers of the caller (e.g. from cust / cudarc); `consume(i, ptr)`
// enqueues whatever reads result i on the context's stream.  Same bytes as one bpp_msm_vartime_dev call per MSM.
pub unsafe fn msm_stream(points: *const sys::bpp_points, n: usize, d_scalars: &[*const core::ffi::c_void],
                         d_out: [*mut core::ffi::c_void; 2], mut consume: impl FnMut(usize, *mut core::ffi::c_void)) {
    with_ctx(|ctx| {
        for (i, sc) in d_scalars.iter().enumerate() {
            assert_eq!(sys::bpp_msm_submit_dev(ctx, *sc, points, 0, n, d_out[i & 1]), 0);
            assert_eq!(sys::bpp_msm_wait_previous(ctx), 0);      // results up to i - 1 are valid in stream order
            if i > 0 { consume(i - 1, d_out[(i - 1) & 1]); }
        }
        assert_eq!(sys::bpp_msm_wait(ctx), 0);
        if !d_scalars.is_empty() { consume(d_scalars.len() - 1, d_out[(d_scalars.len() - 1) & 1]); }
    })
}
