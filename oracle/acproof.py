"""Restatement of the reference's operator layer and arithmetic-circuit protocol.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Every function cites the reference code it
follows (paths relative to /root/reference/bp-perm/src/).  Scalars are Python ints mod l,
points are oracle.ristretto255 tuples.

Modes (SURVEY.md A.3):
  "reference"        bit-for-bit what the reference code does, including its defects 1-5; its
                     verify() rejects every input (circuit_lib.rs:541-544) - that IS the
                     reference's accept/reject behaviour.
  "reference-fixed"  defects 2-5 corrected (T_i commit to the coefficients t_i, "T4" carries T_4,
                     the x^2<z,W_V gamma> term once, cand_P over h'), check 3 enabled.  Defect 1
                     (exp_iter yields Fibonacci exponents) is kept: it is operator-level behaviour
                     of util.rs::exp_iter and does not affect completeness.
"""
from __future__ import annotations

from . import ristretto255 as R
from .merlin import Transcript

L = R.L


# ------------------------------------------------------------------ util.rs ---------------
def hadamard_V(a, b):  # util.rs:6-20
    if len(a) != len(b):
        raise ValueError(f"hadamard_V(a, b): {len(a)} and {len(b)} should have same size")
    return [(x * y) % L for x, y in zip(a, b)]


def inner_product(a, b):  # util.rs:84-94
    if len(a) != len(b):
        raise ValueError(f"inner_product(a,b): lengths dont match, {len(a)}, {len(b)}")
    out = 0
    for x, y in zip(a, b):
        out = (out + x * y) % L
    return out


def vm_mult(a, b):  # util.rs:22-38: out[i] = <a, b[i]>
    if len(a) != len(b[0]):
        raise ValueError("vm_mult(a,b): dimension mismatch")
    return [inner_product(a, row) for row in b]


def mv_mult(a, b):  # util.rs:40-56: out[j] = sum_i a[i][j] * b[i]
    if len(a) != len(b):
        raise ValueError("mv_mult(a,b): dimension mismatch")
    cols = len(a[0])
    return [inner_product([a[i][j] for i in range(len(a))], b) for j in range(cols)]


def lm_mult(a, b):  # util.rs:58-61
    return vm_mult(list(a), b)


def exp_iter(x, count):
    """util.rs:63-65,139-157.  The reference iterator overwrites its base with the value it
    returns, so it yields x^F(i): x, x, x^2, x^3, x^5, x^8, ... (Fibonacci exponents)."""
    base, nxt = 1, x % L
    out = []
    for _ in range(count):
        exp_x = nxt
        nxt = (nxt * base) % L
        base = exp_x
        out.append(exp_x)
    return out


def scalar_exp(x, pow_):  # util.rs:67-82
    r = 1
    for _ in range(pow_):
        r = (r * x) % L
    return r


def give_n(n):  # util.rs:96-103
    return n % L


# ------------------------------------------------------------------ poly.rs ---------------
class Poly6:  # poly.rs:5-18
    def __init__(self, t1, t2, t3, t4, t5, t6):
        self.t = [t1, t2, t3, t4, t5, t6]

    def eval(self, x):
        t1, t2, t3, t4, t5, t6 = self.t
        return (x * (t1 + x * (t2 + x * (t3 + x * (t4 + x * (t5 + x * t6)))))) % L


class VecPoly3:  # poly.rs:21-76
    def __init__(self, n):
        self.c = [[0] * n for _ in range(4)]

    @staticmethod
    def special_inner_product(lhs, rhs):  # poly.rs:39-55
        l, r = lhs.c, rhs.c
        ip = inner_product
        return Poly6(ip(l[1], r[0]),
                     (ip(l[1], r[1]) + ip(l[2], r[0])) % L,
                     (ip(l[2], r[1]) + ip(l[3], r[0])) % L,
                     (ip(l[1], r[3]) + ip(l[3], r[1])) % L,
                     ip(l[2], r[3]),
                     ip(l[3], r[3]))

    def eval(self, x):  # poly.rs:57-76
        c = self.c
        return [(c[0][i] + x * (c[1][i] + x * (c[2][i] + x * c[3][i]))) % L for i in range(len(c[0]))]


# ------------------------------------------------------------------ weights.rs ------------
def create_constants(Q):  # weights.rs:26-36
    return [0] * (Q - 2) + [L - 1, 1]


def transpose(v):  # weights.rs:115-129
    return [list(col) for col in zip(*v)]


def create_weights(card_count):
    """weights.rs:130-204, exactly as coded (Q x n layout, only meaningful for k in {2,3})."""
    n = card_count * 2
    Q = n * 2
    w_l = [[0] * n for _ in range(Q)]
    w_r = [[0] * n for _ in range(Q)]
    w_o = [[0] * n for _ in range(Q)]
    w_v = [[0] * (n + 1) for _ in range(Q)]
    for i in range(Q):
        if i < n:
            w_l[i][i] = 1
            if i != card_count // 2 + 1 and i != 0:
                w_o[i][i - 1] = 1
            else:
                w_v[i][n] = L - 1
                if i == 0:
                    w_v[i][i] = 1
                else:
                    w_v[i][i + 1] = 1
        else:
            w_r[i][i - n] = 1
            if i < Q - 2:
                w_v[i][n] = L - 1
                if i < n + 3:
                    w_v[i][i - n + 1] = 1
                else:
                    w_v[i][i - n + 2] = 1
    w_o[n - 1][card_count - 1] = 1
    return w_l, w_r, w_o, w_v


def create_a(variables):
    """weights.rs:63-113, exactly as coded."""
    n = len(variables) - 1
    a_L, a_R, a_O = [0] * n, [0] * n, [0] * n
    first, second = variables[:n // 2], variables[n // 2:n]
    x = variables[-1]
    offset = (n - 1) // 2
    for i in range(len(first) - 1):
        a_R[i] = (first[i + 1] - x) % L
        a_R[i + offset] = (second[i + 1] - x) % L
        if i == 0:
            a_L[i] = (first[i] - x) % L
            a_L[i + offset] = (second[i] - x) % L
        else:
            a_L[i] = a_O[i - 1]
            a_L[i + offset] = a_O[i + offset - 1]
        a_O[i] = a_L[i] * a_R[i] % L
        a_O[i + offset] = a_L[i + offset] * a_R[i + offset] % L
    a_L[n - 2] = a_O[n - 3]
    a_R[n - 2] = L - 1
    a_O[n - 2] = a_L[n - 2] * a_R[n - 2] % L
    a_L[n - 1] = (a_O[offset] + a_O[n - 2]) % L
    a_R[n - 1] = 1
    a_O[n - 1] = a_L[n - 1] * a_L[n - 1] % L
    return a_L, a_R, a_O


# ---- the corrected k-card shuffle circuit (SURVEY 8f-1), same shape as the reference:
#      n = 2k multipliers, Q = 2n constraints, m = 2k+1 committed values --------------------
def shuffle_circuit(k):
    """Sparse circuit for prod_i (v_i - X) == prod_i (v_{k+i} - X), X = v[2k].
    Returns (n, Q, m, W_L, W_R, W_O, W_V, c) with each W as a list of (wire, constraint, coeff)
    triples; constraint q reads  sum W_L a_L + W_R a_R + W_O a_O = sum W_V v + c."""
    assert k >= 2
    n, Q, m = 2 * k, 4 * k, 2 * k + 1
    WL, WR, WO, WV = [], [], [], []
    q = 0
    for gb, vb in ((0, 0), (k - 1, k)):
        WL.append((gb, q, 1)); WV.append((vb, q, 1)); WV.append((2 * k, q, L - 1)); q += 1
        for i in range(k - 1):
            WR.append((gb + i, q, 1)); WV.append((vb + i + 1, q, 1)); WV.append((2 * k, q, L - 1)); q += 1
        for i in range(1, k - 1):
            WL.append((gb + i, q, 1)); WO.append((gb + i - 1, q, L - 1)); q += 1
    WO.append((k - 2, q, 1)); WO.append((2 * k - 3, q, L - 1)); q += 1
    WL.append((2 * k - 2, q, 1)); q += 1
    WL.append((2 * k - 1, q, 1)); q += 1
    assert q == Q - 1
    return n, Q, m, WL, WR, WO, WV, [0] * Q


def shuffle_witness(k, rng, x=None):
    """Deck 1..k, a Fisher-Yates permutation drawn from the RNG stream, challenge value X.
    (weights.rs:38-56 uses the un-vendored `shuffle` crate with thread_rng and fixes X = 1.)"""
    deck = [give_n(i) for i in range(1, k + 1)]
    perm = list(deck)
    for i in range(k - 1, 0, -1):
        j = int.from_bytes(rng.fill_bytes(8), "little") % (i + 1)
        perm[i], perm[j] = perm[j], perm[i]
    if x is None:
        x = rng.scalar()
    v = deck + perm + [x]
    n = 2 * k
    a_L, a_R, a_O = [0] * n, [0] * n, [0] * n
    for gb, vb in ((0, 0), (k - 1, k)):
        for i in range(k - 1):
            a_L[gb + i] = (v[vb] - x) % L if i == 0 else a_O[gb + i - 1]
            a_R[gb + i] = (v[vb + i + 1] - x) % L
            a_O[gb + i] = a_L[gb + i] * a_R[gb + i] % L
    return v, a_L, a_R, a_O


def dense(triples, rows, cols):
    """(wire, constraint, coeff) triples -> the reference's dense rows x Q matrices (A.1 layout)."""
    M = [[0] * cols for _ in range(rows)]
    for i, q, c in triples:
        M[i][q] = (M[i][q] + c) % L
    return M


def commit_variables(v, gamma, g, h):  # weights.rs:58-61 / PedersenGens::commit: v*B + r*B_blinding
    return [R.pt_add(R.pt_mul(vi, g), R.pt_mul(ri, h)) for vi, ri in zip(v, gamma)]


V_CHUNK = 64


def commitment_digests(V):
    """One 32-byte digest per chunk of V_CHUNK commitments: a Merlin transcript of its own, Transcript::new(b"acp-V"),
    append_u64(b"chunk", index), append_message(b"V", the chunk's encodings concatenated in order),
    challenge_bytes(b"d", 32).  (Fixed-size items whose count is bound by "m" need no framing of their own.)
    The chunks are independent sponges, so a deck of thousands of commitments is hashed in parallel (one serial sponge
    over m = 8193 commitments is ~2000 Keccak permutations in a row on the critical path of every prover and verifier)."""
    enc = [Vj if isinstance(Vj, (bytes, bytearray)) else R.compress(Vj) for Vj in V]
    out = []
    for c in range(0, len(enc), V_CHUNK):
        t = Transcript(b"acp-V")
        t.append_u64(b"chunk", c // V_CHUNK)
        t.append_message(b"V", b"".join(bytes(e) for e in enc[c:c + V_CHUNK]))
        out.append(t.challenge_bytes(b"d", 32))
    return out


def append_commitments(trans: Transcript, V, m: int):
    """Binds the value commitments to the transcript: m as a u64 under the label "m", then the chunk digests of
    commitment_digests, concatenated, as one message under "Vd".  (bulletproofs 4.0.0's R1CS prover appends every V_j to the one transcript at commit
    time; the two-level form binds the same bytes and keeps the hashing off the critical path.)  V: points or encodings."""
    assert V is not None and len(V) == m
    trans.append_u64(b"m", m)
    trans.append_message(b"Vd", b"".join(commitment_digests(V)))


# ------------------------------------------------------------------ circuit_lib.rs --------
class ArithmeticCircuitProof:
    """ACProof::ArithmeticCircuitProof (circuit_lib.rs:90-585).  State lives in attributes where the
    reference keeps string-keyed hash maps (circuit_lib.rs:77-88,236-247,293-297,417-420,470-475)."""

    def __init__(self, mode="reference-fixed", msm=None):
        assert mode in ("reference", "reference-fixed")
        self.mode = mode
        self.msm = msm or R.vartime_multiscalar_mul

    # circuit_lib.rs:139-253
    @classmethod
    def create(cls, trans: Transcript, core: dict, prover: dict, rng, mode="reference-fixed", msm=None, V=None):
        """V: the value commitments (points).  The reference never binds them to the transcript (SURVEY A.3
        defect 12: weak Fiat-Shamir - the prover of a shuffle chooses the output-deck commitments, so it could pick
        the challenges first and solve check 2 for some V_j); `reference` mode reproduces that, `reference-fixed`
        appends m and every V_j right after the domain separator, as dalek's R1CS prover does at commit time."""
        self = cls(mode, msm)
        G, H = core["G_vec"], core["H_vec"]
        n = len(G)
        assert len(H) == n
        for key in ("W_L", "W_R", "W_O"):
            assert len(core[key]) == n              # :157-159
        a_L, a_R, a_O = prover["a_L"], prover["a_R"], prover["a_O"]
        assert len(a_L) == n and len(a_R) == n and len(a_O) == n
        m = len(prover["gamma"])
        assert len(core["W_V"]) == m                # :167
        Q = len(core["W_L"][0])
        for key in ("W_R", "W_O", "W_V"):
            assert len(core[key][0]) == Q
        self.core, self.prover = core, prover
        self.n, self.m, self.Q = n, m, Q
        trans.arithmetic_domain_sep(n)               # :178
        if mode != "reference":
            append_commitments(trans, V, m)
        self.alpha, self.beta, self.ro = rng.scalar(), rng.scalar(), rng.scalar()   # :180-182
        h = core["h_base"]
        self.A_I = self.msm([self.alpha] + a_L + a_R, [h] + G + H)                 # :187-200
        self.A_O = self.msm([self.beta] + a_O, [h] + G)                            # :202-210
        self.s_l = [rng.scalar() for _ in range(n)]                                # :213
        self.s_r = [rng.scalar() for _ in range(n)]                                # :214
        self.S = self.msm([self.ro] + self.s_l + self.s_r, [h] + G + H)            # :216-229
        self.A_I_c, self.A_O_c, self.S_c = R.compress(self.A_I), R.compress(self.A_O), R.compress(self.S)
        trans.append_point(b"A_I", self.A_I_c)       # :231-233
        trans.append_point(b"A_O", self.A_O_c)
        trans.append_point(b"S", self.S_c)
        return self

    def challenge_wit_and_const(self, trans):        # :133-138
        y = trans.challenge_scalar(b"y")
        z = trans.challenge_scalar(b"z")
        return y, z

    def compute_per_challenges(self, y, z):          # :256-302
        core = self.core
        self.y_n = exp_iter(y, self.n)
        self.y_n_inv = [R.sc_inv(k) for k in self.y_n]
        z_q = exp_iter(z, self.Q)
        self.z_W_R = vm_mult(z_q, core["W_R"])
        self.l_in = hadamard_V(self.y_n_inv, self.z_W_R)
        self.z_W_L = vm_mult(z_q, core["W_L"])
        sigma = inner_product(self.l_in, self.z_W_L)
        return self.y_n, z_q, sigma

    def commit_Ts(self, trans, y_n, z_q, sigma, rng):  # :304-423
        core, p, n = self.core, self.prover, self.n
        l_x, r_x = VecPoly3(n), VecPoly3(n)
        l_x.c[1] = [(a + b) % L for a, b in zip(p["a_L"], self.l_in)]
        l_x.c[2] = list(p["a_O"])
        l_x.c[3] = list(self.s_l)
        r_x.c[0] = [(a - b) % L for a, b in zip(vm_mult(z_q, core["W_O"]), y_n)]
        r_x.c[1] = [(a + b) % L for a, b in zip(hadamard_V(y_n, p["a_R"]), vm_mult(z_q, core["W_L"]))]
        r_x.c[3] = hadamard_V(y_n, self.s_r)
        t_x = VecPoly3.special_inner_product(l_x, r_x)
        self.t_poly = t_x
        # :344-356 compute w and t_2 and discard them; no observable effect, not restated.
        g, h = core["g_base"], core["h_base"]
        self.taus, Ts = [], []
        for deg, label in ((1, b"T1"), (3, b"T3"), (4, b"T4"), (5, b"T5"), (6, b"T6")):
            tau = rng.scalar()                                                     # :361,371,382,393,404
            if self.mode == "reference":
                t_i = t_x.eval(deg)           # defect 2: the polynomial evaluated at the integer i
            else:
                t_i = t_x.t[deg - 1]          # the coefficient t_i
            T = R.compress(self.msm([t_i, tau], [g, h]))
            self.taus.append(tau)
            Ts.append(T)
            if self.mode == "reference" and label == b"T4":
                trans.append_point(b"T4", Ts[1])   # defect 3: "T4" carries T_3's bytes (:391)
            else:
                trans.append_point(label, T)
        self.l_x, self.r_x = l_x, r_x
        return Ts

    def random_chall_x(self, trans):                 # :425-432
        return trans.challenge_scalar(b"x")

    def blinding_values(self, trans, x, z_q):        # :434-476
        self.l = self.l_x.eval(x)
        self.r = self.r_x.eval(x)
        self.t = inner_product(self.l, self.r)
        wv_gamma = inner_product(z_q, mv_mult(self.core["W_V"], self.prover["gamma"]))
        xx = x * x % L
        tau_x = 0
        for tau, deg in zip(self.taus, (1, 3, 4, 5, 6)):
            tau_x = (tau_x + tau * scalar_exp(x, deg)) % L
            if self.mode == "reference":
                tau_x = (tau_x + xx * wv_gamma) % L      # defect 4: added five times (:452-456)
        if self.mode != "reference":
            tau_x = (tau_x + xx * wv_gamma) % L
        self.tau_x = tau_x
        self.mu = (self.alpha * x + self.beta * scalar_exp(x, 2) + self.ro * scalar_exp(x, 3)) % L   # :462
        trans.append_scalar(b"TX", self.tau_x)       # :464-468
        trans.append_scalar(b"mu", self.mu)
        trans.append_vec_scalar(b"l", self.l)
        trans.append_vec_scalar(b"r", self.r)
        trans.append_scalar(b"t", self.t)

    def proof_bytes(self, Ts) -> bytes:
        """The observable outputs in a fixed order (the reference has no serialisation):
        A_I, A_O, S, T_1, T_3, T_4, T_5, T_6, tau_x, mu, t, l[0..n), r[0..n)."""
        out = self.A_I_c + self.A_O_c + self.S_c + b"".join(Ts)
        out += R.sc_bytes(self.tau_x) + R.sc_bytes(self.mu) + R.sc_bytes(self.t)
        out += b"".join(R.sc_bytes(s) for s in self.l) + b"".join(R.sc_bytes(s) for s in self.r)
        return out

    def verify(self, trans, z_q, sigma, x, V, Ts):   # :478-585; returns True for Ok(()), False for Err
        core, n = self.core, self.n
        g, h, G, H = core["g_base"], core["h_base"], core["G_vec"], core["H_vec"]
        h_ = [R.pt_mul(yi, Hi) for yi, Hi in zip(self.y_n_inv, H)]                 # :491
        weights_L = self.msm(self.z_W_L, h_)                                       # :498
        weights_R = self.msm(self.l_in, G)                                         # :504
        weights_O = self.msm(vm_mult(z_q, core["W_O"]), h_)                        # :509
        if self.t != inner_product(self.l, self.r):                                # :518
            return False
        xx = scalar_exp(x, 2)
        g_exp = xx * (inner_product(z_q, core["c_vec"]) + sigma) % L
        v_exp = [xx * i % L for i in vm_mult(z_q, core["W_V"])]
        t_exp = [x] + [scalar_exp(x, i) for i in range(3, 7)]
        T_pts = []
        for T in Ts:
            pt = R.decompress(T)
            if pt is None:
                raise ValueError("decompress().unwrap() on an invalid T (circuit_lib.rs:532 panics)")
            T_pts.append(pt)
        cand = self.msm([g_exp] + v_exp + t_exp, [g] + list(V) + T_pts)            # :525-533
        lhs = self.msm([self.t, self.tau_x], [g, h])                              # :535-538
        if not R.pt_eq(lhs, cand):                                                 # :541
            return False
        neg_y_n = [(L - i) % L for i in self.y_n]
        P = self.msm([x, xx] + neg_y_n + [x, x, 1, scalar_exp(x, 3)],
                     [self.A_I, self.A_O] + h_ + [weights_L, weights_R, weights_O, self.S])   # :552-565
        base_H = H if self.mode == "reference" else h_                              # defect 5 (:574)
        cand_P = self.msm([self.mu] + self.l + self.r, [h] + G + base_H)            # :568-575
        if self.mode == "reference":
            return True      # :577-582 the comparison is commented out
        return R.pt_eq(P, cand_P)


def run_flow(core, prover, V, rng, mode="reference-fixed", label=b"test", msm=None):
    """The 7-step call order of lib.rs:219-231.  Returns (proof_bytes, accepted, challenges)."""
    trans = Transcript(label)                                                       # lib.rs:172
    proof = ArithmeticCircuitProof.create(trans, core, prover, rng, mode, msm, V)
    y, z = proof.challenge_wit_and_const(trans)
    y_n, z_q, sigma = proof.compute_per_challenges(y, z)
    Ts = proof.commit_Ts(trans, y_n, z_q, sigma, rng)
    x = proof.random_chall_x(trans)
    proof.blinding_values(trans, x, z_q)
    ok = proof.verify(trans, z_q, sigma, x, V, Ts)
    return proof.proof_bytes(Ts), ok, (y, z, x), proof


def verify_proof_bytes(core, V_enc, proof: bytes, mode="reference-fixed", label=b"test", msm=None) -> bool:
    """The verifier of circuit_lib.rs:478-585 from the proof bytes alone, where ArithmeticCircuitProof.verify reads the
    prover's own state.  proof: A_I, A_O, S, T_1, T_3..T_6, tau_x, mu, t, l[0..n), r[0..n) as proof_bytes writes them;
    V_enc: the m commitments' encodings (a list, or their concatenation).  The transcript is replayed from these bytes
    as create .. random_chall_x append them (mode "reference-fixed"/1: with append_commitments; "reference"/0: without,
    and "T4" carries T_3's bytes), then checks 1-3 run as in verify(), defects and corrections included.
    Decoding rules, those of the library's verifier: a scalar >= l is taken mod l; an undecodable point or commitment is
    a reject (the reference would panic on an undecodable T, circuit_lib.rs:532); the all-zero encoding is the identity."""
    mode = {0: "reference", 1: "reference-fixed"}.get(mode, mode)
    n, Q, m = len(core["G_vec"]), len(core["W_L"][0]), len(core["W_V"])
    if isinstance(V_enc, (bytes, bytearray)):
        V_enc = [bytes(V_enc[32 * j:32 * j + 32]) for j in range(len(V_enc) // 32)]
    if len(proof) != 32 * (11 + 2 * n) or len(V_enc) != m:
        raise ValueError("proof: 32 (11 + 2 n) bytes; V_enc: m encodings")
    enc = [bytes(proof[32 * i:32 * i + 32]) for i in range(11 + 2 * n)]
    pts = [R.decompress(e) for e in enc[:8]]
    V = [R.decompress(bytes(e)) for e in V_enc]
    if any(p is None for p in pts + V):
        return False
    sc = [int.from_bytes(e, "little") % L for e in enc[8:]]
    self = ArithmeticCircuitProof(mode, msm)
    self.core, self.n, self.m, self.Q = core, n, m, Q
    self.A_I, self.A_O, self.S = pts[:3]
    self.tau_x, self.mu, self.t = sc[:3]
    self.l, self.r = sc[3:3 + n], sc[3 + n:]
    trans = Transcript(label)
    trans.arithmetic_domain_sep(n)
    if mode != "reference":
        append_commitments(trans, V_enc, m)
    for lab, e in zip((b"A_I", b"A_O", b"S"), enc[:3]):
        trans.append_point(lab, e)
    y, z = self.challenge_wit_and_const(trans)
    _, z_q, sigma = self.compute_per_challenges(y, z)
    Ts = enc[3:8]
    for lab, e in zip((b"T1", b"T3", b"T4", b"T5", b"T6"), Ts):
        trans.append_point(lab, Ts[1] if mode == "reference" and lab == b"T4" else e)
    x = self.random_chall_x(trans)
    return self.verify(trans, z_q, sigma, x, V, Ts)


def make_instance(k, rng, dense_weights=True):
    """Synthetic k-card instance in the reference's shapes: generators as RistrettoPoint::random
    (lib.rs:164-167,179-180), the corrected shuffle circuit, witness, blindings, commitments.
    RNG draw order: B, B_blinding, G[0..n), H[0..n), permutation, X, gamma[0..m)."""
    g, h = rng.point(), rng.point()
    n, Q, m, WL, WR, WO, WV, c = shuffle_circuit(k)
    G = [rng.point() for _ in range(n)]
    H = [rng.point() for _ in range(n)]
    v, a_L, a_R, a_O = shuffle_witness(k, rng)
    gamma = [rng.scalar() for _ in range(m)]
    V = commit_variables(v, gamma, g, h)
    core = {"g_base": g, "h_base": h, "G_vec": G, "H_vec": H, "c_vec": c, "sparse": (WL, WR, WO, WV),
            "n": n, "Q": Q, "m": m}
    if dense_weights:
        core.update(W_L=dense(WL, n, Q), W_R=dense(WR, n, Q), W_O=dense(WO, n, Q), W_V=dense(WV, m, Q))
    prover = {"a_L": a_L, "a_R": a_R, "a_O": a_O, "gamma": gamma, "v": v}
    return core, prover, V
