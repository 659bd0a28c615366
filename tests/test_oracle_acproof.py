"""CPU tests: the protocol oracle (Python restatement of circuit_lib.rs) and its C restatement agree,
the corrected circuit is satisfiable / sound on small decks, and the product's host-side weights
module agrees with the oracle's."""
import pytest

from oracle import acproof as A, cref, ristretto255 as R
from oracle.chacha import ChaChaRng

L = R.L


def _sb(v):
    return b"".join(R.sc_bytes(s) for s in v)


def _dense_bytes(M):
    return b"".join(_sb(r) for r in M)


def _c_instance(core):
    return cref.AcpInstance(core["n"], core["Q"], core["m"], _dense_bytes(core["W_L"]), _dense_bytes(core["W_R"]),
                            _dense_bytes(core["W_O"]), _dense_bytes(core["W_V"]), _sb(core["c_vec"]),
                            R.compress(core["g_base"]), R.compress(core["h_base"]),
                            b"".join(R.compress(p) for p in core["G_vec"]), b"".join(R.compress(p) for p in core["H_vec"]))


@pytest.mark.parametrize("k", [2, 3, 6])
def test_circuit_is_satisfied_and_flow_is_complete_and_sound(k):
    rng = ChaChaRng(bytes([k]) * 32)
    core, prover, V = A.make_instance(k, rng)
    lhs = [(a + b + c) % L for a, b, c in zip(A.mv_mult(core["W_L"], prover["a_L"]), A.mv_mult(core["W_R"], prover["a_R"]),
                                             A.mv_mult(core["W_O"], prover["a_O"]))]
    rhs = [(a + b) % L for a, b in zip(A.mv_mult(core["W_V"], prover["v"]), core["c_vec"])]
    assert lhs == rhs
    assert all(a * b % L == c for a, b, c in zip(prover["a_L"], prover["a_R"], prover["a_O"]))
    pb, ok, _, _ = A.run_flow(core, prover, V, ChaChaRng(b"\x01" * 32), "reference-fixed")
    assert ok and len(pb) == 32 * (11 + 2 * core["n"])
    pb0, ok0, _, _ = A.run_flow(core, prover, V, ChaChaRng(b"\x01" * 32), "reference")
    assert not ok0                      # circuit_lib.rs:541-544: the reference verifier never accepts
    assert pb0[:96] == pb[:96]          # A_I, A_O, S do not depend on the defects
    # a non-permutation is rejected: change one shuffled card
    bad_v = list(prover["v"])
    bad_v[k] = (bad_v[k] + 1) % L
    x = bad_v[-1]
    a_L, a_R, a_O = [0] * (2 * k), [0] * (2 * k), [0] * (2 * k)
    for gb, vb in ((0, 0), (k - 1, k)):
        for i in range(k - 1):
            a_L[gb + i] = (bad_v[vb] - x) % L if i == 0 else a_O[gb + i - 1]
            a_R[gb + i] = (bad_v[vb + i + 1] - x) % L
            a_O[gb + i] = a_L[gb + i] * a_R[gb + i] % L
    V2 = A.commit_variables(bad_v, prover["gamma"], core["g_base"], core["h_base"])
    _, ok2, _, _ = A.run_flow(core, dict(prover, a_L=a_L, a_R=a_R, a_O=a_O, v=bad_v), V2, ChaChaRng(b"\x01" * 32),
                              "reference-fixed")
    assert not ok2


@pytest.mark.parametrize("k", [2, 4])
@pytest.mark.parametrize("mode", [("reference-fixed", 1), ("reference", 0)])
def test_c_restatement_equals_python_oracle(k, mode):
    rng = ChaChaRng(bytes([k + 100]) * 32)
    core, prover, V = A.make_instance(k, rng)
    inst = _c_instance(core)
    Vp = inst.commit(_sb(prover["v"]), _sb(prover["gamma"]))
    assert cref.compress(Vp) == b"".join(R.compress(p) for p in V)
    for sd in (b"\x05" * 32, b"\x06" * 32):
        pb, rc = inst.prove_verify(_sb(prover["a_L"]), _sb(prover["a_R"]), _sb(prover["a_O"]), _sb(prover["gamma"]), Vp, sd, mode[1])
        want, ok, _, _ = A.run_flow(core, prover, V, ChaChaRng(sd), mode[0])
        assert pb == want and bool(rc) == ok


def test_reference_weights_as_coded_and_product_weights_module():
    import bpperm_b200
    W = bpperm_b200.weights
    for k in (2, 3):
        assert W.create_weights(k) == A.create_weights(k)
        v = [A.give_n(i) for i in range(1, k + 1)] * 2 + [1]
        assert W.create_a(v) == A.create_a(v)
        assert W.create_constants(4 * k) == A.create_constants(4 * k)
    wl, wr, wo, wv = A.create_weights(2)
    assert len(wl) == 8 and len(wl[0]) == 4 and len(wv[0]) == 5       # Q x n, Q x (n+1): weights.rs:133-136
    assert len(A.transpose(wl)) == 4 and W.transpose(wl) == A.transpose(wl)
    for k in (2, 5, 52):
        assert W.shuffle_circuit(k) == A.shuffle_circuit(k)
    n, Q, m = W.shuffle_circuit(52)[:3]
    assert (n, Q, m) == (104, 208, 105)                               # SURVEY 2.2 sizes at 52 cards
    rng = ChaChaRng(b"\x33" * 32)
    v, a_L, a_R, a_O = A.shuffle_witness(5, rng)
    perm = [v[:5].index(c) for c in v[5:10]]
    assert W.shuffle_witness(5, perm, v[-1]) == (v, a_L, a_R, a_O)


def test_transcript_vec_scalar_encoding_is_stable():
    t = A.Transcript(b"test")
    t.append_vec_scalar(b"l", [0, 1, L - 1])
    assert len(t.challenge_bytes(b"c", 8)) == 8


# ---- the verifier from proof bytes: oracle.acproof.verify_proof_bytes and cref.AcpInstance.verify -------------------
def _flow(k, seed, mode):
    core, prover, V = A.make_instance(k, ChaChaRng(bytes([seed]) * 32))
    pb, ok, _, _ = A.run_flow(core, prover, V, ChaChaRng(bytes([seed + 1]) * 32), mode)
    return core, V, pb, ok


def _both(core, inst, V_enc, proof, mode):
    """(Python, C) decisions; the C side decodes the commitments itself."""
    py = A.verify_proof_bytes(core, V_enc, proof, mode)
    c = inst.verify(proof, None, mode, V_enc=b"".join(V_enc))
    return py, c


def _sc_field(proof, f, value):
    return proof[:32 * f] + value.to_bytes(32, "little") + proof[32 * f + 32:]


@pytest.mark.parametrize("k", [2, 3, 5])
@pytest.mark.parametrize("mode", [("reference-fixed", 1), ("reference", 0)])
def test_from_bytes_verifiers_equal_run_flow_on_honest_proofs(k, mode):
    core, V, pb, ok = _flow(k, 60 + k, mode[0])
    assert ok == (mode[1] == 1)
    inst = _c_instance(core)
    V_enc = [R.compress(p) for p in V]
    assert A.verify_proof_bytes(core, V_enc, pb, mode[0]) == ok
    assert A.verify_proof_bytes(core, b"".join(V_enc), pb, mode[1]) == ok
    assert inst.verify(pb, None, mode[1], V_enc=b"".join(V_enc)) == ok
    Vp = cref.decompress(b"".join(V_enc))
    assert inst.verify(pb, Vp, mode[1]) == ok                      # the transcript binds the compressed points
    assert inst.verify(pb, Vp, mode[1], V_enc=b"".join(V_enc)) == ok
    # the same bytes under the other transcript label are a different proof
    assert not A.verify_proof_bytes(core, V_enc, pb, mode[0], label=b"other")
    assert not inst.verify(pb, Vp, mode[1], label=b"other")


def _corruptions(pb, n):
    """(name, proof bytes): every 32-byte field with a bit flip, each point field with another valid point, the
    identity, an invalid encoding and bit 255 set; each scalar field with +1 mod l, s + l and bit 255 set; A_I <-> A_O."""
    out = []
    other = R.compress(R.pt_mul(7, R.BASEPOINT))
    for f in range(11 + 2 * n):
        b = bytearray(pb)
        b[32 * f + (f % 31)] ^= 1 << (f % 8)
        out.append((f"flip{f}", bytes(b)))
        if f < 8:
            out.append((f"other{f}", pb[:32 * f] + other + pb[32 * f + 32:]))
            out.append((f"identity{f}", pb[:32 * f] + bytes(32) + pb[32 * f + 32:]))
            out.append((f"invalid{f}", pb[:32 * f] + b"\x01" + bytes(31) + pb[32 * f + 32:]))
            s = int.from_bytes(pb[32 * f:32 * f + 32], "little")
            out.append((f"bit255_{f}", _sc_field(pb, f, s | 1 << 255)))
        else:
            s = int.from_bytes(pb[32 * f:32 * f + 32], "little")
            out.append((f"plus1_{f}", _sc_field(pb, f, (s + 1) % L)))
            out.append((f"plusl_{f}", _sc_field(pb, f, s + L)))
            out.append((f"bit255_{f}", _sc_field(pb, f, s | 1 << 255)))
    out.append(("swapAIAO", pb[32:64] + pb[:32] + pb[64:]))
    return out


@pytest.mark.parametrize("mode", [("reference-fixed", 1), ("reference", 0)])
def test_from_bytes_verifiers_agree_on_a_tamper_matrix(mode):
    k = 2
    core, V, pb, ok = _flow(k, 70, mode[0])
    n, m = core["n"], core["m"]
    inst = _c_instance(core)
    V_enc = [R.compress(p) for p in V]
    want_accept = set()
    for name, bad in _corruptions(pb, n):
        py, c = _both(core, inst, V_enc, bad, mode[0])
        assert py == c, name
        if py:
            want_accept.add(name)
    # s + l is s to the verifier: only those stay accepted, and only where the honest proof is
    assert want_accept == ({f"plusl_{f}" for f in range(8, 11 + 2 * n)} if ok else set())
    # the commitments: one V_j replaced by another valid point, by an invalid encoding, by the identity
    for j in (0, m - 1):
        for name, enc in (("other", R.compress(R.pt_mul(5, R.BASEPOINT))), ("invalid", b"\x01" + bytes(31)),
                          ("identity", bytes(32))):
            V2 = list(V_enc)
            V2[j] = enc
            assert _both(core, inst, V2, pb, mode[0]) == (False, False), (name, j)


def test_scalar_taken_mod_l_pinned():
    """tau_x + l decodes to tau_x (accepted); tau_x + 1 is another scalar (rejected)."""
    core, V, pb, ok = _flow(3, 80, "reference-fixed")
    assert ok
    inst = _c_instance(core)
    V_enc = [R.compress(p) for p in V]
    tau_x = int.from_bytes(pb[256:288], "little")
    assert _both(core, inst, V_enc, _sc_field(pb, 8, tau_x + L), 1) == (True, True)
    assert _both(core, inst, V_enc, _sc_field(pb, 8, (tau_x + 1) % L), 1) == (False, False)
