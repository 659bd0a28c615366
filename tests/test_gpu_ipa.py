"""GPU parity for the `fixed` protocol mode (SURVEY 8 row a16: inner-product argument): proof bytes and
accept/reject decisions against oracle/ipa.py (Python) and oracle/c (C restatement that folds the generators
explicitly like bulletproofs 4.0.0, while the CUDA path folds the scalars)."""
import pytest

from oracle import cref, ipa, ristretto255 as R
from oracle.chacha import ChaChaRng

pytestmark = pytest.mark.gpu
L = R.L


def _sb(v):
    return b"".join(R.sc_bytes(s) for s in v)


def _setup(backend, k, seed, window_bits=0):
    from bpperm_b200 import acproof as G
    rng = ChaChaRng(bytes([seed]) * 32)
    core, prover, V = ipa.make_instance(k, rng, dense_weights=k <= 16)
    WL, WR, WO, WV = core["sparse"]
    cir = G.Circuit(backend, core["n"], core["Q"], core["m"], WL, WR, WO, WV, core["c_vec"])
    gens = G.Generators(backend, R.compress(core["g_base"]), R.compress(core["h_base"]),
                        [R.compress(p) for p in core["G_vec"]], [R.compress(p) for p in core["H_vec"]], window_bits)
    return core, prover, V, cir, gens, cref.AcpFixedInstance.from_core(core)


@pytest.mark.parametrize("k", [2, 3, 5, 8])
def test_small_decks_fixed_mode_bytes_and_decisions(backend, k):
    from bpperm_b200 import acproof as G
    core, prover, V, cir, gens, inst = _setup(backend, k, 60 + k)
    seeds = [bytes([i + 1]) * 32 for i in range(3)]
    B = len(seeds)
    n = core["n"]
    Vc = b"".join(R.compress(p) for p in V)
    proofs = G.prove_batch(backend, cir, gens, _sb(prover["a_L"]) * B, _sb(prover["a_R"]) * B, _sb(prover["a_O"]) * B,
                           _sb(prover["gamma"]) * B, b"".join(seeds), B, "fixed", V=Vc * B)
    plen = G.proof_len(n, "fixed")
    assert plen == ipa.proof_len(n) and len(proofs) == B * plen
    for i, sd in enumerate(seeds):
        pb, _ = ipa.prove(core, prover, V, ChaChaRng(sd))
        assert proofs[i * plen:(i + 1) * plen] == pb, (k, i)
        assert ipa.verify(core, V, pb)
    assert list(G.verify_batch(backend, cir, gens, proofs, Vc * B, B, "fixed")) == [1] * B


def test_52_card_fixed_mode_proof_is_byte_identical_to_the_c_restatement(backend):
    """BASELINE configs[1] in `fixed` mode: k = 52 -> n = 104 padded to 128, 7 rounds, 864-byte proofs."""
    from bpperm_b200 import acproof as G
    core, prover, V, cir, gens, inst = _setup(backend, 52, 53)
    seeds = [b"\x77" * 32, b"\x78" * 32, b"\x79" * 32]
    B = len(seeds)
    Vp = inst.commit(_sb(prover["v"]), _sb(prover["gamma"]))
    Vc = cref.compress(Vp)
    proofs = G.prove_batch(backend, cir, gens, _sb(prover["a_L"]) * B, _sb(prover["a_R"]) * B, _sb(prover["a_O"]) * B,
                           _sb(prover["gamma"]) * B, b"".join(seeds), B, "fixed", V=Vc * B)
    plen = G.proof_len(104, "fixed")
    assert plen == 864
    for i, sd in enumerate(seeds):
        want = inst.prove(_sb(prover["a_L"]), _sb(prover["a_R"]), _sb(prover["a_O"]), _sb(prover["gamma"]), Vp, sd)
        assert proofs[i * plen:(i + 1) * plen] == want
        assert inst.verify(want, Vp)
    assert list(G.verify_batch(backend, cir, gens, proofs, Vc * B, B, "fixed")) == [1] * B


def test_fixed_mode_tampering_matches_the_oracle_decision_per_proof(backend):
    from bpperm_b200 import acproof as G
    core, prover, V, cir, gens, inst = _setup(backend, 6, 15)
    n, m = core["n"], core["m"]
    plen = G.proof_len(n, "fixed")
    words = plen // 32
    B = words + 3
    seeds = b"".join(bytes([50 + i]) * 32 for i in range(B))
    Vp = inst.commit(_sb(prover["v"]), _sb(prover["gamma"]))
    Vc = bytearray(cref.compress(Vp) * B)
    proofs = bytearray(G.prove_batch(backend, cir, gens, _sb(prover["a_L"]) * B, _sb(prover["a_R"]) * B, _sb(prover["a_O"]) * B,
                                     _sb(prover["gamma"]) * B, seeds, B, "fixed", V=bytes(Vc)))
    assert list(G.verify_batch(backend, cir, gens, bytes(proofs), bytes(Vc), B, "fixed")) == [1] * B
    for f in range(words):                   # proof f: one bit flipped in field f
        proofs[f * plen + 32 * f + 5] ^= 0x04
    proofs[words * plen + 32 * 11: words * plen + 32 * 12] = bytes(32)                                  # identity L_0
    proofs[(words + 1) * plen + 32 * 12: (words + 1) * plen + 32 * 13] = R.compress(R.pt_mul(9, R.BASEPOINT))  # wrong R_0
    Vc[(words + 2) * 32 * m: (words + 2) * 32 * m + 32] = R.compress(R.pt_mul(5, R.BASEPOINT))          # wrong V_0
    acc = list(G.verify_batch(backend, cir, gens, bytes(proofs), bytes(Vc), B, "fixed"))
    want = []
    for i in range(B):
        Ve = bytes(Vc[i * 32 * m:(i + 1) * 32 * m])
        want.append(1 if inst.verify(bytes(proofs[i * plen:(i + 1) * plen]), cref.decompress(Ve), V_enc=Ve) else 0)
    assert acc == want
    assert sum(acc) <= 1     # a flipped high bit of a scalar field may stay the same value mod l; everything else rejects


@pytest.mark.parametrize("k,window_bits", [(200, 8), (100, 6)])
def test_larger_deck_single_proof_uses_split_msm_and_matches_c(backend, k, window_bits):
    """One proof of a 200-card deck (n = 400 -> 512, 9 rounds): the (proof, output) grid is tiny, so every
    fixed-base MSM is split over several blocks; bytes must not change."""
    from bpperm_b200 import acproof as G
    core, prover, V, cir, gens, inst = _setup(backend, k, 77, window_bits)
    sd = b"\x42" * 32
    Vp = inst.commit(_sb(prover["v"]), _sb(prover["gamma"]))
    proof = G.prove_batch(backend, cir, gens, _sb(prover["a_L"]), _sb(prover["a_R"]), _sb(prover["a_O"]), _sb(prover["gamma"]),
                          sd, 1, "fixed", V=cref.compress(Vp))
    want = inst.prove(_sb(prover["a_L"]), _sb(prover["a_R"]), _sb(prover["a_O"]), _sb(prover["gamma"]), Vp, sd)
    assert proof == want
    assert inst.verify(want, Vp)
    assert list(G.verify_batch(backend, cir, gens, proof, cref.compress(Vp), 1, "fixed")) == [1]
    # the same circuit in the other modes still needs exactly n generators
    with pytest.raises(Exception):
        G.Batch(backend, cir, gens, 1, "reference-fixed")


def _large_instance(k, seed):
    """k-card instance with generators derived by the C oracle from seeded uniform bytes (the Python oracle's
    elligator is too slow for 2^14 generators); same circuit / witness generators as the small cases."""
    import numpy as np
    from oracle import acproof as A
    n, Q, m, WL, WR, WO, WV, c = A.shuffle_circuit(k)
    npad = 1
    while npad < n:
        npad *= 2
    rs = np.random.RandomState(seed)
    enc = cref.compress(cref.from_uniform(rs.randint(0, 256, size=(2 * npad + 2, 64), dtype=np.uint8).tobytes()))
    rng = ChaChaRng(bytes([seed & 0xFF]) * 32)
    v, aL, aR, aO = A.shuffle_witness(k, rng)
    gamma = [rng.scalar() for _ in range(m)]
    g, h, Gb, Hb = enc[:32], enc[32:64], enc[64:64 + 32 * npad], enc[64 + 32 * npad:]
    inst = cref.AcpFixedInstance(n, Q, m, WL, WR, WO, WV, _sb(c), g, h, Gb, Hb)
    return (n, Q, m, npad, WL, WR, WO, WV, c), (g, h, Gb, Hb), (v, aL, aR, aO, gamma), inst


def test_large_deck_4096_cards_single_proof_is_byte_identical(backend):
    """BASELINE configs[2]: 4096 committed card values -> k = 4096, n = 8192 multipliers, 2^14 generators,
    13 inner-product rounds, one proof on one GPU; bytes and decision against the C restatement."""
    from bpperm_b200 import acproof as G
    (n, Q, m, npad, WL, WR, WO, WV, c), (g, h, Gb, Hb), (v, aL, aR, aO, gamma), inst = _large_instance(4096, 99)
    assert (n, npad, m) == (8192, 8192, 8193)
    cir = G.Circuit(backend, n, Q, m, WL, WR, WO, WV, c)
    gens = G.Generators(backend, g, h, [Gb[32 * i:32 * i + 32] for i in range(npad)], [Hb[32 * i:32 * i + 32] for i in range(npad)], 8)
    sd = b"\x42" * 32
    Vp = inst.commit(_sb(v), _sb(gamma))
    Vc = cref.compress(Vp)
    proof = G.prove_batch(backend, cir, gens, _sb(aL), _sb(aR), _sb(aO), _sb(gamma), sd, 1, "fixed", V=Vc)
    assert len(proof) == 32 * (13 + 2 * 13)
    want = inst.prove(_sb(aL), _sb(aR), _sb(aO), _sb(gamma), Vp, sd, V_enc=Vc)
    assert proof == want
    assert inst.verify(want, Vp, V_enc=Vc)
    assert list(G.verify_batch(backend, cir, gens, proof, Vc, 1, "fixed")) == [1]
    bad = bytearray(proof)
    bad[32 * 20 + 3] ^= 2      # one of the L_j
    assert list(G.verify_batch(backend, cir, gens, bytes(bad), Vc, 1, "fixed")) == [0]
    gens.free()
    cir.free()


def test_batch_verification_with_one_percent_corrupted_proofs_matches_the_oracle_per_proof(backend):
    """BASELINE configs[3] in miniature: a batch of 512 independent 52-card proofs, 6 of them (>1 %) corrupted in
    different fields; the accept bytes must equal the C restatement's decision for every single proof, with the
    combined batch check (which must fall back) and with strictly per-proof verification."""
    from bpperm_b200 import acproof as G
    core, prover, V, cir, gens, inst = _setup(backend, 52, 54, 8)
    n, m = core["n"], core["m"]
    B = 512
    plen = G.proof_len(n, "fixed")
    seeds = b"".join((1000 + i).to_bytes(4, "little") * 8 for i in range(B))
    batch = G.Batch(backend, cir, gens, B, "fixed", b"test")
    batch.upload_witness(_sb(prover["a_L"]) * B, _sb(prover["a_R"]) * B, _sb(prover["a_O"]) * B, _sb(prover["gamma"]) * B, seeds)
    Vp = inst.commit(_sb(prover["v"]), _sb(prover["gamma"]))
    Vc1 = cref.compress(Vp)
    batch.upload_commitments(Vc1 * B)
    batch.prove()
    good = batch.download_proofs()
    # all valid: the combined check decides
    batch.upload_proofs(good, Vc1 * B)
    batch.verify(b"\x21" * 32)
    assert batch.download_accept() == b"\x01" * B
    proofs, Vc = bytearray(good), bytearray(Vc1 * B)
    victims = {3: 0, 77: 5, 128: 8, 300: 11, 400: 12, 511: plen // 32 - 1}     # A_I, T_4, t, L_0, R_0, b
    for p, f in victims.items():
        if f in (0, 5, 11, 12):
            proofs[p * plen + 32 * f: p * plen + 32 * f + 32] = R.compress(R.pt_mul(p + 2, R.BASEPOINT))
        else:
            s = (int.from_bytes(proofs[p * plen + 32 * f: p * plen + 32 * f + 32], "little") + 1) % L
            proofs[p * plen + 32 * f: p * plen + 32 * f + 32] = R.sc_bytes(s)
    Vc[32 * (m * 222 + 7): 32 * (m * 222 + 8)] = R.compress(R.pt_mul(3, R.BASEPOINT))              # commitment 7 of proof 222
    want = []
    for i in range(B):
        if i in victims or i == 222 or i % 64 == 0:      # every corrupted proof + a sample of the valid ones
            Ve = bytes(Vc[i * 32 * m:(i + 1) * 32 * m])
            want.append(1 if inst.verify(bytes(proofs[i * plen:(i + 1) * plen]), cref.decompress(Ve), V_enc=Ve) else 0)
        else:
            want.append(1)
    assert sum(want) == B - 7
    for rlc in (True, False):
        batch.set_batch_rlc(rlc)
        batch.upload_proofs(bytes(proofs), bytes(Vc))
        batch.verify(b"\x21" * 32)
        assert list(batch.download_accept()) == want, rlc
    batch.free()


def test_wire_records_parse_then_verify(backend):
    """f-2 end to end: proofs -> wire records -> parser -> verifier.  A record with a non-canonical scalar is a format
    error (flagged by from_wire, rejected by the verifier on its zeroed bytes); a record with an invalid point encoding
    parses and is rejected by the verifier; a record with a wrong version byte is a format error; the others accept.
    The decisions equal the oracle's (from_bytes + verify)."""
    from bpperm_b200 import acproof as G
    from oracle import wire as W
    core, prover, V, cir, gens, inst = _setup(backend, 5, 91)
    n = core["n"]
    seeds = [bytes([40 + i]) * 32 for i in range(5)]
    B = len(seeds)
    Vc = b"".join(R.compress(p) for p in V)
    proofs = G.prove_batch(backend, cir, gens, _sb(prover["a_L"]) * B, _sb(prover["a_R"]) * B, _sb(prover["a_O"]) * B,
                           _sb(prover["gamma"]) * B, b"".join(seeds), B, "fixed", V=Vc * B)
    plen, wlen = G.proof_len(n, "fixed"), G.wire_len(n, "fixed")
    recs = bytearray(G.to_wire(proofs, n, B, "fixed"))
    assert len(recs) == B * wlen and wlen == plen + 1
    recs[1 * wlen + 1 + 32 * 9:1 * wlen + 1 + 32 * 10] = (L + 5).to_bytes(32, "little")   # proof 1: t_x_blinding >= l
    recs[2 * wlen + 1:2 * wlen + 33] = b"\xff" * 32                                      # proof 2: A_I not a valid encoding
    recs[3 * wlen] = 0x01                                                                 # proof 3: unknown version
    back, status = G.from_wire(bytes(recs), n, B, "fixed")
    assert list(status) == [0, 1, 0, 1, 0]
    acc = list(G.verify_batch(backend, cir, gens, back, Vc * B, B, "fixed"))
    assert acc == [1, 0, 0, 0, 1]
    for i in range(B):
        pb = W.from_bytes(bytes(recs[i * wlen:(i + 1) * wlen]), n, 2)
        want = 0 if pb is None else int(bool(ipa.verify(core, V, pb)))
        assert acc[i] == want, i


def test_generator_fold_operator_matches_the_oracle_and_the_scalar_fold_form(backend):
    """K7 (G'_i = u^-1 G_i + u G_{i+n/2}) against big-int arithmetic, and - the equivalence the prover relies on - an MSM
    over the folded generators against the MSM over the ORIGINAL generators with the folded scalars (a_i u^-1 | a_i u)."""
    n = 16
    rng = ChaChaRng(b"\x5c" * 32)
    pts = [rng.point() for _ in range(n)]
    enc = [R.compress(p) for p in pts]
    us = [rng.scalar() for _ in range(3)] + [1, L - 1]
    uis = [R.sc_inv(u) for u in us]
    table = backend.upload_points(enc)
    out, ms = backend.ipa_fold_generators(table, n, _sb(us), _sb(uis))
    half = n // 2
    assert ms > 0 and len(out) == 32 * len(us) * half
    for f, (u, ui) in enumerate(zip(us, uis)):
        for i in range(half):
            want = R.compress(R.pt_add(R.pt_mul(ui, pts[i]), R.pt_mul(u, pts[i + half])))
            assert out[32 * (f * half + i):32 * (f * half + i + 1)] == want, (f, i)
    a = [rng.scalar() for _ in range(half)]
    folded = [out[32 * i:32 * i + 32] for i in range(half)]                       # fold 0
    lhs = backend.vartime_multiscalar_mul(_sb(a), folded)
    rhs = backend.vartime_multiscalar_mul(_sb([x * uis[0] % L for x in a] + [x * us[0] % L for x in a]), enc)
    assert lhs == rhs
    table.free()


@pytest.mark.parametrize("window_bits", [16, 8, 11])
def test_large_batch_uses_the_warp_per_output_msm_and_stays_byte_identical(backend, window_bits):
    """From 16 outputs per SM the commitments go through the warp-per-output fixed-base kernels (c = 16, 8:
    k_fb_msm_warp_d, digits staged in shared memory, the inner-product rounds' L / R selection compacted while staging;
    c = 11: k_fb_msm_warp<true>, the scalar-staged form).  A 5-card `fixed` batch of 2400 proofs with different prover
    seeds: a sample of proofs must equal the CPU restatement byte for byte, and every proof must verify."""
    from bpperm_b200 import acproof as G
    core, prover, V, cir, gens, inst = _setup(backend, 5, 71, window_bits)
    B = 2400
    seeds = [(7000 + i).to_bytes(4, "little") * 8 for i in range(B)]
    Vc = b"".join(R.compress(p) for p in V)
    batch = G.Batch(backend, cir, gens, B, "fixed", b"test")
    batch.upload_witness(_sb(prover["a_L"]) * B, _sb(prover["a_R"]) * B, _sb(prover["a_O"]) * B, _sb(prover["gamma"]) * B,
                         b"".join(seeds))
    batch.upload_commitments(Vc * B)
    batch.prove()
    proofs = batch.download_proofs()
    plen = G.proof_len(core["n"], "fixed")
    for i in (0, 1, 31, 32, 1199, 2399):
        pb, _ = ipa.prove(core, prover, V, ChaChaRng(seeds[i]))
        assert proofs[i * plen:(i + 1) * plen] == pb, i
    batch.upload_proofs(proofs, Vc * B)
    batch.verify(b"\x05" * 32)
    assert batch.download_accept() == b"\x01" * B
    batch.free()
