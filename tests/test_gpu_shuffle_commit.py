"""The shuffle prover's A_I from a device-generated witness: a_R = v' - x lets the library commit <a_R, H> as
<v', H> + (-x) H_sum with the small card values spread over all lanes (bpp_acp_batch_prove, k_fb_msm_warp_d<C, true>).
Proofs and commitments must be byte-identical to those of the same a_L, a_R, a_O uploaded with
bpp_acp_batch_upload_witness (the generic A_I), A_I must equal the oracle's MSM, and the verifier must accept.  Batches of
at least 16 x 148 proofs reach the warp form, which is the only form that takes the structured A_I; smaller ones check that
every other form keeps the generic one."""
import numpy as np
import pytest

from oracle import cref, ristretto255 as R
from oracle.chacha import ChaChaRng

pytestmark = pytest.mark.gpu
L = R.L
WARP_B = 2400   # >= 16 outputs per SM on a 148-SM B200: the warp-per-output form


def _sb(v):
    return b"".join(R.sc_bytes(s) for s in v)


def _witness(k, deck, perm, x):
    """oracle.acproof.shuffle_witness for this deck, permutation and challenge value."""
    n = 2 * k
    v = deck + [deck[j] for j in perm] + [x]
    aL, aR, aO = [0] * n, [0] * n, [0] * n
    for gb, vb in ((0, 0), (k - 1, k)):
        for i in range(k - 1):
            aL[gb + i] = (v[vb] - x) % L if i == 0 else aO[gb + i - 1]
            aR[gb + i] = (v[vb + i + 1] - x) % L
            aO[gb + i] = aL[gb + i] * aR[gb + i] % L
    return v, aL, aR, aO


_GENS = {}


def _gens(backend, ng, c):
    """ng G and ng H generators (plus g, h) with tables of width c, shared across the tests of this module."""
    from bpperm_b200 import acproof as G
    key = (ng, c)
    if key not in _GENS:
        rs = np.random.RandomState(4100 + ng)
        raw = cref.from_uniform(rs.randint(0, 256, size=(2 * ng + 2, 64), dtype=np.uint8).tobytes())
        enc = cref.compress(raw)
        pts = [enc[32 * i:32 * i + 32] for i in range(2 * ng + 2)]
        _GENS[key] = (G.Generators(backend, pts[0], pts[1], pts[2:2 + ng], pts[2 + ng:], c), raw)
    return _GENS[key]


@pytest.fixture(scope="module", autouse=True)
def _free_gens():
    yield
    for g, _ in _GENS.values():
        g.free()
    _GENS.clear()


def _decks(k, kind, rs):
    if kind == "1..k":
        return list(range(1, k + 1))
    if kind == "random":
        return [int.from_bytes(rs.bytes(32), "little") % L for _ in range(k)]
    edge = [0, 2 ** 15 - 1, 2 ** 15, 2 ** 15 + 1, L - 1]     # one, two and many non-zero 16-bit / 8-bit digits
    return [edge[i] if i < len(edge) else i + 1 for i in range(k)]


def _run(backend, k, B, c, mode, deck_kind, seed, upload_after=False):
    from bpperm_b200 import acproof as G
    n, m = 2 * k, 2 * k + 1
    ng = G.next_pow2(n) if mode == "fixed" else n
    gens, raw = _gens(backend, ng, c)
    rs = np.random.RandomState(seed)
    deck = _decks(k, deck_kind, rs)
    xs = [int.from_bytes(rs.bytes(32), "little") % L for _ in range(B)]
    xs[0] = 0
    if B > 1:
        xs[1] = L - 1
    if B > 2:
        xs[2] = 1
    perms = [rs.permutation(k) for _ in range(B)]
    wit = [_witness(k, deck, perms[p], xs[p]) for p in range(B)]
    gam_b = rs.randint(0, 256, size=(B, m, 32), dtype=np.uint8)
    gam_b[:, :, 31] &= 0x0F
    gam_b = gam_b.tobytes()
    seeds = rs.randint(0, 256, size=(B, 32), dtype=np.uint8).tobytes()
    perm_b = np.stack(perms).astype(np.uint32).tobytes()
    cir = G.Circuit.shuffle(backend, k)
    aL = b"".join(_sb(w[1]) for w in wit)
    aR = b"".join(_sb(w[2]) for w in wit)
    aO = b"".join(_sb(w[3]) for w in wit)
    # uploaded witness: the generic A_I
    b1 = G.Batch(backend, cir, gens, B, mode)
    b1.upload_witness(aL, aR, aO, gam_b, seeds)
    V1 = b1.commit(b"".join(_sb(w[0]) for w in wit))
    b1.prove()
    p1 = b1.download_proofs()
    # generated witness: the structured A_I where the batch runs the warp form
    b2 = G.Batch(backend, cir, gens, B, mode)
    if upload_after:   # a generated witness, then an uploaded one: the uploaded one's generic A_I
        other = list(range(k + 1, 1, -1))
        b2.gen_shuffle_witness(_sb(other), perm_b, _sb(xs), gam_b, seeds)
        b2.upload_witness(aL, aR, aO, gam_b, seeds)
        V2 = b2.commit(b"".join(_sb(w[0]) for w in wit))
    else:
        b2.gen_shuffle_witness(_sb(deck), perm_b, _sb(xs), gam_b, seeds)
        V2 = b2.commit(None)
    b2.prove()
    p2 = b2.download_proofs()
    assert V1 == V2
    assert p1 == p2
    # A_I of a few proofs against the oracle: alpha h + <a_L, G> + <a_R, H>
    PT = len(raw) // (2 * ng + 2)
    pts = raw[PT:2 * PT] + raw[2 * PT:(2 + n) * PT] + raw[(2 + ng) * PT:(2 + ng + n) * PT]
    plen = b2.proof_len
    for p in range(min(B, 3)):
        alpha = ChaChaRng(seeds[32 * p:32 * p + 32]).scalar()
        want = cref.msm(_sb([alpha] + wit[p][1] + wit[p][2]), pts)
        assert p2[p * plen:p * plen + 32] == want, p
    b2.upload_proofs(p2, V2)
    b2.verify(b"\x05" * 32)
    assert b2.download_accept() == b"\x01" * B
    for o in (b1, b2, cir):
        o.free()


@pytest.mark.parametrize("deck_kind", ["1..k", "random", "edge"])
@pytest.mark.parametrize("c", [16, 8])
def test_warp_form_52_cards(backend, c, deck_kind):
    _run(backend, 52, WARP_B, c, "reference-fixed", deck_kind, 10 + c)


@pytest.mark.parametrize("c", [16, 8])
def test_warp_form_fixed_mode(backend, c):
    _run(backend, 52, WARP_B, c, "fixed", "1..k", 20 + c)


@pytest.mark.parametrize("k", [2, 3])
def test_warp_form_small_decks(backend, k):
    _run(backend, k, WARP_B, 8, "reference-fixed", "edge" if k == 3 else "1..k", 30 + k)


@pytest.mark.parametrize("B", [1, 64])
@pytest.mark.parametrize("c", [16, 8])
def test_thread_and_block_forms(backend, B, c):
    _run(backend, 52, B, c, "reference-fixed", "edge", 40 + B)


@pytest.mark.parametrize("mode", ["reference-fixed", "fixed"])
def test_long_chain(backend, mode):
    """k = 300 with 3 proofs: the block-scan witness kernel (k_shuffle_witness)."""
    _run(backend, 300, 3, 8, mode, "1..k", 50)


def test_upload_after_generated_witness_takes_the_generic_shape(backend):
    _run(backend, 52, WARP_B, 16, "reference-fixed", "1..k", 60, upload_after=True)
