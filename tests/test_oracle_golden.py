"""CPU tests: the oracles against the committed golden vectors (generated from the reference's
own code by tests/golden/make_golden.py) and against each other."""
import numpy as np
import pytest

from conftest import load_golden
from helpers import crf_case_inputs, digest, make_golden, srg_case_inputs
from oracle import crf_oracle, loss_oracle, srg_oracle

SRG_NAMES = [c[0] for c in make_golden.SRG_CASES]


@pytest.mark.parametrize("name", SRG_NAMES)
def test_srg_closed_form_matches_reference_golden(name):
    g = load_golden("srg_ref_%s.npz" % name)
    labels, cues, probs = srg_case_inputs(name)
    assert digest(labels, cues, probs) == str(g["inputs_sha256"]), "synthetic generator drifted"
    want = np.unpackbits(g["seeds_bits"])[: int(np.prod(g["seeds_shape"]))].reshape(g["seeds_shape"]).astype(np.float32)
    got = srg_oracle.srg_closed_form(labels, cues, probs, float(g["th1"]), float(g["th2"]))
    assert got.dtype == np.float32 and np.array_equal(got, want)


@pytest.mark.parametrize("name", [n for n in SRG_NAMES if n not in ("i", "j", "h")])
def test_srg_faithful_port_matches_reference_golden(name):
    g = load_golden("srg_ref_%s.npz" % name)
    labels, cues, probs = srg_case_inputs(name)
    want = np.unpackbits(g["seeds_bits"])[: int(np.prod(g["seeds_shape"]))].reshape(g["seeds_shape"]).astype(np.float32)
    got = srg_oracle.srg_faithful(labels, cues, probs, 0.99, 0.85)
    assert np.array_equal(got, want)


def test_srg_reference_in_place_random_sweep():
    """Both restatements against the reference's own generate_seed_step on six random problems (srg_ref_sweep.npz)."""
    g = load_golden("srg_ref_sweep.npz")
    for k, case in enumerate(make_golden.SRG_SWEEP):
        labels, cues, probs = make_golden.srg_sweep_inputs(*case)
        assert digest(labels, cues, probs) == str(g["%d/inputs_sha256" % k]), "synthetic generator drifted"
        shape = g["%d/seeds_shape" % k]
        want = np.unpackbits(g["%d/seeds_bits" % k])[: int(np.prod(shape))].reshape(shape).astype(np.float32)
        assert np.array_equal(srg_oracle.srg_closed_form(labels, cues, probs, 0.99, 0.85), want)
        assert np.array_equal(srg_oracle.srg_faithful(labels, cues, probs, 0.99, 0.85), want)


@pytest.mark.parametrize("case", make_golden.LATTICE_CASES, ids=[c[0] for c in make_golden.LATTICE_CASES])
def test_oracle_lattice_matches_reference_permutohedral_golden(case):
    """oracle/crf_oracle.c lattice vs the golden digests of the reference's own permutohedral.cpp."""
    from dsrg_b200 import synth
    name, H, W, var, sxy, srgb = case
    g = load_golden("lattice_ref.npz")
    im = None if var is None else synth.make_image(np.random.RandomState(77), H, W, var)
    f = make_golden.features(H, W, im, sxy, sxy, srgb)
    L = crf_oracle.OracleLattice(f)
    assert L.M == int(g[name + "/M"])
    assert digest(L.offset, L.bary, L.rank, L.n1, L.n2) == str(g[name + "/sha_struct"])
    x = np.random.RandomState(5).rand(H * W, 21).astype(np.float32)
    assert digest(L.compute(x, "sse")) == str(g[name + "/sha_sse"])
    assert digest(L.compute(np.ones((H * W, 1), np.float32), "seq")) == str(g[name + "/sha_seq"])
    np.testing.assert_allclose(L.bary.sum(1), 1.0, atol=2e-6)  # barycentric weights sum to one


def test_oracle_lattice_bit_exact_vs_ref_so_live():
    """oracle/crf_oracle.c lattice vs the digests of the reference's own permutohedral.cpp (lattice_ref_random.npz)
    on random feature matrices: every structure array and the dispatching compute() bit for bit."""
    g = load_golden("lattice_ref_random.npz")
    for k, (f, x) in enumerate(make_golden.lattice_random_inputs()):
        assert digest(f, x) == str(g["%d/inputs_sha256" % k]), "input generator drifted"
        a = crf_oracle.OracleLattice(f)
        assert a.M == int(g["%d/M" % k])
        for name in make_golden.LATTICE_FIELDS:
            assert digest(getattr(a, name)) == str(g["%d/sha_%s" % (k, name)]), name
        assert digest(a.compute(x, "sse")) == str(g["%d/sha_compute" % k])


@pytest.mark.parametrize("name", [c[0] for c in make_golden.CRF_CASES])
def test_crf_oracle_matches_frozen_golden(name):
    g = load_golden("crf_oracle_%s.npz" % name)
    im, unary, sf = crf_case_inputs(name)
    assert digest(im, unary) == str(g["inputs_sha256"])
    q = crf_oracle.CRF(im, unary, maxiter=10, scale_factor=sf)
    np.testing.assert_allclose(q, g["Q"], atol=1e-6, rtol=0)
    np.testing.assert_allclose(q.sum(-1), 1.0, atol=1e-5)


def test_crf_oracle_map_and_object_api():
    im, unary, sf = crf_case_inputs("train41_smooth")
    H, W, M = unary.shape
    c = crf_oracle.DenseCRF(W, H, M)
    c.set_unary_energy(-unary.ravel())
    c.add_pairwise_energy(10, 80 / sf, 80 / sf, 13, 13, 13, 3, 3 / sf, 3 / sf, im.ravel())
    q = c.inference(5).reshape(H, W, M)
    assert np.array_equal(c.map(5).reshape(H, W), q.argmax(-1))
    assert c.lattice(0).M > 0 and c.norm(1).shape == (H * W,)


def test_loss_oracle_gradient_is_consistent():
    rng = np.random.RandomState(0)
    p = rng.rand(2, 5, 6, 7) * 0.9 + 0.05
    lab = (rng.rand(2, 5, 6, 7) < 0.2).astype(np.float64)
    lab[1, 1:] = 0  # an image without foreground seeds: max(count, 1e-4) branch
    g = loss_oracle.balanced_seed_loss_grad(p, lab)
    eps = 1e-6
    for idx in [(0, 0, 1, 2), (0, 3, 2, 2), (1, 0, 5, 6)]:
        pp, pm = p.copy(), p.copy()
        pp[idx] += eps
        pm[idx] -= eps
        num = (loss_oracle.balanced_seed_loss(pp, lab) - loss_oracle.balanced_seed_loss(pm, lab)) / (2 * eps)
        assert abs(num - g[idx]) < 1e-5


def test_zoom_restatement_is_bit_exact_vs_scipy():
    """The bilinear-zoom restatement the CUDA preprocessing kernel mirrors, against scipy itself."""
    from scipy.ndimage import zoom
    rng = np.random.RandomState(4)
    for (ih, iw, oh, ow) in ((321, 321, 41, 41), (97, 131, 33, 57), (50, 40, 50, 40), (17, 9, 40, 31), (8, 8, 1, 1),
                             (5, 7, 1, 4), (33, 33, 321, 321), (31, 31, 97, 131), (51, 51, 60, 45)):
        im = (rng.rand(2, 3, ih, iw) * 255 - 110).astype(np.float32)
        want = zoom(im, (1.0, 1.0, float(oh) / ih, float(ow) / iw), order=1)
        got = crf_oracle.zoom_order1_restated(im, oh, ow)
        assert want.shape == got.shape and want.dtype == got.dtype and np.array_equal(want, got)


def test_zoom_restatement_covers_score_maps():
    """(h,w,M) score maps zoomed with a trailing identity axis (test-ms.py:96): same taps, same bits."""
    from scipy.ndimage import zoom
    rng = np.random.RandomState(5)
    for (h, w, H, W) in ((41, 41, 375, 500), (31, 31, 97, 131), (51, 51, 60, 45), (41, 41, 20, 30), (7, 9, 1, 5),
                         (33, 33, 321, 321)):
        blob = (rng.randn(21, h, w) * 5).astype(np.float32)
        want = zoom(np.transpose(blob, [1, 2, 0]), (float(H) / h, float(W) / w, 1.0), order=1)
        got = crf_oracle.zoom_order1_restated(blob[None], H, W)[0].transpose(1, 2, 0)
        assert want.shape == (H, W, 21) and np.array_equal(want, got)


@pytest.mark.parametrize("case", make_golden.POST_CASES, ids=[c[0] for c in make_golden.POST_CASES])
def test_post_oracle_matches_frozen_golden(case):
    from oracle import post_oracle
    name, mode, H, W, sizes, index = case
    g = load_golden("post_oracle_%s.npz" % name)
    im, blobs, tags = make_golden.post_inputs(H, W, sizes, index)
    assert digest(im, *blobs) == str(g["inputs_sha256"])
    if mode == "ms":
        lab, probs = post_oracle.predict_mask_ms(im, blobs, smooth=True)
        sel = list(range(21))
    else:
        lab, probs = post_oracle.predict_mask_gt(im, blobs[0], tags, smooth=True)
        sel = [0] + list(tags)
        assert set(np.unique(lab)) <= set(sel)
    np.testing.assert_allclose(probs, g["probs"], atol=1e-6, rtol=0)
    bad = lab != g["labels"]
    if bad.any():   # another libm may flip an exact near-tie
        top2 = np.sort(g["probs"][:, :, sel], axis=2)[:, :, -2:]
        assert ((top2[:, :, 1] - top2[:, :, 0])[bad] < 1e-5).all()
    # smooth=False is plain numpy: arg-max of the clamped soft-max
    lab0, p0 = post_oracle.predict_mask_ms(im, blobs, smooth=False)
    assert np.array_equal(lab0, p0.argmax(2)) and p0.min() >= np.float32(1e-5)


@pytest.mark.parametrize("name", [c[0] for c in make_golden.CRF_CASES])
def test_crf_oracle_is_bit_exact_vs_the_reference_build(name):
    """The C restatement against the reference's OWN CRF sources (densecrf.cpp, pairwise.cpp, ... compiled
    unmodified, oracle/Makefile) through DenseCRFWrapper: marginals and MAP labels, several iteration counts,
    compared with the digests of that build's outputs (crf_ref_build.npz)."""
    g = load_golden("crf_ref_build.npz")
    im, unary, sf = crf_case_inputs(name)
    assert digest(im, unary) == str(g[name + "/inputs_sha256"])
    assert digest(crf_oracle.CRF(im, unary, 10, sf)) == str(g[name + "/crf"])
    o = make_golden.crf_objects(crf_oracle.DenseCRF, im, unary, sf)
    for it in make_golden.CRF_REF_ITERS:
        assert digest(o.inference(it)) == str(g["%s/inference%d" % (name, it)]), it
        assert digest(o.map(it)) == str(g["%s/map%d" % (name, it)]), it


@pytest.mark.parametrize("H,W,M,sf,img", make_golden.CRF_REF_SHAPES)
def test_crf_oracle_vs_reference_build_other_shapes(H, W, M, sf, img):
    """incl. M = 2, where Permutohedral::compute takes the seqCompute branch (permutohedral.cpp:600-601)."""
    g = load_golden("crf_ref_build.npz")
    key = make_golden.crf_shape_key(H, W, M, sf, img)
    im, unaries = make_golden.crf_shape_inputs(H, W, M, img)
    assert digest(im, *unaries) == str(g[key + "/inputs_sha256"])
    for kind, unary in zip(("logp", "p"), unaries):
        assert digest(crf_oracle.CRF(im, unary, 10, sf, color_factor=13)) == str(g["%s/%s" % (key, kind)]), kind


# ---- a12 / f1 / f4: the loss and annotation oracles against the reference's own layer classes -------------------
# tests/golden/layers_ref.npz holds the outputs of the reference's SoftmaxLayer / BalancedSeedLossLayer /
# ConstrainLossLayer / AnnotationLayer class bodies executed in place (oracle/ref_layers.py; Theano is replaced by
# oracle/theano_shim.py, float64 and float32 evaluation).
@pytest.mark.parametrize("seed", [0, 1])
def test_loss_oracles_match_the_reference_layers_golden(seed):
    g = load_golden("layers_ref.npz")
    logits, p, lab, td, ls = make_golden.layer_inputs(seed)
    assert digest(logits, p, lab, td, ls) == str(g["in%d_sha256" % seed]), "input generator drifted"
    k = "s%d_float64_" % seed
    tight = dict(rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(loss_oracle.softmax_layer_forward(logits), g[k + "softmax_probs"], **tight)
    np.testing.assert_allclose(loss_oracle.softmax_layer_backward(logits, td), g[k + "softmax_grad"], **tight)
    np.testing.assert_allclose(loss_oracle.balanced_seed_loss(p, lab), g[k + "seed_loss"], **tight)
    np.testing.assert_allclose(loss_oracle.balanced_seed_loss_grad(p, lab), g[k + "seed_grad"], **tight)
    np.testing.assert_allclose(loss_oracle.constrain_loss(p, ls), g[k + "constrain_loss"], **tight)
    w0, w1 = loss_oracle.constrain_loss_grad(p, ls)
    np.testing.assert_allclose(w0, g[k + "constrain_g0"], **tight)
    np.testing.assert_allclose(w1, g[k + "constrain_g1"], **tight)
    # the float32 evaluation (what T.ftensor4 computes in) stays within the tolerance the GPU tests use
    k32 = "s%d_float32_" % seed
    for name in ("softmax_probs", "softmax_grad", "seed_loss", "seed_grad", "constrain_loss", "constrain_g0", "constrain_g1"):
        np.testing.assert_allclose(g[k32 + name], g[k + name], rtol=2e-5, atol=1e-7)


@pytest.mark.parametrize("mirror", [False, True])
def test_annotation_oracle_matches_the_reference_layer_golden(mirror):
    from oracle import annot_oracle
    g = load_golden("layers_ref.npz")
    d, ids, images = make_golden.annot_inputs()
    np.random.seed(11)
    t0, t1, t2 = annot_oracle.annotation_forward(d, ids, images, mirror)
    k = "annot_m%d_" % int(mirror)
    shape = tuple(g[k + "cues_shape"])
    want1 = np.unpackbits(g[k + "cues_bits"])[: int(np.prod(shape))].reshape(shape).astype(np.float32)
    assert np.array_equal(t0, g[k + "labels"]) and np.array_equal(t1, want1) and digest(t2) == str(g[k + "images_sha256"])


def test_reference_layers_run_in_place_random_sweep():
    """The reference's own layer classes (through the Theano stand-in) against the restatements on three more shapes:
    losses in full, a fixed sample of every gradient (layers_ref_sweep.npz)."""
    g = load_golden("layers_ref_sweep.npz")
    for seed in make_golden.LAYER_SWEEP_SEEDS:
        logits, p, lab, td, ls = make_golden.layer_sweep_inputs(seed)
        k = "s%d_" % seed
        assert digest(logits, p, lab, td, ls) == str(g[k + "inputs_sha256"]), "input generator drifted"

        def sample(a):
            return make_golden.layer_sample(a, seed)
        np.testing.assert_allclose(g[k + "seed_loss"], loss_oracle.balanced_seed_loss(p, lab), rtol=1e-12)
        np.testing.assert_allclose(g[k + "seed_grad"], sample(loss_oracle.balanced_seed_loss_grad(p, lab)),
                                   rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(g[k + "softmax_probs"], sample(loss_oracle.softmax_layer_forward(logits)), rtol=1e-12)
        np.testing.assert_allclose(g[k + "softmax_grad"], sample(loss_oracle.softmax_layer_backward(logits, td)),
                                   rtol=1e-10, atol=1e-15)
        np.testing.assert_allclose(g[k + "constrain_loss"], loss_oracle.constrain_loss(p, ls), rtol=1e-12)
        w0, w1 = loss_oracle.constrain_loss_grad(p, ls)
        np.testing.assert_allclose(g[k + "constrain_g0"], sample(w0), rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(g[k + "constrain_g1"], sample(w1), rtol=1e-12, atol=1e-15)
