"""tests/golden/make_golden.py -- regenerates the committed golden fixtures.

Runs ONLY in the dev container (needs /root/reference):
  * SRG: the reference's own generate_seed_step + CC_labeling_8, executed in place
    (oracle/srg_oracle.py:reference_generate_seed_step) on seeded synthetic problems
    -> tests/golden/srg_ref_*.npz (outputs stored as packed bits; inputs are regenerated
       from the seed by dsrg_b200/synth.py, a checksum of the inputs guards against drift)
  * lattice: the reference's own CRF/src/permutohedral.cpp (oracle/_ref) on real feature
    matrices -> tests/golden/lattice_ref.npz (vertex counts, exact sums / checksums of
    offsets, barycentrics, ranks, neighbours and of seq/sse compute outputs)
  * layers: the reference's own SoftmaxLayer / BalancedSeedLossLayer / ConstrainLossLayer / AnnotationLayer
    class bodies executed in place (oracle/ref_layers.py, Theano stand-in oracle/theano_shim.py), float64
    and float32 -> tests/golden/layers_ref.npz (pins oracle/loss_oracle.py and oracle/annot_oracle.py)
  * CRF: oracle/crf_oracle.c marginals (restatement; its lattice is pinned by the previous
    item) -> tests/golden/crf_oracle_*.npz, so GPU runs have a frozen target even if the
    oracle sources change later.
  * the reference's own code on further seeded inputs, so that the tests compare the restatements
    with it without the reference at hand:
      srg_sweep      generate_seed_step on six random problems -> srg_ref_sweep.npz (packed bits)
      lattice_random permutohedral.cpp on three random feature matrices -> lattice_ref_random.npz
      crf_ref        the compiled CRF sources (oracle/_ref/libdensecrf_ref.so) -> crf_ref_build.npz:
                     sha256 of the marginals / MAP labels, bit-exact targets of the restatement
      layers_sweep   the loss layer classes on three more shapes -> layers_ref_sweep.npz (float64,
                     a fixed sample of each gradient)

usage: python tests/golden/make_golden.py [srg lattice crf post layers srg_sweep lattice_random crf_ref layers_sweep]
       (default: all)
"""
import hashlib
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from dsrg_b200 import synth  # noqa: E402
from oracle import crf_oracle, post_oracle, srg_oracle  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

SRG_CASES = [  # name, H, W, cues variant, image index, tweak
    ("a", 41, 41, "cam", 0, None),
    ("b", 41, 41, "random", 1, None),
    ("c", 33, 57, "random", 2, "ties"),
    ("d", 64, 48, "cam", 3, "ties"),
    ("e", 1, 1, "random", 4, None),
    ("f", 1, 37, "random", 5, None),
    ("g", 29, 1, "cam", 6, None),
    ("h", 96, 96, "random", 7, None),
    ("i", 321, 321, "cam", 8, None),
    ("j", 161, 161, "random", 9, "ties"),
]


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def srg_inputs(H, W, cues, index, tweak):
    p = synth.make_problem(index, H, W, cues=cues, image="noise")
    probs = p["probs"].copy()
    if tweak == "ties":  # values exactly at the thresholds, and exact ties between classes
        probs[:, ::3, ::2] = np.float32(0.85)
        probs[0, 1::4, :] = np.float32(0.99)
        probs[:, 2::5, 1::3] = np.float32(1.0 / 21)
    return p["labels"], p["cues"], probs


def make_srg():
    for name, H, W, cues, index, tweak in SRG_CASES:
        labels, cu, probs = srg_inputs(H, W, cues, index, tweak)
        t = time.time()
        out = srg_oracle.run_reference(labels, cu, probs, 0.99, 0.85)
        dt = time.time() - t
        assert set(np.unique(out)) <= {0.0, 1.0}
        np.savez_compressed(os.path.join(OUT, "srg_ref_%s.npz" % name), H=H, W=W, cues=cues, index=index,
                            tweak=str(tweak), th1=0.99, th2=0.85, inputs_sha256=digest(labels, cu, probs),
                            seeds_bits=np.packbits(out.astype(np.uint8)), seeds_shape=np.array(out.shape),
                            ref_seconds=dt)
        print("srg", name, H, W, "ref %.2fs" % dt, int(cu.sum()), "->", int(out.sum()))


def features(H, W, image, sx, sy, sr):
    ys, xs = np.mgrid[0:H, 0:W]
    d = 2 if image is None else 5
    f = np.empty((H * W, d), np.float32)
    f[:, 0] = xs.ravel().astype(np.float32) / np.float32(sx)
    f[:, 1] = ys.ravel().astype(np.float32) / np.float32(sy)
    if image is not None:
        for c in range(3):
            f[:, 2 + c] = image.reshape(-1, 3)[:, c].astype(np.float32) / np.float32(sr)
    return f


LATTICE_CASES = [  # name, H, W, image variant or None, sigma_xy, sigma_rgb
    ("sp3_41", 41, 41, None, 3.0, 0),
    ("sp025_41", 41, 41, None, 0.25, 0),
    ("sp3_321", 321, 321, None, 3.0, 0),
    ("bi_smooth_41_s12", 41, 41, "smooth", 80 / 12.0, 13),
    ("bi_noise_57x33", 33, 57, "noise", 80.0, 13),
    ("bi_smooth_321", 321, 321, "smooth", 80.0, 13),
    ("bi_noise_161", 161, 161, "noise", 80.0, 13),
]


def make_lattice():
    rec = {}
    for name, H, W, var, sxy, srgb in LATTICE_CASES:
        im = None if var is None else synth.make_image(np.random.RandomState(77), H, W, var)
        f = features(H, W, im, sxy, sxy, srgb)
        L = crf_oracle.RefLattice(f)
        x = np.random.RandomState(5).rand(H * W, 21).astype(np.float32)
        sse = L.compute(x, "sse")
        seq = L.compute(np.ones((H * W, 1), np.float32), "seq")
        rec[name + "/M"] = L.M
        rec[name + "/sha_struct"] = digest(L.offset, L.bary, L.rank, L.n1, L.n2)
        rec[name + "/sha_sse"] = digest(sse)
        rec[name + "/sha_seq"] = digest(seq)
        rec[name + "/seq_sum"] = float(seq.astype(np.float64).sum())
        print("lattice", name, "M", L.M)
    np.savez_compressed(os.path.join(OUT, "lattice_ref.npz"), **rec)


CRF_CASES = [  # name, H, W, image variant, scale_factor, unary kind
    ("train41_smooth", 41, 41, "smooth", 12.0, "p"),
    ("train41_noise", 41, 41, "noise", 12.0, "p"),
    ("test_57x33_smooth", 33, 57, "smooth", 1.0, "logp"),
    ("test_64_noise", 64, 64, "noise", 1.0, "logp"),
]


def crf_inputs(H, W, var, kind, index):
    p = synth.make_problem(100 + index, H, W, image=var)
    pr = np.transpose(p["probs"], (1, 2, 0)).copy()
    pr[pr < 1e-5] = 1e-5
    unary = pr if kind == "p" else np.log(pr)
    return p["image"], unary.astype(np.float32)


def make_crf():
    for i, (name, H, W, var, sf, kind) in enumerate(CRF_CASES):
        im, unary = crf_inputs(H, W, var, kind, i)
        q = crf_oracle.CRF(im, unary, maxiter=10, scale_factor=sf)
        np.savez_compressed(os.path.join(OUT, "crf_oracle_%s.npz" % name), H=H, W=W, image_variant=var,
                            scale_factor=sf, unary_kind=kind, index=i, inputs_sha256=digest(im, unary), Q=q)
        print("crf", name, q.shape, float(q.max()))


POST_CASES = [  # name, mode, H, W, network sizes, index
    ("ms_48x64", "ms", 48, 64, (17, 21, 25), 20),
    ("gt_40x56", "gt", 40, 56, (21,), 21),
]


def post_inputs(H, W, sizes, index):
    s = synth.make_score_blobs(index, H, W, sizes)
    return s["image"], s["blobs"], s["tags"]


def make_post():
    for name, mode, H, W, sizes, index in POST_CASES:
        im, blobs, tags = post_inputs(H, W, sizes, index)
        if mode == "ms":
            lab, probs = post_oracle.predict_mask_ms(im, blobs, smooth=True)
        else:
            lab, probs = post_oracle.predict_mask_gt(im, blobs[0], tags, smooth=True)
        np.savez_compressed(os.path.join(OUT, "post_oracle_%s.npz" % name), inputs_sha256=digest(im, *blobs),
                            tags=tags, labels=lab.astype(np.uint8), probs=probs.astype(np.float32))
        print("post", name, lab.shape, np.unique(lab))


def layer_inputs(seed=0, N=3, C=21, H=9, W=7):
    """Small seeded inputs of the loss layers: probs with values at the 1e-4 clamp, seed masks with an image
    without foreground and one without background seeds, smoothed log-probs on both sides of the clip range."""
    rng = np.random.RandomState(4242 + seed)
    logits = (3 * rng.randn(N, C, H, W)).astype(np.float32)
    p = np.exp(logits - logits.max(1, keepdims=True))
    p = np.maximum(p / p.sum(1, keepdims=True), 1e-4).astype(np.float32)
    lab = (rng.rand(N, C, H, W) < 0.1).astype(np.float32)
    lab[N - 2, 1:] = 0
    lab[N - 1, 0] = 0
    top_diff = rng.randn(N, C, H, W).astype(np.float32)
    log_smooth = np.log(np.maximum(p * rng.uniform(0.01, 30, p.shape), 1e-6)).astype(np.float32)
    return logits, p, lab, top_diff, log_smooth


def annot_inputs(n_images=6, seed=3, h=41, w=41, M=21):
    rng = np.random.RandomState(seed)
    d = {}
    for i in range(n_images):
        k = rng.randint(1, 4)
        tags = np.sort(rng.choice(np.arange(1, M), size=k, replace=False))
        d['%i_labels' % i] = tags
        cls = np.concatenate([[0], tags])
        K = 0 if i == 3 else rng.randint(1, 300)
        d['%i_cues' % i] = np.stack([rng.choice(cls, K), rng.randint(0, h, K), rng.randint(0, w, K)]).astype(np.int64)
    ids = np.array([5, 0, 3, 1, 2, 2], np.float32)
    images = (rng.rand(len(ids), 3, 17, 23) * 255 - 110).astype(np.float32)
    return d, ids, images


def make_layers():
    from oracle import ref_layers
    rec = {}
    for seed in (0, 1):
        logits, p, lab, td, ls = layer_inputs(seed)
        rec["in%d_sha256" % seed] = digest(logits, p, lab, td, ls)
        for dt in ("float64", "float32"):
            k = "s%d_%s_" % (seed, dt)
            rec[k + "softmax_probs"], rec[k + "softmax_grad"] = ref_layers.softmax_layer(logits, td, dt)
            rec[k + "seed_loss"], rec[k + "seed_grad"] = ref_layers.balanced_seed_loss_layer(p, lab, dt)
            rec[k + "constrain_loss"], rec[k + "constrain_g0"], rec[k + "constrain_g1"] = \
                ref_layers.constrain_loss_layer(p, ls, dt)
        print("layers seed", seed, float(rec["s%d_float64_seed_loss" % seed]), float(rec["s%d_float64_constrain_loss" % seed]))
    d, ids, images = annot_inputs()
    for mirror in (False, True):
        t0, t1, t2 = ref_layers.annotation_layer_forward(d, ids, images, mirror, seed=11)
        k = "annot_m%d_" % int(mirror)
        rec[k + "labels"], rec[k + "cues_bits"], rec[k + "images_sha256"] = t0, np.packbits(t1.astype(np.uint8)), digest(t2)
        rec[k + "cues_shape"] = np.array(t1.shape)
        print("annotation mirror", mirror, int(t1.sum()))
    np.savez_compressed(os.path.join(OUT, "layers_ref.npz"), **rec)


SRG_SWEEP = [(500 + i, 19 + 3 * i, 31 - 2 * i, ["cam", "random"][i % 2]) for i in range(6)]  # index, H, W, cues


def srg_sweep_inputs(index, H, W, cues):
    p = synth.make_problem(index, H, W, cues=cues, image="noise")
    return p["labels"], p["cues"], p["probs"]


def make_srg_sweep():
    rec = {}
    for k, case in enumerate(SRG_SWEEP):
        labels, cu, probs = srg_sweep_inputs(*case)
        out = srg_oracle.run_reference(labels, cu, probs, 0.99, 0.85)
        rec["%d/inputs_sha256" % k] = digest(labels, cu, probs)
        rec["%d/seeds_bits" % k], rec["%d/seeds_shape" % k] = np.packbits(out.astype(np.uint8)), np.array(out.shape)
        print("srg sweep", case, int(cu.sum()), "->", int(out.sum()))
    np.savez_compressed(os.path.join(OUT, "srg_ref_sweep.npz"), **rec)


LATTICE_FIELDS = ("offset", "bary", "rank", "n1", "n2")


def lattice_random_inputs():
    """(features, values) pairs: random 2-d (spatial) and 5-d (bilateral) feature matrices, 21 values per point."""
    rng = np.random.RandomState(3)
    cases = []
    for H, W, d in ((23, 31, 2), (23, 31, 5), (40, 17, 5)):
        f = (rng.rand(H * W, d) * [3, 3, 19, 19, 19][:d]).astype(np.float32)
        cases.append((f, rng.rand(H * W, 21).astype(np.float32)))
    return cases


def make_lattice_random():
    rec = {}
    for k, (f, x) in enumerate(lattice_random_inputs()):
        L = crf_oracle.RefLattice(f)
        rec["%d/inputs_sha256" % k] = digest(f, x)
        rec["%d/M" % k] = L.M
        for name in LATTICE_FIELDS:
            rec["%d/sha_%s" % (k, name)] = digest(getattr(L, name))
        rec["%d/sha_compute" % k] = digest(L.compute(x, "dispatch"))
        print("lattice random", k, f.shape, "M", L.M)
    np.savez_compressed(os.path.join(OUT, "lattice_ref_random.npz"), **rec)


CRF_REF_ITERS = (0, 1, 4)
CRF_REF_SHAPES = [(97, 131, 21, 1.0, "smooth"), (60, 45, 5, 12.0, "noise"), (33, 33, 2, 1.0, "noise"),  # H, W, M, sf, image
                  (161, 161, 21, 1.0, "smooth"), (120, 90, 21, 1.0, "photo")]
CRF_DIRECT_CASES = [(41, 41, 12.0, "smooth"), (97, 131, 1.0, "smooth"), (64, 64, 1.0, "noise")]  # H, W, sf, image


def crf_shape_key(H, W, M, sf, img):
    return "shape_%d_%d_%d_%g_%s" % (H, W, M, sf, img)


def crf_shape_inputs(H, W, M, img):
    """(image, [log-probability unary, probability unary])."""
    rng = np.random.RandomState(H * 7 + M)
    im = synth.make_image(rng, H, W, img)
    logits = rng.randn(H, W, M) * 2
    logits[H // 4: H // 2, W // 3:, 0] += 4
    e = np.exp(logits - logits.max(2, keepdims=True))
    pr = (e / e.sum(2, keepdims=True)).astype(np.float32)
    pr[pr < 1e-5] = 1e-5
    return im, [np.log(pr), pr]


def crf_direct_key(H, W):
    return "direct_%dx%d" % (H, W)


def crf_direct_inputs(H, W, sf, img):
    """(image, unary) of the GPU test against the reference build: probabilities at scale_factor 12, else log p."""
    p = synth.make_problem(950 + H, H, W, image=img)
    pr = np.transpose(p["probs"], (1, 2, 0)).copy()
    pr[pr < 1e-5] = 1e-5
    return p["image"], pr if sf > 1 else np.log(pr)


def crf_objects(cls, im, unary, sf):
    """A DenseCRF-like object of class ``cls`` set up the way CRF.py:21-33 does."""
    H, W, M = unary.shape
    c = cls(W, H, M)
    c.set_unary_energy(-unary.ravel())
    c.add_pairwise_energy(10, 80 / sf, 80 / sf, 13, 13, 13, 3, 3 / sf, 3 / sf, im.ravel())
    return c


def make_crf_ref():
    rec = {}
    for i, (name, H, W, var, sf, kind) in enumerate(CRF_CASES):
        im, unary = crf_inputs(H, W, var, kind, i)
        rec[name + "/inputs_sha256"] = digest(im, unary)
        rec[name + "/crf"] = digest(crf_oracle.CRF_reference(im, unary, 10, sf))
        r = crf_objects(crf_oracle.RefDenseCRF, im, unary, sf)
        for it in CRF_REF_ITERS:
            rec["%s/inference%d" % (name, it)] = digest(r.inference(it))
            rec["%s/map%d" % (name, it)] = digest(r.map(it))
    for H, W, M, sf, img in CRF_REF_SHAPES:
        im, unaries = crf_shape_inputs(H, W, M, img)
        key = crf_shape_key(H, W, M, sf, img)
        rec[key + "/inputs_sha256"] = digest(im, *unaries)
        for kind, unary in zip(("logp", "p"), unaries):
            rec["%s/%s" % (key, kind)] = digest(crf_oracle.CRF_reference(im, unary, 10, sf, color_factor=13))
    for H, W, sf, img in CRF_DIRECT_CASES:
        im, unary = crf_direct_inputs(H, W, sf, img)
        key = crf_direct_key(H, W)
        rec[key + "/inputs_sha256"] = digest(im, unary)
        rec[key + "/crf"] = digest(crf_oracle.CRF_reference(im, unary, 10, sf))
        rec[key + "/map"] = digest(crf_objects(crf_oracle.RefDenseCRF, im, unary, sf).map(10))
    print("crf ref", len(rec), "digests")
    np.savez_compressed(os.path.join(OUT, "crf_ref_build.npz"), **rec)


LAYER_SWEEP_SEEDS = (5, 6, 7)
LAYER_SAMPLE = 512   # elements kept of each gradient array (float64; the whole array would exceed what a fixture needs)


def layer_sweep_inputs(seed):
    return layer_inputs(seed, N=2 + seed % 3, H=5 + seed, W=11 - seed)


def layer_sample(a, seed):
    """A fixed, seeded sample of the flattened array ``a`` (all of it when it is small)."""
    a = np.ravel(a)
    if a.size <= LAYER_SAMPLE:
        return a
    return a[np.sort(np.random.RandomState(seed).choice(a.size, LAYER_SAMPLE, replace=False))]


def make_layers_sweep():
    from oracle import ref_layers
    rec = {}
    for seed in LAYER_SWEEP_SEEDS:
        logits, p, lab, td, ls = layer_sweep_inputs(seed)
        k = "s%d_" % seed
        rec[k + "inputs_sha256"] = digest(logits, p, lab, td, ls)
        loss, grad = ref_layers.balanced_seed_loss_layer(p, lab, "float64")
        pr, gd = ref_layers.softmax_layer(logits, td, "float64")
        cl, g0, g1 = ref_layers.constrain_loss_layer(p, ls, "float64")
        rec[k + "seed_loss"], rec[k + "constrain_loss"] = loss, cl
        for name, a in (("seed_grad", grad), ("softmax_probs", pr), ("softmax_grad", gd), ("constrain_g0", g0),
                        ("constrain_g1", g1)):
            rec[k + name] = layer_sample(a, seed)
        print("layers sweep seed", seed, float(loss), float(cl))
    np.savez_compressed(os.path.join(OUT, "layers_ref_sweep.npz"), **rec)


if __name__ == "__main__":
    assert srg_oracle.reference_available(), "needs the reference checkout (oracle/srg_oracle.py:REF_ROOT)"
    what = sys.argv[1:] or ["srg", "lattice", "crf", "post", "layers", "srg_sweep", "lattice_random", "crf_ref",
                            "layers_sweep"]
    crf_oracle.build(force=True)
    for w in what:
        {"srg": make_srg, "lattice": make_lattice, "crf": make_crf, "post": make_post, "layers": make_layers,
         "srg_sweep": make_srg_sweep, "lattice_random": make_lattice_random, "crf_ref": make_crf_ref,
         "layers_sweep": make_layers_sweep}[w]()
