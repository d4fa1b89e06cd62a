"""GPU parity: dense-CRF mean field through the C ABI vs the CPU oracle (tolerance 1e-4 max-abs on
the marginals, BASELINE.json north_star) and vs the frozen golden vectors."""
import numpy as np
import pytest

from conftest import load_golden
from helpers import crf_case_inputs, digest, make_golden
from dsrg_b200 import api, synth
from oracle import crf_oracle

pytestmark = pytest.mark.gpu
TOL = 1e-4  # max |Q_gpu - Q_ref| (north_star: "within 1e-4 on the CRF's float marginals")


@pytest.mark.parametrize("name", [c[0] for c in make_golden.CRF_CASES])
def test_crf_golden_cases_object_api(torch_cuda, name):
    """krahenbuhl2013-shaped per-image object API (host pointers) vs the frozen golden marginals."""
    g = load_golden("crf_oracle_%s.npz" % name)
    im, unary, sf = crf_case_inputs(name)
    H, W, M = unary.shape
    c = api.DenseCRF(W, H, M)
    c.set_unary_energy(-unary.ravel().astype("float32"))
    c.add_pairwise_energy(10, 80 / sf, 80 / sf, 13, 13, 13, 3, 3 / sf, 3 / sf, im.ravel().astype("ubyte"))
    q = c.inference(10).reshape(H, W, M)
    assert np.abs(q - g["Q"]).max() <= TOL
    # map(): arg-max labels agree wherever the oracle's top-2 margin exceeds the tolerance
    lab = c.map(10).reshape(H, W)
    top2 = np.sort(g["Q"], -1)[..., -2:]
    clear = (top2[..., 1] - top2[..., 0]) > 4 * TOL
    assert np.array_equal(lab[clear], g["Q"].argmax(-1)[clear])


@pytest.mark.parametrize("H,W,sf,img,kind", [
    (41, 41, 12.0, "smooth", "p"),      # training shape (pylayers.py:82: scale_factor=12, unary=p)
    (41, 41, 12.0, "noise", "p"),
    (64, 48, 1.0, "smooth", "logp"),    # test-time shape (test-ms.py:106: unary=log p)
    (50, 75, 1.0, "noise", "logp"),
    (97, 113, 1.0, "smooth", "logp"),
    (321, 321, 1.0, "smooth", "p"),     # BASELINE.json config 3 shape (batch shortened to 3)
    (161, 200, 1.0, "noise", "p"),      # noise image: tiles overflow the shared-memory path -> direct path
    (5, 3, 1.0, "noise", "p"),          # tiny, N % 4 == 3 (one phantom lane)
    (4, 4, 12.0, "smooth", "p"),        # N % 4 == 0 (no phantom lanes)
    (1, 1, 1.0, "noise", "logp"),
])
def test_crf_batch_vs_oracle_both_layouts(torch_cuda, H, W, sf, img, kind):
    torch = torch_cuda
    B, M = 3, 21
    batch = synth.make_batch(B, H, W, image=img, start=40)
    pr = np.transpose(batch["probs"], (0, 2, 3, 1)).copy()
    pr[pr < 1e-5] = 1e-5
    unary = (pr if kind == "p" else np.log(pr)).astype(np.float32)
    want = np.stack([crf_oracle.CRF(batch["image"][b], unary[b], 10, sf) for b in range(B)])
    eng = api.Engine(B, H, W, M)
    params = api.crf_params(sf)
    d_im = torch.from_numpy(batch["image"]).cuda()
    # NHWC in / NHWC out
    d_un = torch.from_numpy(unary).cuda()
    d_out = torch.empty_like(d_un)
    eng.crf_dev(d_un, d_im, params, d_out)
    got = d_out.cpu().numpy()
    assert np.abs(got - want).max() <= TOL
    # NCHW in / NCHW out
    d_un2 = torch.from_numpy(np.ascontiguousarray(np.transpose(unary, (0, 3, 1, 2)))).cuda()
    d_out2 = torch.empty_like(d_un2)
    eng.crf_dev(d_un2, d_im, params, d_out2, api.LAYOUT_NCHW, api.LAYOUT_NCHW)
    got2 = np.transpose(d_out2.cpu().numpy(), (0, 2, 3, 1))
    assert np.abs(got2 - want).max() <= TOL
    # host entry point (H2D/D2H inside)
    got3 = eng.crf_host(unary, batch["image"], params)
    assert np.abs(got3 - want).max() <= TOL
    np.testing.assert_allclose(got.sum(-1), 1.0, atol=1e-5)
    eng.close()


def test_lattice_structure_matches_oracle(torch_cuda):
    """Vertex counts (incl. the phantom tail lanes, permutohedral.cpp:196) and the symmetric
    normalisation vectors (pairwise.cpp:54-57) against the CPU restatement."""
    torch = torch_cuda
    for H, W, sf, img in ((41, 41, 12.0, "smooth"), (37, 53, 1.0, "noise"), (64, 64, 1.0, "smooth")):
        B, M = 2, 21
        batch = synth.make_batch(B, H, W, image=img, start=7)
        unary = np.transpose(batch["probs"], (0, 2, 3, 1)).copy()
        eng = api.Engine(B, H, W, M)
        d_un = torch.from_numpy(unary).cuda()
        eng.crf_dev(d_un, torch.from_numpy(batch["image"]).cuda(), api.crf_params(sf, maxiter=1), torch.empty_like(d_un))
        vs, vb = eng.lattice_sizes(B)
        ns, nb = eng.norms(B)
        for b in range(B):
            c = crf_oracle.DenseCRF(W, H, M)
            c.set_unary_energy(-unary[b].ravel())
            c.add_pairwise_energy(10, 80 / sf, 80 / sf, 13, 13, 13, 3, 3 / sf, 3 / sf, batch["image"][b].ravel())
            assert vs == c.lattice(0).M and vb[b] == c.lattice(1).M
            np.testing.assert_allclose(ns, c.norm(0), rtol=2e-6)
            np.testing.assert_allclose(nb[b], c.norm(1), rtol=2e-6)
        eng.close()


def test_crf_error_paths(torch_cuda):
    torch = torch_cuda
    eng = api.Engine(2, 16, 16, 21)
    u = torch.zeros(3, 16, 16, 21, device="cuda")
    im = torch.zeros(3, 16, 16, 3, dtype=torch.uint8, device="cuda")
    with pytest.raises(api.DsrgError) as ei:      # batch larger than the engine
        eng.crf_dev(u, im, api.crf_params(), torch.empty_like(u))
    assert ei.value.code == -1
    p = api.crf_params()
    p.theta_alpha_x = 0.001                        # sigma so small that keys leave the packed range
    with pytest.raises(api.DsrgError) as ei:
        eng.crf_dev(u[:2], im[:2], p, torch.empty_like(u[:2]))
    assert ei.value.code == -3
    c = api.DenseCRF(8, 8, 21)
    im8 = np.zeros(8 * 8 * 3, np.uint8)
    c.add_pairwise_energy(10, 80, 80, 13, 13, 13, 3, 3, 3, im8)
    with pytest.raises(api.DsrgError) as ei:      # a second pairwise pair is refused (the reference would append it)
        c.add_pairwise_energy(10, 80, 80, 13, 13, 13, 3, 3, 3, im8)
    assert ei.value.code == -4
    eng.close()


@pytest.mark.parametrize("M", [2, 5, 8, 13, 32])
def test_crf_and_srg_other_label_counts(torch_cuda, M):
    """DenseCRF(W, H, nlabels) is generic in the label count (wrapper.pyx:23); the kernels are
    instantiated for every multiple of 4 up to DSRG_MAX_LABELS = 32."""
    from oracle import srg_oracle
    torch = torch_cuda
    H, W, B = 37, 45, 2
    rng = np.random.RandomState(M)
    logits = rng.randn(B, H, W, M).astype(np.float32) * 2
    pr = np.exp(logits - logits.max(-1, keepdims=True))
    pr /= pr.sum(-1, keepdims=True)
    unary = np.log(np.maximum(pr, 1e-5)).astype(np.float32)
    image = synth.make_batch(B, H, W, C=21, image="smooth", start=3)["image"]
    want = np.stack([crf_oracle.CRF(image[b], unary[b], 10, 1.0) for b in range(B)])
    eng = api.Engine(B, H, W, M)
    d_un = torch.from_numpy(unary).cuda()
    d_out = torch.empty_like(d_un)
    eng.crf_dev(d_un, torch.from_numpy(image).cuda(), api.crf_params(1.0), d_out)
    assert np.abs(d_out.cpu().numpy() - want).max() <= TOL
    # SRG with the same label count
    labels = np.zeros((B, M), np.float32)
    labels[:, 0] = 1
    labels[:, M - 1] = 1
    probs = np.ascontiguousarray(np.transpose(pr, (0, 3, 1, 2)))
    cues = (rng.rand(B, M, H, W) < 0.02).astype(np.float32)
    out = torch.empty(B, M, H, W, device="cuda")
    eng.srg_dev(torch.from_numpy(labels).cuda(), torch.from_numpy(probs).cuda(), torch.from_numpy(cues).cuda(), 0.6, 0.4, out)
    got = out.cpu().numpy()
    for b in range(B):
        assert np.array_equal(got[b], srg_oracle.srg_closed_form(labels[b], cues[b], probs[b], 0.6, 0.4))
    eng.close()


def test_label_count_limit_is_reported(torch_cuda):
    with pytest.raises(api.DsrgError):
        api.Engine(1, 8, 8, 256)
    eng = api.Engine(1, 8, 8, 33)       # wide path: CRF and SRG only
    with pytest.raises(api.DsrgError):
        eng.softmax_forward_host(np.zeros((1, 33, 8, 8), np.float32))
    eng.close()


@pytest.mark.parametrize("M,H,W,sf,img", [(33, 23, 31, 1.0, "smooth"), (81, 37, 45, 1.0, "smooth"), (81, 30, 26, 12.0, "noise")])
def test_crf_and_srg_wide_label_counts(torch_cuda, M, H, W, sf, img):
    """Label counts above 32 (the reference's COCO tool: DenseCRF(W, H, 81), training/tools/test-coco.py) run on the
    generic label-chunked path (csrc/meanfield_wide.cu): batch entry point in both layouts, the DenseCRF object,
    map(), and the SRG with the same label count -- against the oracles."""
    from oracle import srg_oracle
    torch = torch_cuda
    B = 2
    rng = np.random.RandomState(M + H)
    logits = rng.randn(B, H, W, M).astype(np.float32) * 2
    logits[:, H // 4: H // 2, W // 3:, 5] += 4
    pr = np.exp(logits - logits.max(-1, keepdims=True))
    pr /= pr.sum(-1, keepdims=True)
    unary = np.log(np.maximum(pr, 1e-5)).astype(np.float32)
    image = np.stack([synth.make_image(np.random.RandomState(9 + b), H, W, img) for b in range(B)])
    want = np.stack([crf_oracle.CRF(image[b], unary[b], 10, sf) for b in range(B)])
    eng = api.Engine(B, H, W, M)
    d_un = torch.from_numpy(unary).cuda()
    d_out = torch.empty_like(d_un)
    eng.crf_dev(d_un, torch.from_numpy(image).cuda(), api.crf_params(sf), d_out)
    assert np.abs(d_out.cpu().numpy() - want).max() <= TOL
    d_nchw = d_un.permute(0, 3, 1, 2).contiguous()
    d_out2 = torch.empty_like(d_nchw)
    eng.crf_dev(d_nchw, torch.from_numpy(image).cuda(), api.crf_params(sf), d_out2, unary_layout=1, out_layout=1)
    assert np.abs(d_out2.permute(0, 2, 3, 1).cpu().numpy() - want).max() <= TOL
    c = api.DenseCRF(W, H, M)
    c.set_unary_energy(-unary[0].ravel())
    c.add_pairwise_energy(10, 80 / sf, 80 / sf, 13, 13, 13, 3, 3 / sf, 3 / sf, image[0].ravel())
    assert np.abs(c.inference(10).reshape(H, W, M) - want[0]).max() <= TOL
    top2 = np.sort(want[0], -1)[..., -2:]
    clear = (top2[..., 1] - top2[..., 0]) > 4 * TOL
    assert np.array_equal(c.map(10).reshape(H, W)[clear], want[0].argmax(-1)[clear])
    # SRG with the same label count
    labels = np.zeros((B, M), np.float32)
    labels[:, [0, 5, M - 1]] = 1
    probs = np.ascontiguousarray(np.transpose(want, (0, 3, 1, 2)))
    cues = (rng.rand(B, M, H, W) < 0.01).astype(np.float32)
    seeds = eng.srg_host(labels, probs, cues, 0.99, 0.3)
    for b in range(B):
        assert np.array_equal(seeds[b], srg_oracle.srg_closed_form(labels[b], cues[b], probs[b], 0.99, 0.3))
    eng.close()


@pytest.mark.parametrize("n_iters", [0, 1, 2, 3])
def test_crf_iteration_counts(torch_cuda, n_iters):
    """maxiter = 0 returns softmax(unary) (densecrf.cpp:120); 1 and 2 exercise the first / last / middle
    variants of the fused kernel."""
    torch = torch_cuda
    B, H, W, M = 2, 33, 47, 21
    batch = synth.make_batch(B, H, W, image="smooth", start=21)
    unary = np.ascontiguousarray(np.log(np.maximum(np.transpose(batch["probs"], (0, 2, 3, 1)), 1e-5)), np.float32)
    want = np.stack([crf_oracle.CRF(batch["image"][b], unary[b], n_iters, 1.0) for b in range(B)])
    eng = api.Engine(B, H, W, M)
    for layout in (api.LAYOUT_NHWC, api.LAYOUT_NCHW):
        u = unary if layout == api.LAYOUT_NHWC else np.ascontiguousarray(np.transpose(unary, (0, 3, 1, 2)))
        d_un = torch.from_numpy(u).cuda()
        d_out = torch.empty_like(d_un)
        eng.crf_dev(d_un, torch.from_numpy(batch["image"]).cuda(), api.crf_params(1.0, maxiter=n_iters), d_out, layout, layout)
        got = d_out.cpu().numpy()
        if layout == api.LAYOUT_NCHW:
            got = np.transpose(got, (0, 2, 3, 1))
        assert np.abs(got - want).max() <= TOL
    eng.close()


def test_engine_reuse_changing_parameters_and_batch(torch_cuda):
    """One engine, many calls: partial batches, changing sigmas (the spatial lattice cache must be
    invalidated), changing images; every call must still match a fresh oracle run."""
    torch = torch_cuda
    H, W, M, Bmax = 40, 52, 21, 5
    eng = api.Engine(Bmax, H, W, M)
    calls = [(5, 1.0, 13, "smooth", 0), (2, 12.0, 13, "noise", 9), (3, 1.0, 13, "smooth", 4), (1, 3.0, 20, "smooth", 2),
             (5, 1.0, 13, "smooth", 0)]
    for B, sf, cf, img, start in calls:
        batch = synth.make_batch(B, H, W, image=img, start=start)
        unary = np.ascontiguousarray(np.transpose(batch["probs"], (0, 2, 3, 1)))
        want = np.stack([crf_oracle.CRF(batch["image"][b], unary[b], 10, sf, cf) for b in range(B)])
        got = eng.crf_host(unary, batch["image"], api.crf_params(sf, cf, 10))
        assert np.abs(got - want).max() <= TOL, (B, sf, cf, img)
    eng.close()


def test_crf_random_shapes_fuzz(torch_cuda):
    """Seeded fuzz over small odd shapes (narrower than a tile, single rows / columns, ...)."""
    rng = np.random.RandomState(2024)
    for case in range(10):
        H, W = int(rng.randint(1, 70)), int(rng.randint(1, 70))
        M = int(rng.choice([3, 21]))
        sf = float(rng.choice([1.0, 12.0]))
        B = int(rng.randint(1, 4))
        logits = rng.randn(B, H, W, M).astype(np.float32)
        unary = logits - np.log(np.exp(logits).sum(-1, keepdims=True))
        image = rng.randint(0, 256, (B, H, W, 3)).astype(np.uint8) if case % 2 else \
            np.stack([synth.make_image(rng, H, W, "smooth") for _ in range(B)])
        want = np.stack([crf_oracle.CRF(image[b], unary[b], 10, sf) for b in range(B)])
        eng = api.Engine(B, H, W, M)
        got = eng.crf_host(np.ascontiguousarray(unary, np.float32), np.ascontiguousarray(image), api.crf_params(sf))
        assert np.abs(got - want).max() <= TOL, (case, H, W, M, sf, B)
        eng.close()


def test_densecrf_objects_share_one_engine(torch_cuda):
    """The reference makes one DenseCRF per image (CRF.py:21); ours borrow a pooled engine, so objects of
    different sizes can be created up front and run in any order without leaking state into each other."""
    from dsrg_b200 import _lib
    cases = []
    for i, (H, W) in enumerate([(24, 40), (40, 24), (70, 90), (24, 40)]):
        p = synth.make_problem(900 + i, H, W, image="smooth" if i % 2 else "noise")
        pr = np.transpose(p["probs"], (1, 2, 0)).copy()
        pr[pr < 1e-5] = 1e-5
        c = api.DenseCRF(W, H, 21)
        c.set_unary_energy(-np.log(pr).ravel())
        c.add_pairwise_energy(10, 80, 80, 13, 13, 13, 3, 3, 3, p["image"].ravel())
        cases.append((c, p["image"], np.log(pr), H, W))
    for k in (2, 0, 3, 1, 2):
        c, im, unary, H, W = cases[k]
        want = crf_oracle.CRF(im, unary, scale_factor=1.0)
        got = c.inference(10).reshape(H, W, 21)
        assert np.abs(got - want).max() <= 1e-4
        lab = c.map(10).reshape(H, W)
        bad = lab != want.argmax(2)
        if bad.any():
            top2 = np.sort(want, axis=2)[:, :, -2:]
            assert ((top2[:, :, 1] - top2[:, :, 0])[bad] <= 4e-4).all()
    with pytest.raises(api.DsrgError):
        api.DenseCRF(8, 8, 256)              # DSRG_MAX_LABELS_WIDE = 255
    _lib.lib().dsrg_densecrf_release_engines()
    got = cases[0][0].inference(10)            # the pool is re-created on demand
    assert np.isfinite(got).all()


@pytest.mark.parametrize("H,W,sf,img", make_golden.CRF_DIRECT_CASES)
def test_crf_against_the_reference_build_directly(torch_cuda, H, W, sf, img):
    """CUDA path vs the reference's OWN CRF sources (compiled unmodified, oracle/Makefile): marginals within 1e-4,
    MAP labels equal except at near-ties.  The reference build's outputs are the C restatement's, bit for bit:
    the digests of that build's outputs in crf_ref_build.npz say so for these very inputs."""
    g = load_golden("crf_ref_build.npz")
    key = make_golden.crf_direct_key(H, W)
    im, unary = make_golden.crf_direct_inputs(H, W, sf, img)
    assert digest(im, unary) == str(g[key + "/inputs_sha256"])
    want = crf_oracle.CRF(im, unary, 10, sf)
    assert digest(want) == str(g[key + "/crf"]), "the restatement no longer reproduces the reference build"
    eng = api.Engine(1, H, W, 21)
    got = eng.crf_host(unary[None], im[None], api.crf_params(sf))[0]
    assert np.abs(got - want).max() <= 1e-4
    b = make_golden.crf_objects(crf_oracle.DenseCRF, im, unary, sf).map(10)
    assert digest(b) == str(g[key + "/map"]), "the restatement no longer reproduces the reference build"
    a = make_golden.crf_objects(api.DenseCRF, im, unary, sf).map(10)
    bad = a != b
    if bad.any():
        top2 = np.sort(want.reshape(-1, 21), axis=1)[:, -2:]
        assert ((top2[:, 1] - top2[:, 0])[bad] <= 4e-4).all()
    eng.close()


def test_densecrf_object_without_pairwise_and_second_pairwise_call(torch_cuda):
    """DenseCRFWrapper semantics at the edges: with no pairwise term inference() is softmax(-unary) after any
    number of iterations (densecrf.cpp:115-131 with an empty pairwise list) -- checked against the reference-built
    oracle object; a second add_pairwise_energy (which the reference would APPEND, densecrf_wrapper.cpp:25-29) is
    refused with a clear error instead of silently replacing the first."""
    rng = np.random.RandomState(3)
    H, W, M = 9, 7, 5
    unary = rng.randn(H, W, M).astype(np.float32)
    c = api.DenseCRF(W, H, M)
    c.set_unary_energy(unary.ravel())
    o = crf_oracle.DenseCRF(W, H, M)
    o.set_unary_energy(unary.ravel())
    for it in (0, 3):
        got = c.inference(it).reshape(H, W, M)
        np.testing.assert_allclose(got, o.inference(it).reshape(H, W, M), atol=2e-6)
        assert np.array_equal(c.map(it), o.map(it))
    im = synth.make_image(rng, H, W, "noise")
    c.add_pairwise_energy(10, 80, 80, 13, 13, 13, 3, 3, 3, im.ravel())
    with pytest.raises(api.DsrgError):
        c.add_pairwise_energy(10, 80, 80, 13, 13, 13, 3, 3, 3, im.ravel())


def test_entry_points_keep_the_callers_current_device(torch_cuda):
    """ADVICE r1: a drop-in call must not leave the calling (solver) thread on another CUDA device."""
    torch = torch_cuda
    from dsrg_b200 import _lib
    L = _lib.lib()
    assert L.dsrg_current_device() == torch.cuda.current_device()
    n = torch.cuda.device_count()
    target = n - 1                       # another device when the box has more than one
    eng = api.Engine(1, 16, 16, 21, device=target)
    assert torch.cuda.current_device() == 0 and L.dsrg_current_device() == 0
    b = synth.make_batch(1, 16, 16, start=5)
    out = eng.crf_host(np.ascontiguousarray(np.transpose(b["probs"], (0, 2, 3, 1))), b["image"], api.crf_params(1.0))
    assert np.isfinite(out).all()
    assert torch.cuda.current_device() == 0 and L.dsrg_current_device() == 0
    eng.close()
    assert api.Engine(1, 8, 8, 3).device == 0   # default = the current device


def test_crf_hybrid_tiles_on_textured_images(torch_cuda):
    """Textured images (1/f spectrum): nearly every tile has more distinct bilateral vertices than k_mf_tile's shared
    memory holds.  Such tiles keep their most-touched vertices in a tile-local list and send the other incidences
    straight to global memory (k_mf_tile_hy, csrc/tiles.cu).  Parity with the oracle as everywhere else, for a
    batch that mixes textured and smooth images (both kernels work on the same lattices), replayed as a graph; a
    batch with only a few overflow tiles hands them back to the plain kernel's direct path, and so does a pass
    that is too small to be worth the extra launches."""
    torch = torch_cuda
    H = W = 321
    B, M = 6, 21
    ph = synth.make_batch(5, H, W, image="photo", start=70)
    sm = synth.make_batch(B, H, W, image="smooth", start=75)
    image = np.concatenate([ph["image"][:1], sm["image"][:1], ph["image"][1:]])
    probs = np.concatenate([ph["probs"][:1], sm["probs"][:1], ph["probs"][1:]])

    def unary_of(p):
        pr = np.transpose(p, (0, 2, 3, 1)).copy()
        pr[pr < 1e-5] = 1e-5
        return np.log(pr).astype(np.float32)

    unary = unary_of(probs)
    want = np.stack([crf_oracle.CRF(image[b], unary[b], 10, 1.0) for b in range(B)])
    eng = api.Engine(B, H, W, M)
    params = api.crf_params(1.0)
    d_im = torch.from_numpy(image).cuda()
    d_un = torch.from_numpy(unary).cuda()
    d_out = torch.empty_like(d_un)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        for rnd in range(4):                       # eager, captured, replayed, replayed
            d_out.zero_()
            eng.crf_dev(d_un, d_im, params, d_out, stream=stream.cuda_stream)
            stream.synchronize()
            assert np.abs(d_out.cpu().numpy() - want).max() <= TOL, rnd
    assert eng.graph_replays >= 2
    ntiles = 11 * 41                               # 30x8-pixel tiles at 321x321
    nh = eng.hybrid_tiles
    assert 8 * 148 <= nh <= 5 * ntiles + 0.1 * ntiles, nh   # the five textured images, a few tiles of the smooth one
    # six smooth images: their few overflow tiles do not make a hybrid pass (k_tile_demote)
    un2 = unary_of(sm["probs"])
    d_out2 = torch.empty((B, H, W, M), dtype=torch.float32, device="cuda")
    eng.crf_dev(torch.from_numpy(un2).cuda(), torch.from_numpy(sm["image"]).cuda(), params, d_out2)
    torch.cuda.synchronize()
    got2 = d_out2.cpu().numpy()
    assert np.abs(got2[0] - want[1]).max() <= TOL
    assert np.abs(got2[3] - crf_oracle.CRF(sm["image"][3], un2[3], 10, 1.0)).max() <= TOL
    assert eng.hybrid_tiles == 0
    # two textured images alone: a pass below 16 tiles per SM stays on the plain kernel
    d_out3 = torch.empty((2, H, W, M), dtype=torch.float32, device="cuda")
    eng.crf_dev(d_un[2:4].contiguous(), d_im[2:4].contiguous(), params, d_out3)
    torch.cuda.synchronize()
    assert np.abs(d_out3.cpu().numpy() - want[2:4]).max() <= TOL
    assert eng.hybrid_tiles == 0
    eng.close()
