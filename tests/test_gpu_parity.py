"""GPU parity tests: the CUDA product (through the public API -> C ABI) against
  (a) the re-hosted reference kernels (oracle/refhost.py, exact oracle: face_index_map bit-exact, values <= 1e-4),
      through the digests of their results stored under tests/golden/ref (tests/refgolden.py),
  (b) the CPU oracle (oracle/nr_oracle.c) at sizes it finishes in seconds,
  (c) the committed golden fixtures of the reference's own tests,
  (d) size-independent properties at the BASELINE.json headline shape.
Tolerance (BASELINE.json north_star): face_index_map bit-exact; rgb / alpha / depth / gradients within 1e-4 relative
(max-abs-error / max-abs-reference per tensor)."""
import zlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-4

from helpers import np_, rel_err, to_minibatch  # noqa: E402
from refgolden import RefGolden  # noqa: E402


def _skip_without_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="module", autouse=True)
def _gpu():
    _skip_without_gpu()
    from neural_renderer_b200 import _lib
    _lib.load()  # fail loudly if the CUDA library is missing on a GPU box
    yield


def _inputs(kind, B, F, ts, seed):
    from neural_renderer_b200 import synthetic
    if kind == "soup":
        faces = synthetic.triangle_soup(B, F, seed=seed)
    elif kind == "big":
        faces = synthetic.triangle_soup(B, F, seed=seed, size=(0.6, 1.6))
    elif kind == "sphere":
        faces = synthetic.sphere_faces(B, F, seed=seed)
    else:
        raise ValueError(kind)
    tex = synthetic.random_textures(B, F, ts, seed=seed + 7) if ts else None
    return faces, tex


def _run_product(faces, tex, image_size, aa, near, far, eps, bg, flags, grads=None):
    import importlib
    R = importlib.import_module("neural_renderer_b200.rasterize")
    dev = torch.device("cuda")
    f = torch.from_numpy(faces).to(dev).requires_grad_(True)
    t = torch.from_numpy(tex).to(dev).requires_grad_(True) if (tex is not None and flags[0]) else None
    rgb, alpha, depth, fim, wmap = R._run(f, t, image_size, aa, near, far, eps, bg, *flags)
    out = {"rgb": rgb, "alpha": alpha, "depth": depth, "fim": fim, "wmap": wmap, "faces": f, "tex": t}
    if grads is not None:
        loss = 0
        for k in ("rgb", "alpha", "depth"):
            if out[k] is not None and grads.get(k) is not None:
                loss = loss + (out[k] * grads[k]).sum()
        loss.backward()
        out["grad_faces"] = f.grad
        out["grad_tex"] = t.grad if t is not None else None
    torch.cuda.synchronize()
    return out


def _grads(shape_src, seed):
    g = {}
    gen = torch.Generator(device="cpu").manual_seed(seed)
    for k in ("rgb", "alpha", "depth"):
        if shape_src[k] is not None:
            g[k] = torch.randn(shape_src[k].shape, generator=gen).to(shape_src[k].device)
    return g


def _reference(gold, faces, tex, image_size, aa, near, far, eps, bg, flags):
    """While `gold` records: the reference kernels' forward on these inputs, its maps put into `gold`; the result
    (whose .backward gives the reference gradients) is returned.  None when the stored digests are compared."""
    if not gold.recording:
        return None
    import refhost
    dev = torch.device("cuda")
    faces = torch.as_tensor(faces).to(dev)
    tex = torch.as_tensor(tex).to(dev) if flags[0] else None
    S = image_size * 2 if aa else image_size
    assert refhost.available(S, faces.shape[1], tex.shape[2] if flags[0] else 0, near, far, eps, *flags), \
        "reference kernels for this configuration were not built (oracle/build_ref.py)"
    ref = refhost.rasterize_rgbad(faces, tex, image_size, aa, near, far, eps, bg, *flags)
    gold.put("fim", ref.fn.face_index_map, exact_only=True)
    gold.put("wmap", ref.fn.weight_map, exact_only=True)
    for k in ("rgb", "alpha", "depth"):
        if ref[k] is not None:
            gold.put(k, ref[k], exact_only=not aa)
    return ref


def _record_backward(gold, ref, grads, flags):
    """While `gold` records: the reference gradients for upstream `grads`, put into `gold`, which is saved."""
    if gold.recording:
        gf, gt = ref.backward(grads.get("rgb"), grads.get("alpha"), grads.get("depth"))
        gold.put("grad_faces", gf)
        if flags[0]:
            gold.put("grad_tex", gt)
        gold.save()


def _compare_forward(gold, got, aa):
    # face_index_map: bit-exact (ours is stored in image orientation, the reference's un-flipped)
    assert gold.equal("fim", got["fim"].flip(1)), "face_index_map differs"
    # the forward maps replay the reference's fp32 expression trees, so they are expected to match bit for bit
    # (the contract only asks for 1e-4; the stricter check guards the pinned arithmetic of nr_math.cuh)
    assert gold.equal("wmap", got["wmap"].permute(0, 2, 3, 1).flip(1)), "weight_map not bit-exact"
    for k in ("rgb", "alpha", "depth"):
        if k in gold:
            if aa:
                assert gold.rel_err(k, got[k]) <= TOL, k
            else:
                assert gold.equal(k, got[k]), "%s: values differ in the last bits" % k


def _compare_backward(gold, got, flags):
    assert gold.rel_err("grad_faces", got["grad_faces"]) <= TOL, "grad_faces"
    if flags[0]:
        assert gold.rel_err("grad_tex", got["grad_tex"]) <= TOL, "grad_textures"


# (name, image_size, anti_aliasing, F, ts, (rgb, alpha, depth), near, far, eps, mesh kind, B)
CASES = [
    ("tiny_all", 32, False, 64, 2, (1, 1, 1), 0.1, 100, 1e-4, "soup", 3),
    ("soup_rgb", 64, False, 200, 4, (1, 0, 0), 0.1, 100, 1e-4, "soup", 4),
    ("soup_alpha", 64, False, 200, 4, (0, 1, 0), 0.1, 100, 1e-4, "soup", 4),
    ("soup_depth", 64, False, 200, 4, (0, 0, 1), 0.1, 100, 1e-4, "soup", 4),
    ("soup_all", 64, False, 200, 4, (1, 1, 1), 0.1, 100, 1e-4, "soup", 4),
    ("npot_all", 100, False, 150, 3, (1, 1, 1), 0.1, 100, 1e-4, "soup", 2),
    ("aa_all", 64, True, 200, 4, (1, 1, 1), 0.1, 100, 1e-4, "soup", 3),
    ("nearfar", 64, False, 200, 2, (1, 1, 1), 2.2, 3.0, 1e-4, "sphere", 2),
    ("bigfaces", 128, False, 24, 2, (1, 1, 1), 0.1, 100, 1e-4, "big", 2),
    ("sphere192", 192, False, 2000, 2, (1, 1, 0), 0.1, 100, 1e-4, "sphere", 2),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_forward_backward_vs_reference_kernels(case):
    name, image_size, aa, F, ts, flags, near, far, eps, kind, B = case
    faces, tex = _inputs(kind, B, F, ts, seed=zlib.crc32(name.encode()) % 1000)
    bg = (0.1, 0.3, 0.5) if name != "soup_all" else np.linspace(0.0, 0.9, B * 3).reshape(B, 3).astype(np.float32)
    gold = RefGolden("parity_" + name)
    ref = _reference(gold, faces, tex, image_size, aa, near, far, eps, bg, flags)
    grads = _grads(_run_product(faces, tex, image_size, aa, near, far, eps, bg, flags), seed=99)
    _record_backward(gold, ref, grads, flags)
    got = _run_product(faces, tex, image_size, aa, near, far, eps, bg, flags, grads)
    _compare_forward(gold, got, aa)
    _compare_backward(gold, got, flags)


def _outside_box_wins(fim, faces, S):
    """Pixels whose winning face does not contain them in the pixel box of its three vertices (+- 1/256 px)."""
    n = 0
    for b in range(fim.shape[0]):
        ys, xs = np.nonzero(fim[b] >= 0)
        v = faces[b, fim[b, ys, xs]]  # [n,3,3]
        px, py = 0.5 * (v[:, :, 0] * S + S - 1), 0.5 * (v[:, :, 1] * S + S - 1)
        n += int(((xs > np.ceil(px.max(1) + 1 / 256)) | (xs < np.floor(px.min(1) - 1 / 256)) |
                  (ys > np.ceil(py.max(1) + 1 / 256)) | (ys < np.floor(py.min(1) - 1 / 256))).sum())
    return n


@pytest.mark.parametrize("flags", [(0, 1, 0), (1, 1, 1)], ids=["alpha", "all"])
def test_needle_faces(flags):
    """Needles whose long edges meet at 1e-7 .. 1e-4 rad win pixels BEYOND their tip in the reference (the fp32 edge
    tests of rasterize.py:309-311 accept a pixel centre on the needle's axis): the forward's conservative pixel box has
    to reach them (nr_bbox.cuh thin_face_margin).  Half of the faces are ordinary triangles that compete for the pixels."""
    from neural_renderer_b200 import synthetic
    image_size, F, ts, B, near, far, eps = 64, 200, 4, 3, 0.1, 100, 1e-4
    faces = synthetic.triangle_soup(B, F, seed=11, z_range=(1.5, 3.0))
    faces[:, : F // 2] = synthetic.needle_faces(B, F // 2, image_size, seed=5)
    tex = synthetic.random_textures(B, F, ts, seed=3)
    bg = (0.1, 0.3, 0.5)
    gold = RefGolden("parity_needles_" + "".join(map(str, flags)))
    _reference(gold, faces, tex, image_size, False, near, far, eps, bg, flags)
    gold.save()
    got = _run_product(faces, tex, image_size, False, near, far, eps, bg, flags)
    # (the face_index_map equals the reference's bit for bit, so the product's map shows the reference's winners)
    _compare_forward(gold, got, False)
    assert _outside_box_wins(np_(got["fim"].flip(1)), faces, image_size) >= 20, \
        "the case does not exercise the thin-face margin"


@pytest.mark.parametrize("case", [c for c in CASES if c[0] in ("tiny_all", "soup_all", "npot_all", "aa_all")],
                         ids=lambda c: c[0])
def test_forward_backward_vs_cpu_oracle(case):
    import nr_oracle as o
    name, image_size, aa, F, ts, flags, near, far, eps, kind, B = case
    faces, tex = _inputs(kind, B, F, ts, seed=zlib.crc32(name.encode()) % 1000 + 1)
    bg = (0.2, 0.4, 0.6)
    ref = o.rasterize_rgbad(faces, tex, image_size, aa, near, far, eps, bg, *flags)
    got0 = _run_product(faces, tex, image_size, aa, near, far, eps, bg, flags)
    grads = _grads(got0, seed=5)
    got = _run_product(faces, tex, image_size, aa, near, far, eps, bg, flags, grads)
    assert np.array_equal(np_(got["fim"].flip(1)), ref.fn.face_index_map)
    for k in ("rgb", "alpha", "depth"):
        assert rel_err(np_(got[k]), ref[k]) <= TOL, k
    gf, gt = ref.backward(*[np_(grads[k]) for k in ("rgb", "alpha", "depth")])
    assert rel_err(np_(got["grad_faces"]), gf) <= TOL
    assert rel_err(np_(got["grad_tex"]), gt) <= TOL


# (name, image_size, aa, F, ts, flags, near, far, eps, kind, B, z_range)
MORE = [
    ("one_face", 16, False, 1, 2, (1, 1, 1), 0.1, 100, 1e-4, "big", 1, (1.0, 3.0)),
    ("f33_ts3", 48, False, 33, 3, (1, 1, 1), 0.1, 100, 1e-4, "soup", 2, (1.0, 3.0)),
    ("f257_ts5", 130, False, 257, 5, (1, 0, 1), 0.1, 100, 1e-3, "soup", 1, (1.0, 3.0)),
    ("ts8_aa", 40, True, 40, 8, (1, 1, 0), 0.1, 100, 1e-4, "soup", 2, (1.0, 3.0)),
    ("behind_camera", 64, False, 120, 2, (1, 1, 1), 0.1, 100, 1e-4, "soup", 2, (-1.0, 3.0)),
    ("depth_aa", 32, True, 60, 2, (0, 0, 1), 0.5, 2.5, 1e-4, "soup", 2, (1.0, 3.0)),
    ("alpha_aa_big", 96, True, 12, 2, (0, 1, 0), 0.1, 100, 1e-4, "big", 2, (1.0, 3.0)),
]


@pytest.mark.parametrize("case", MORE, ids=[c[0] for c in MORE])
def test_more_shapes_vs_cpu_oracle(case):
    """Odd sizes the tiling has to clip (rasters smaller than / not a multiple of the 64-pixel tile, face counts that
    are not a multiple of the 32-face groups), every texture size, faces behind the camera, anti-aliased single
    outputs -- all against the CPU oracle."""
    import nr_oracle as o
    from neural_renderer_b200 import synthetic
    name, image_size, aa, F, ts, flags, near, far, eps, kind, B, zr = case
    seed = zlib.crc32(name.encode()) % 1000
    size = (0.6, 1.6) if kind == "big" else (0.05, 0.5)
    faces = synthetic.triangle_soup(B, F, seed=seed, size=size, z_range=zr)
    tex = synthetic.random_textures(B, F, ts, seed=seed + 7)
    bg = (0.3, 0.2, 0.1)
    ref = o.rasterize_rgbad(faces, tex if flags[0] else None, image_size, aa, near, far, eps, bg, *flags)
    got0 = _run_product(faces, tex, image_size, aa, near, far, eps, bg, flags)
    grads = _grads(got0, seed=11)
    got = _run_product(faces, tex, image_size, aa, near, far, eps, bg, flags, grads)
    assert np.array_equal(np_(got["fim"].flip(1)), ref.fn.face_index_map)
    for k in ("rgb", "alpha", "depth"):
        if ref[k] is not None:
            assert rel_err(np_(got[k]), ref[k]) <= TOL, k
    gf, gt = ref.backward(*[np_(grads[k]) if k in grads else None for k in ("rgb", "alpha", "depth")])
    assert rel_err(np_(got["grad_faces"]), gf) <= TOL
    if flags[0]:
        assert rel_err(np_(got["grad_tex"]), gt) <= TOL


def test_partial_upstream_gradients():
    """rasterize_rgbad with all three outputs but a loss on alpha only: missing upstream gradients are zeros
    (rasterize.py:858-878)."""
    import nr_oracle as o
    faces, tex = _inputs("soup", 2, 64, 2, seed=21)
    ref = o.rasterize_rgbad(faces, tex, 32, False, 0.1, 100, 1e-4, (0, 0, 0), True, True, True)
    got0 = _run_product(faces, tex, 32, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 1, 1))
    g = _grads(got0, seed=3)
    got = _run_product(faces, tex, 32, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 1, 1), {"alpha": g["alpha"]})
    gf, gt = ref.backward(None, np_(g["alpha"]), None)
    assert rel_err(np_(got["grad_faces"]), gf) <= TOL
    assert got["grad_tex"] is None or float(got["grad_tex"].abs().max()) == 0.0


def test_reference_exact_switch_changes_only_texture_depths():
    """rasterize.py:389 quirk: with per-item geometry the sampler reads batch item 0's vertex depths."""
    import nr_oracle as o
    import neural_renderer_b200 as nrb
    faces, tex = _inputs("soup", 3, 64, 2, seed=3)
    try:
        nrb.set_reference_exact(False)
        got = _run_product(faces, tex, 32, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 0, 0))
    finally:
        nrb.set_reference_exact(True)
    ref = o.rasterize_rgbad(faces, tex, 32, False, 0.1, 100, 1e-4, (0, 0, 0), True, False, False, tex_z_batch0=False)
    assert rel_err(np_(got["rgb"]), ref["rgb"]) <= TOL


# ------------------------------------------------------------------------------------------------ golden fixtures
def _teapot_batch(teapot, dev):
    v, f = teapot
    tex = np.ones((f.shape[0], 4, 4, 4, 3), np.float32)
    v, f, tex = to_minibatch((v, f, tex))
    return torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev), torch.from_numpy(tex).to(dev)


def test_golden_teapot_images(teapot, golden_images):
    import neural_renderer as nr
    dev = torch.device("cuda")
    v, f, tex = _teapot_batch(teapot, dev)
    r = nr.Renderer()
    r.image_size, r.anti_aliasing = 256, False
    sil = np_(r.render_silhouettes(v, f))[2]
    assert (sil != golden_images["silhouette"]).sum() == 0            # test_rasterize_silhouettes.py:15-35
    d = np_(r.render_depth(v, f))[2]
    assert ((d != d.max()).astype(np.float32) != golden_images["silhouette"]).sum() == 0  # test_rasterize_depth.py:16-37
    d[d == d.max()] = d.min()
    d = (d - d.min()) / (d.max() - d.min())
    np.testing.assert_allclose(d, golden_images["depth_u8"].astype(np.float32) / 255., atol=1e-2)  # :39-58
    r.light_intensity_ambient, r.light_intensity_directional = 1.0, 0.0
    img = np_(r.render(v, f, tex))[2].mean(0)
    np.testing.assert_allclose(img, golden_images["silhouette"], rtol=1e-4, atol=1e-5)  # test_rasterize.py:52-74


@pytest.mark.parametrize("mode", ["silhouette", "rgb"])
def test_golden_known_answer_gradients(kat, mode):
    import neural_renderer as nr
    dev = torch.device("cuda")
    for c in kat["cases"]:
        r = nr.Renderer()
        r.image_size, r.anti_aliasing, r.perspective = 64, False, False
        vv, ff, gref = to_minibatch((np.array(c["vertices"], np.float32), np.array(c["faces"], np.int32),
                                     np.array(c["grad_ref"], np.float32)))
        vertices = torch.from_numpy(vv).to(dev).requires_grad_(True)
        faces = torch.from_numpy(ff).to(dev)
        minus = 1.0 if c["name"] == "out_of_face" else 0.0
        if mode == "silhouette":
            images = r.render_silhouettes(vertices, faces)
            tol = 1e-3
        else:
            r.light_intensity_ambient, r.light_intensity_directional = 1.0, 0.0
            tt, = to_minibatch((np.ones((1, 4, 4, 4, 3), np.float32),))
            images = r.render(vertices, faces, torch.from_numpy(tt).to(dev)).mean(dim=1)
            tol = 1e-2
        loss = (images[:, c["pyi"], c["pxi"]] - minus).abs().sum()
        loss.backward()
        np.testing.assert_allclose(np_(vertices.grad), gref, rtol=tol, atol=tol * 1e-2)


def test_teapot_renderer_defaults_vs_reference_kernels(teapot):
    """BASELINE.json config 2 shape: teapot through Renderer defaults (fill_back, anti-aliasing, lighting), fwd+bwd."""
    import neural_renderer as nr
    dev = torch.device("cuda")
    v, f = teapot
    B = 2
    vertices = torch.from_numpy(np.stack([v, v])).to(dev)
    faces_idx = torch.from_numpy(np.stack([f, f])).to(dev)
    tex = torch.rand((B, f.shape[0], 4, 4, 4, 3), generator=torch.Generator().manual_seed(1)).to(dev)
    r = nr.Renderer()
    r.eye = nr.get_points_from_angles(2.732, 30, 40)
    # build the rasterizer inputs exactly as Renderer.render does, then compare both rasterizers on them
    fi = torch.cat((faces_idx, faces_idx.flip(2)), dim=1)
    tx = torch.cat((tex, tex.permute(0, 1, 4, 3, 2, 5)), dim=1)
    tx = nr.lighting(nr.vertices_to_faces(vertices, fi), tx)
    faces = nr.vertices_to_faces(nr.perspective(nr.look_at(vertices, r.eye)), fi).contiguous()
    gold = RefGolden("parity_teapot_renderer_defaults")
    ref = _reference(gold, faces, tx.contiguous(), 256, True, 0.1, 100, 1e-3, [0, 0, 0], (1, 0, 0))
    g = torch.randn((B, 3, 256, 256), generator=torch.Generator().manual_seed(2)).to(dev)
    _record_backward(gold, ref, {"rgb": g}, (1, 0, 0))
    fa = faces.clone().requires_grad_(True)
    ta = tx.clone().requires_grad_(True)
    img = nr.rasterize(fa, ta, 256, True, 0.1, 100, 1e-3, [0, 0, 0])
    (img * g).sum().backward()
    assert gold.rel_err("rgb", img) <= TOL
    assert gold.rel_err("grad_faces", fa.grad) <= TOL
    assert gold.rel_err("grad_tex", ta.grad) <= TOL
    # and the facade itself produces that image
    img2 = r.render(vertices, faces_idx, tex)
    assert gold.rel_err("rgb", img2) <= TOL


# ---------------------------------------------------------------------- properties at the headline shape (B=64)
@pytest.fixture(scope="module")
def headline():
    from neural_renderer_b200 import synthetic
    B, F, ts = 64, 5000, 4
    return synthetic.sphere_faces(B, F), synthetic.random_textures(B, F, ts)


def test_headline_properties(headline):
    faces, tex = headline
    bg = (0.25, 0.5, 0.75)
    a = _run_product(faces, tex, 256, False, 0.1, 100, 1e-4, bg, (1, 1, 1))
    b = _run_product(faces, tex, 256, False, 0.1, 100, 1e-4, bg, (1, 1, 1))
    # forward is deterministic (bit-identical maps on repeated runs)
    for k in ("fim", "rgb", "alpha", "depth", "wmap"):
        assert torch.equal(a[k], b[k]), k
    covered = a["fim"] >= 0
    assert covered.float().mean().item() > 0.3                     # the spheres cover about half of each image
    assert torch.equal(a["alpha"], covered.float())                 # alpha == coverage
    assert torch.all(a["depth"][~covered] == 100.0)                 # uncovered depth == far
    assert torch.all((a["depth"][covered] > 1.8) & (a["depth"][covered] < 3.7))
    for c in range(3):
        assert torch.all(a["rgb"][:, c][~covered] == bg[c])         # uncovered rgb == background
    w = a["wmap"]
    assert torch.all(w[:, 0][~covered] == 0) and torch.allclose(w.sum(1)[covered], torch.ones(()).cuda(), atol=1e-5)
    # batch items are independent: a slice rendered alone reproduces its rows (alpha / depth / fim; rgb is excluded
    # because of the batch-0 quirk of the texture sampler)
    s = _run_product(faces[5:9], tex[5:9], 256, False, 0.1, 100, 1e-4, bg, (0, 1, 1))
    assert torch.equal(s["fim"], a["fim"][5:9]) and torch.equal(s["depth"], a["depth"][5:9])
    # permuting the face order permutes face indices but cannot change depth or coverage
    perm = np.random.default_rng(0).permutation(faces.shape[1])
    pm = _run_product(np.ascontiguousarray(faces[:4, perm]), None, 256, False, 0.1, 100, 1e-4, bg, (0, 1, 1))
    assert torch.equal(pm["depth"], a["depth"][:4]) and torch.equal(pm["alpha"], a["alpha"][:4])
    inv = torch.from_numpy(perm).cuda()
    same = pm["fim"] >= 0
    assert torch.equal(inv[pm["fim"][same].long()], a["fim"][:4][same].long())


def test_headline_gradient_checksums(headline):
    faces, tex = headline
    fwd = _run_product(faces, tex, 256, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 0, 0))
    grads = _grads(fwd, seed=99)
    out = _run_product(faces, tex, 256, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 0, 0), grads)
    covered = (out["fim"] >= 0)[:, None].float()
    # trilinear weights sum to 1: per item and channel, sum of texture gradients == sum of upstream grads on covered pixels
    lhs = out["grad_tex"].sum(dim=(1, 2, 3, 4)).double()
    rhs = (grads["rgb"] * covered).sum(dim=(2, 3)).double()
    assert rel_err(np_(lhs), np_(rhs)) <= 1e-4
    # backward is linear in the upstream gradient for textures
    out2 = _run_product(faces, tex, 256, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 0, 0), {"rgb": grads["rgb"] * 2})
    assert rel_err(np_(out2["grad_tex"]), np_(out["grad_tex"] * 2)) <= 1e-5
    # edge gradients never touch z (K5 writes x, y only; no depth output requested)
    assert torch.all(out["grad_faces"][..., 2] == 0)
    assert torch.isfinite(out["grad_faces"]).all()


def test_headline_vs_reference_kernels(headline):
    faces, tex = headline
    B = 8  # the brute-force reference needs ~B * 3.3e8 face tests
    args = (faces[:B], tex[:B], 256, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 0, 0))
    gold = RefGolden("parity_headline8")
    ref = _reference(gold, *args)
    grads = _grads(_run_product(*args), seed=99)
    _record_backward(gold, ref, grads, (1, 0, 0))
    got = _run_product(*args, grads)
    assert gold.equal("fim", got["fim"].flip(1))
    assert gold.equal("rgb", got["rgb"])  # bit-exact, as at every anti-aliasing-off shape
    _compare_backward(gold, got, (1, 0, 0))


def test_vertices_to_faces_kernels(teapot):
    """Fused gather / scatter-add (nr_b200_vertices_to_faces*) against plain torch indexing (vertices_to_faces.py:16-21)."""
    import neural_renderer as nr
    dev = torch.device("cuda")
    v, f = teapot
    B = 3
    vert = torch.from_numpy(np.stack([v * (1 + 0.1 * i) for i in range(B)])).to(dev).requires_grad_(True)
    faces = torch.from_numpy(np.stack([f] * B)).to(dev)
    out = nr.vertices_to_faces(vert, faces)
    idx = faces.long() + (torch.arange(B, device=dev) * v.shape[0])[:, None, None]
    ref_in = vert.detach().clone().requires_grad_(True)
    ref = ref_in.reshape(-1, 3)[idx]
    assert torch.equal(out, ref)
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(4)).to(dev)
    (out * g).sum().backward()
    (ref * g).sum().backward()
    assert rel_err(np_(vert.grad), np_(ref_in.grad)) <= 1e-5


def test_cuda_graph_capture_and_side_stream():
    """The C ABI only enqueues work on the caller's stream (no hidden allocation or synchronisation), so a forward +
    backward pass can run on a side stream and be captured in a CUDA graph and replayed."""
    import neural_renderer as nr
    faces_np, tex_np = _inputs("sphere", 2, 200, 2, seed=5)
    dev = torch.device("cuda")
    faces = torch.from_numpy(faces_np).to(dev).requires_grad_(True)
    tex = torch.from_numpy(tex_np).to(dev).requires_grad_(True)
    g = torch.randn((2, 3, 64, 64), generator=torch.Generator().manual_seed(1)).to(dev)

    def step():
        faces.grad = None
        tex.grad = None
        img = nr.rasterize(faces, tex, 64, False)
        img.backward(g)
        return img.detach().clone(), faces.grad.clone(), tex.grad.clone()

    ref = step()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):  # warm-up on the side stream (allocator, autograd engine)
            on_side = step()
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(on_side[0], ref[0]) and rel_err(np_(on_side[1]), np_(ref[1])) <= 1e-5
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    for t in out:
        t.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], ref[0])
    assert rel_err(np_(out[1]), np_(ref[1])) <= 1e-5 and rel_err(np_(out[2]), np_(ref[2])) <= 1e-5


def test_examples_optimise():
    """The reference's example 2 / 3 / 4 call sequences (torch instead of Chainer) make progress end to end."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for name, iters in (("example2_optimize_vertices", 30), ("example3_optimize_textures", 15)):
        spec = importlib.util.spec_from_file_location(name, os.path.join(root, "examples", name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        losses = mod.run(iters)
        assert np.isfinite(losses).all() and losses[-1] < 0.8 * losses[0], (name, losses[0], losses[-1])
    # example 4: the camera position is the parameter (gradients through the fused camera kernel)
    spec = importlib.util.spec_from_file_location("example4", os.path.join(root, "examples", "example4_optimize_camera.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    losses, eye = mod.run(150)
    assert np.isfinite(losses).all() and np.isfinite(eye).all()
    assert min(losses) < 0.9 * losses[0], (losses[0], min(losses))


def test_edge_cases():
    """Empty / degenerate inputs the reference's tests exercise implicitly (all-zero batch slots of to_minibatch),
    single face, faces entirely off screen, rgb + per-batch background."""
    import neural_renderer as nr
    dev = torch.device("cuda")
    z = torch.zeros((2, 5, 3, 3), device=dev)
    assert nr.rasterize_silhouettes(z, 32, False).abs().sum().item() == 0
    d = nr.rasterize_depth(z, 32, True)
    assert torch.all(d == 100)
    off = torch.tensor([[[[3.0, 3.0, 1.0], [4.0, 3.0, 1.0], [3.0, 4.0, 1.0]]]], device=dev)
    assert nr.rasterize_silhouettes(off, 16, False).sum().item() == 0
    tri = torch.tensor([[[[-0.5, -0.5, 1.0], [0.5, -0.5, 1.0], [0.0, 0.6, 1.0]]]], device=dev)
    a = nr.rasterize_silhouettes(tri, 16, False)
    b = nr.rasterize_silhouettes(tri.flip(2), 16, False)  # one winding is back-facing
    assert (a.sum().item() > 0) != (b.sum().item() > 0)
    nan = tri.clone()
    nan[0, 0, 0, 0] = float("nan")
    assert nr.rasterize_silhouettes(nan, 16, False).sum().item() == 0  # NaN vertices never win a pixel
