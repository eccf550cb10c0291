"""GPU parity tests at the shapes BASELINE.json names (configs[0..4]) and the headline's other output modes, against the
reference's own kernels (oracle/refhost.py over oracle/_ref/*.so, built by oracle/build_ref.py from the reference's
source tree), through the digests of their results stored under tests/golden/ref (tests/refgolden.py).

  configs[0]  teapot silhouette 64x64 (anti-aliased -> raster 128), batch 1      reference tests/test_rasterize_silhouettes.py:15-35
  configs[1]  teapot RGB 256x256 batch 8 fwd+bwd                                 -> tests/test_gpu_parity.py::test_teapot_renderer_defaults_vs_reference_kernels
  configs[2]  ~70k faces, depth + RGB, 512x512                                   forward on 2 items, backward on 1 item
  configs[3]  headline, all 64 items, plus its silhouette / depth / ts=2 variants
  configs[4]  one shared mesh, many viewpoints: reduced size vs the reference kernels (100k faces, 512^2, 2 views) and
              size-independent properties at the full 1M faces / 1024^2 (22-bit face field of the z-key, 32-bit strip
              list offsets of the backward binning).

Tolerances (BASELINE.json north_star): face_index_map bit-exact; images / gradients <= 1e-4 relative
(max-abs-error / max-abs-reference per tensor); K5 (edge-scan gradient) additionally per element, see
test_edge_scan_per_element.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-4

from helpers import np_, rel_err  # noqa: E402
from refgolden import RefGolden  # noqa: E402
from test_gpu_parity import (_compare_backward, _compare_forward, _grads, _record_backward, _reference,  # noqa: E402
                             _run_product)


@pytest.fixture(scope="module", autouse=True)
def _gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from neural_renderer_b200 import _lib
    _lib.load()
    yield


# ----------------------------------------------------------------------------------------------------- configs[0]
def test_config0_teapot_silhouette_64_aa(teapot):
    """BASELINE configs[0]: teapot silhouette at 64x64 (anti-aliased: raster 128), batch 1, through Renderer."""
    import neural_renderer as nr
    dev = torch.device("cuda")
    v, f = teapot
    vertices = torch.from_numpy(v[None]).to(dev).requires_grad_(True)
    faces_idx = torch.from_numpy(f[None]).to(dev)
    r = nr.Renderer()
    r.image_size = 64
    img = r.render_silhouettes(vertices, faces_idx)
    assert img.shape == (1, 64, 64)
    # the rasterizer inputs exactly as Renderer.render_silhouettes builds them (renderer.py:41-52)
    fi = torch.cat((faces_idx, faces_idx.flip(2)), dim=1)
    faces = nr.vertices_to_faces(nr.perspective(nr.look_at(vertices.detach(), r.eye)), fi).contiguous()
    args = (np_(faces), None, 64, True, 0.1, 100, 1e-4, (0, 0, 0), (0, 1, 0))
    gold = RefGolden("configs_config0")
    ref = _reference(gold, *args)
    assert gold.rel_err("alpha", img) <= TOL
    grads = _grads(_run_product(*args), seed=3)
    _record_backward(gold, ref, grads, (0, 1, 0))
    got = _run_product(*args, grads)
    _compare_forward(gold, got, True)
    _compare_backward(gold, got, (0, 1, 0))


# ----------------------------------------------------------------------------------------------------- configs[2]
def test_config2_70k_faces_depth_rgb_512():
    """BASELINE configs[2] (bunny-scale): 70k faces, depth + RGB, 512x512 -- forward on 2 items, backward on 1."""
    from neural_renderer_b200 import synthetic
    flags = (1, 0, 1)
    faces = synthetic.sphere_faces(2, 70000, seed=77)
    tex = synthetic.random_textures(2, 70000, 2, seed=78)
    gold = RefGolden("configs_config2_forward")
    _reference(gold, faces, tex, 512, False, 0.1, 100, 1e-4, (0.2, 0.3, 0.4), flags)
    gold.save()
    got = _run_product(faces, tex, 512, False, 0.1, 100, 1e-4, (0.2, 0.3, 0.4), flags)
    _compare_forward(gold, got, False)
    assert int(got["fim"].max().item()) > 60000  # high face indices do win pixels
    args1 = (faces[:1], tex[:1], 512, False, 0.1, 100, 1e-4, (0.2, 0.3, 0.4), flags)
    gold1 = RefGolden("configs_config2_item0")
    ref1 = _reference(gold1, *args1)
    grads = _grads(_run_product(*args1), seed=5)
    _record_backward(gold1, ref1, grads, flags)
    got1 = _run_product(*args1, grads)
    _compare_forward(gold1, got1, False)
    _compare_backward(gold1, got1, flags)


# ------------------------------------------------------------------------------------- configs[3]: headline shapes
@pytest.fixture(scope="module")
def headline64():
    from neural_renderer_b200 import synthetic
    return synthetic.sphere_faces(64, 5000), synthetic.random_textures(64, 5000, 4), synthetic.random_textures(64, 5000, 2, seed=5)


@pytest.mark.parametrize("mode", ["rgb_ts4", "rgb_ts2", "silhouette", "depth"])
def test_headline_all_64_items_vs_reference_kernels(headline64, mode):
    """The BASELINE metric's shape (256x256, 5000 faces, batch 64), every item, every output mode, fwd + bwd."""
    faces, tex4, tex2 = headline64
    flags, tex = {"rgb_ts4": ((1, 0, 0), tex4), "rgb_ts2": ((1, 0, 0), tex2), "silhouette": ((0, 1, 0), None),
                  "depth": ((0, 0, 1), None)}[mode]
    args = (faces, tex, 256, False, 0.1, 100, 1e-4, (0, 0, 0), flags)
    gold = RefGolden("configs_headline64_" + mode)
    ref = _reference(gold, *args)
    grads = _grads(_run_product(*args), seed=99)
    _record_backward(gold, ref, grads, flags)
    got = _run_product(*args, grads)
    _compare_forward(gold, got, False)
    _compare_backward(gold, got, flags)


def test_reference_digests_catch_a_single_face_gradient_error(headline64):
    """The large gradient tensors are compared through signed block sums and their largest elements
    (tests/refgolden.py), not element by element.  Mutation check at the headline shape: the product's gradients pass,
    and the same gradients with ONE face's gradient (one batch item, one face; faces or texture cube) scaled by 1.5
    fail -- for randomly drawn faces whose error a full-tensor comparison would see (above 2 x TOL of the tensor
    maximum) -- as do the same gradients with one NaN."""
    faces, tex4, _ = headline64
    args = (faces, tex4, 256, False, 0.1, 100, 1e-4, (0, 0, 0), (1, 0, 0))
    gold = RefGolden("configs_headline64_rgb_ts4")
    if gold.recording:
        pytest.skip("compares with the stored digests")
    got = _run_product(*args, _grads(_run_product(*args), seed=99))
    rng = np.random.default_rng(2024)
    for name, key, tries in (("grad_faces", "grad_faces", 24), ("grad_tex", "grad_tex", 8)):
        g = np_(got[key])
        assert gold.rel_err(name, g) <= TOL, name
        per_face = np.abs(g.reshape(g.shape[0] * g.shape[1], -1)).max(1)
        seen = np.flatnonzero(0.5 * per_face > 2 * TOL * gold.absmax(name))
        assert seen.size > 1000, (name, seen.size)
        for k in rng.choice(seen, tries, replace=False):
            b, f = divmod(int(k), g.shape[1])
            keep = g[b, f].copy()
            g[b, f] *= 1.5
            assert gold.rel_err(name, g) > TOL, (name, b, f)
            g[b, f] = keep
        # a NaN anywhere (here away from the stored largest elements) fails the comparison as well
        k = int(rng.choice(np.flatnonzero(per_face == 0)))
        b, f = divmod(k, g.shape[1])
        g[b, f].flat[0] = np.nan
        assert not gold.rel_err(name, g) <= TOL, (name, "NaN", b, f)
        g[b, f] = 0


# ----------------------------------------------------------------------------------------------------- configs[4]
def _shared_mesh_views(F, V, dev, scale=0.55):
    """One mesh seen from V viewpoints, prepared as Renderer.render does (no fill_back): faces [V,F,3,3]."""
    import neural_renderer as nr
    from neural_renderer_b200 import synthetic
    v_np, f_np = synthetic.sphere_mesh(F)
    vertices = torch.from_numpy((v_np * scale).astype(np.float32)).to(dev)
    faces_idx = torch.from_numpy(f_np).to(dev)
    az = torch.arange(V, dtype=torch.float32) * (360.0 / V) + 10.0
    eyes = nr.get_points_from_angles(torch.full_like(az, 2.732), torch.full_like(az, 30.0), az).to(dev)
    vv = nr.perspective(nr.look_at(vertices[None].expand(V, -1, -1), eyes))
    return nr.vertices_to_faces(vv, faces_idx[None].expand(V, -1, -1)).contiguous(), vertices, faces_idx, eyes


def test_config4_reduced_shared_mesh_vs_reference_kernels():
    """configs[4] at reduced size: one 100k-face mesh, 2 viewpoints, 512x512, RGB (eps 1e-3 as Renderer.render passes),
    forward + backward vs the reference kernels; the per-view face gradients summed over the views are what
    Mesh.get_batch's broadcast backward (mesh.py:29-34) hands to the shared parameters."""
    flags = (1, 0, 0)
    F, V, S, ts = 100000, 2, 512, 2
    dev = torch.device("cuda")
    faces, _, _, _ = _shared_mesh_views(F, V, dev)
    tex = torch.rand((1, F, ts, ts, ts, 3), generator=torch.Generator().manual_seed(7)).to(dev).expand(V, -1, -1, -1, -1, -1).contiguous()
    args = (np_(faces), np_(tex), S, False, 0.1, 100, 1e-3, (0, 0, 0), flags)
    gold = RefGolden("configs_config4_reduced")
    ref = _reference(gold, *args)
    grads = _grads(_run_product(*args), seed=11)
    if gold.recording:
        gf, gt = ref.backward(grads["rgb"], None, None)
        gold.put("grad_tex_sum", gt.sum(0))
        gold.put("grad_faces_sum", gf.sum(0))
    _record_backward(gold, ref, grads, flags)
    got = _run_product(*args, grads)
    _compare_forward(gold, got, False)
    _compare_backward(gold, got, flags)
    assert int(got["fim"].max().item()) > 60000  # (the camera looks down from 30 degrees: the lowest rings are hidden)
    # shared-parameter gradients = sum over the views
    assert gold.rel_err("grad_tex_sum", got["grad_tex"].sum(0)) <= TOL
    assert gold.rel_err("grad_faces_sum", got["grad_faces"].sum(0)) <= TOL


def test_config4_full_size_properties():
    """configs[4] at full size per GPU share: 1M faces, 1024x1024, 2 of the viewpoints.  No brute-force oracle can run
    here (2e12 face tests per view), so size-independent properties: determinism, alpha == coverage, uncovered depth,
    face indices above 2^19 win pixels, face-order invariance (reversed face order -> same depth / coverage, mapped
    indices), texture-gradient checksum, finite vertex gradients, batch independence."""
    dev = torch.device("cuda")
    F, V, S, ts = 1000000, 2, 1024, 2
    faces_t, _, _, _ = _shared_mesh_views(F, V, dev)
    faces = np_(faces_t)
    del faces_t
    tex = np.random.default_rng(3).random((1, F, ts, ts, ts, 3), dtype=np.float32).repeat(V, axis=0)
    bg = (0.1, 0.2, 0.3)
    a = _run_product(faces, tex, S, False, 0.1, 100, 1e-3, bg, (1, 1, 1))
    grads = _grads(a, seed=5)
    b = _run_product(faces, tex, S, False, 0.1, 100, 1e-3, bg, (1, 1, 1), {"rgb": grads["rgb"], "alpha": grads["alpha"]})
    for k in ("fim", "rgb", "alpha", "depth", "wmap"):
        assert torch.equal(a[k], b[k]), k
    covered = a["fim"] >= 0
    assert 0.05 < covered.float().mean().item() < 0.9
    assert torch.equal(a["alpha"], covered.float())
    assert torch.all(a["depth"][~covered] == 100.0)
    assert int(a["fim"].max().item()) >= (1 << 19) and int(a["fim"].max().item()) < F
    w = a["wmap"]
    assert torch.allclose(w.sum(1)[covered], torch.ones((), device=dev), atol=1e-5)
    # reversed face order: indices map through the permutation, depth and coverage cannot change
    rev = _run_product(np.ascontiguousarray(faces[:1, ::-1]), None, S, False, 0.1, 100, 1e-3, bg, (0, 1, 1))
    assert torch.equal(rev["depth"], a["depth"][:1]) and torch.equal(rev["alpha"], a["alpha"][:1])
    m = rev["fim"] >= 0
    assert torch.equal((F - 1 - rev["fim"][m]), a["fim"][:1][m])
    # batch independence (alpha / depth / fim; rgb is excluded because of the batch-0 quirk of the sampler)
    one = _run_product(faces[1:2], None, S, False, 0.1, 100, 1e-3, bg, (0, 1, 1))
    assert torch.equal(one["fim"], a["fim"][1:2]) and torch.equal(one["depth"], a["depth"][1:2])
    # backward: trilinear weights sum to 1 -> per view and channel, sum of texture gradients == sum of upstream
    # gradients over covered pixels; vertex gradients finite and x/y only
    lhs = b["grad_tex"].sum(dim=(1, 2, 3, 4)).double()
    rhs = (grads["rgb"] * covered[:, None].float()).sum(dim=(2, 3)).double()
    assert rel_err(np_(lhs), np_(rhs)) <= 1e-4
    assert torch.isfinite(b["grad_faces"]).all()
    assert torch.all(b["grad_faces"][..., 2] == 0)
    assert float(b["grad_faces"].abs().max()) > 0
    # the edge-scan gradient of view 1 rendered alone equals its rows in the 2-view batch (strip lists of different
    # items never mix; fp32 atomics reorder sums, hence the tolerance)
    one_b = _run_product(faces[1:2], None, S, False, 0.1, 100, 1e-3, bg, (0, 1, 0), {"alpha": grads["alpha"][1:2]})
    two_b = _run_product(faces, None, S, False, 0.1, 100, 1e-3, bg, (0, 1, 0), {"alpha": grads["alpha"]})
    assert rel_err(np_(one_b["grad_faces"][0]), np_(two_b["grad_faces"][1])) <= 1e-5


# -------------------------------------------------------------------------- K5 (edge scan) beyond the per-tensor norm
@pytest.mark.parametrize("case", ["soup64", "sphere192", "headline8"])
def test_edge_scan_per_element(case, capsys):
    """grad_faces per element (components above 1e-3 of the tensor maximum) vs the reference's deterministic K5
    (rasterize.py:528-748, plain store :736), plus the run-to-run spread of this implementation's fp32 atomics.
    The per-tensor norm of the other tests hides relative error on small components; this one does not.  Every such
    component is compared for soup64 and sphere192; for headline8 (about 10^5 of them) a fixed sample of 2048 is
    (tests/refgolden.py), beside the per-tensor comparison of the whole tensor."""
    from neural_renderer_b200 import synthetic
    if case == "soup64":
        S, F, ts, B, flags = 64, 200, 4, 4, (1, 1, 1)
        faces, tex = synthetic.triangle_soup(B, F, seed=31), synthetic.random_textures(B, F, ts, seed=32)
    elif case == "sphere192":
        S, F, ts, B, flags = 192, 2000, 2, 2, (1, 1, 0)
        faces, tex = synthetic.sphere_faces(B, F, seed=33), synthetic.random_textures(B, F, ts, seed=34)
    else:
        S, F, ts, B, flags = 256, 5000, 4, 8, (1, 0, 0)
        faces, tex = synthetic.sphere_faces(B, F), synthetic.random_textures(B, F, ts)
    args = (faces, tex, S, False, 0.1, 100, 1e-4, (0.1, 0.2, 0.3), flags)
    gold = RefGolden("configs_edge_scan_" + case)
    ref = _reference(gold, *args)
    g = _grads(_run_product(*args), seed=17)
    g.pop("depth", None)  # K5 only (the depth term is K7's)
    if gold.recording:
        gold.put("grad_faces", ref.backward(g.get("rgb"), g.get("alpha"), None)[0], per_element=True)
        gold.save()
    runs = [np_(_run_product(*args, g)["grad_faces"]) for _ in range(3)]
    err, n = gold.per_element("grad_faces", runs[0])
    per_tensor = gold.rel_err("grad_faces", runs[0])
    spread = max(rel_err(r, runs[0]) for r in runs[1:])
    with capsys.disabled():
        print("\n[K5 %s] per-element max rel err %.3g over %d compared components (> 1e-3 of max); per-tensor %.3g; "
              "run-to-run spread %.3g of max" % (case, err, n, per_tensor, spread))
    assert per_tensor <= TOL, per_tensor
    assert err <= 2e-3, err
    assert spread <= 1e-5, spread


def test_edge_scan_sparse_gradient_vs_reference_kernels():
    """Single-pixel losses (like the reference's known-answer tests, test_rasterize_silhouettes.py:39-83): the upstream
    gradient is non-zero at a handful of pixels only, so every surviving term of K5 is visible on its own."""
    from neural_renderer_b200 import synthetic
    S, F, ts, B, flags = 64, 200, 4, 4, (1, 1, 1)
    dev = torch.device("cuda")
    faces, tex = synthetic.triangle_soup(B, F, seed=41), synthetic.random_textures(B, F, ts, seed=42)
    gold = RefGolden("configs_edge_scan_sparse")
    ref = _reference(gold, faces, tex, S, False, 0.1, 100, 1e-4, (0.5, 0.5, 0.5), flags)
    rng = np.random.default_rng(43)
    for trial in range(6):
        g_rgb = torch.zeros((B, 3, S, S), device=dev)
        g_alpha = torch.zeros((B, S, S), device=dev)
        for _ in range(3):
            b, y, x = int(rng.integers(B)), int(rng.integers(S)), int(rng.integers(S))
            g_rgb[b, :, y, x] = torch.from_numpy(rng.normal(size=3).astype(np.float32)).to(dev)
            g_alpha[b, y, x] = float(rng.normal())
        gf_name, gt_name = "grad_faces%d" % trial, "grad_tex%d" % trial
        if gold.recording:
            gf_ref, gt_ref = ref.backward(g_rgb, g_alpha, None)
            gold.put(gf_name, gf_ref, whole=True)
            gold.put(gt_name, gt_ref, whole=True)
        got = _run_product(faces, tex, S, False, 0.1, 100, 1e-4, (0.5, 0.5, 0.5), flags, {"rgb": g_rgb, "alpha": g_alpha})
        gf_ref, gt_ref = gold.dense(gf_name), gold.dense(gt_name)
        if float(np.abs(gf_ref).max()) == 0.0:
            assert float(got["grad_faces"].abs().max()) == 0.0
            continue
        assert rel_err(np_(got["grad_faces"]), gf_ref) <= TOL
        err, _ = gold.per_element(gf_name, got["grad_faces"])
        assert err <= 1e-3, (trial, err)
        # components the reference leaves at exactly zero stay (numerically) zero: the discrete decisions of K5 --
        # crossing pixels, face_index_map gates, scan limits -- are reproduced exactly; only a diff_grad that is an
        # exact 0 in the reference's (I - ref) * g form may round to +-1e-8 in the A - ref * g form used here
        zero = torch.from_numpy(gf_ref == 0).to(dev)
        assert float(got["grad_faces"][zero].abs().max()) <= 1e-6 * float(np.abs(gf_ref).max())
        assert rel_err(np_(got["grad_tex"]), gt_ref) <= TOL
    gold.save()
