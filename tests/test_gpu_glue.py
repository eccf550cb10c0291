"""GPU tests of the rows either side of the rasterizer (SURVEY.md section 8(f)): fused camera pipeline and lighting /
fill_back folded into the sampler, each against the op-by-op formulation of the reference."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from neural_renderer_b200 import _lib
    _lib.load()  # fail loudly if the CUDA library is missing on a GPU box
    yield


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _cpu64(fn, vertices, *args, **kw):
    """Run a glue function op by op on the CPU in float64 (the non-CUDA branch is the reference's formulation)."""
    v = vertices.detach().cpu().double().requires_grad_(True)
    return v, fn(v, *args, **kw)


@pytest.mark.parametrize("mode", ["look_at", "look", "none"])
@pytest.mark.parametrize("persp", [True, False])
def test_camera_transform_vs_op_by_op(mode, persp):
    from neural_renderer_b200 import functional as F
    if mode == "none" and not persp:
        pytest.skip("identity")
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(5)
    v = (torch.rand((3, 700, 3), generator=gen) - 0.5)
    eye = [0.3, 1.1, -2.6]
    direction = [0.1, -0.2, 1.0]
    g = torch.randn((3, 700, 3), generator=gen)
    vc, ref = _cpu64(F.camera_transform, v, eye, mode, direction, persp, 30.)
    (ref * g.double()).sum().backward()
    vg = v.to(dev).requires_grad_(True)
    out = F.camera_transform(vg, eye, mode, direction, persp, 30.)
    (out * g.to(dev)).sum().backward()
    assert rel_err(out.detach().cpu(), ref.detach()) <= 2e-6
    assert rel_err(vg.grad.cpu(), vc.grad) <= 2e-5


def test_camera_gradients_reach_the_eye():
    """examples/example4.py optimises the camera position: the fused backward must deliver d loss / d eye (through
    the translation and through the look_at rotation) -- also with one eye per batch item."""
    from neural_renderer_b200 import functional as F
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(6)
    v = (torch.rand((4, 300, 3), generator=gen) - 0.5)
    g = torch.randn((4, 300, 3), generator=gen)
    for eye0 in (torch.tensor([0.5, 0.8, -2.5]), torch.tensor([[0.5, 0.8, -2.5], [0, 0, -3.0], [1, 1, -2], [-1, 0.3, -2.2]])):
        e_ref = eye0.double().requires_grad_(True)
        ref = F.perspective(F.look_at(v.double(), e_ref), 30.)
        (ref * g.double()).sum().backward()
        e = eye0.to(dev).requires_grad_(True)
        out = F.perspective(F.look_at(v.to(dev), e), 30.)       # two kernels
        (out * g.to(dev)).sum().backward()
        assert rel_err(out.detach().cpu(), ref.detach()) <= 2e-6
        assert rel_err(e.grad.cpu(), e_ref.grad) <= 1e-4
        e2 = eye0.to(dev).requires_grad_(True)
        out2 = F.camera_transform(v.to(dev), e2, "look_at", None, True, 30.)  # one kernel
        (out2 * g.to(dev)).sum().backward()
        assert rel_err(out2.detach().cpu(), ref.detach()) <= 2e-6
        assert rel_err(e2.grad.cpu(), e_ref.grad) <= 1e-4


def test_viewing_angle_gradient():
    from neural_renderer_b200 import functional as F
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(7)
    v = torch.rand((2, 100, 3), generator=gen) + torch.tensor([0.0, 0.0, 2.0])
    g = torch.randn((2, 100, 3), generator=gen)
    a_ref = torch.tensor([25.0, 40.0], dtype=torch.float64, requires_grad=True)
    (F.perspective(v.double(), a_ref) * g.double()).sum().backward()
    a = torch.tensor([25.0, 40.0], device=dev, requires_grad=True)
    (F.perspective(v.to(dev), a) * g.to(dev)).sum().backward()
    assert rel_err(a.grad.cpu(), a_ref.grad) <= 1e-4


@pytest.mark.parametrize("fill_back", [True, False])
def test_renderer_fused_lighting_matches_materialised(teapot, fill_back):
    """Renderer.render with lighting / fill_back folded into the sampler == the op-by-op pipeline that materialises
    `textures * light` and the doubled texture tensor: identical pixels, same gradients."""
    import neural_renderer as nr
    dev = torch.device("cuda")
    v, f = teapot
    B = 2
    rot = torch.tensor([[0.9, 0.0, 0.43], [0.0, 1.0, 0.0], [-0.43, 0.0, 0.9]])
    vertices = torch.from_numpy(np.stack([v, v @ rot.numpy().T.astype(np.float32)])).to(dev)
    faces_idx = torch.from_numpy(np.stack([f, f])).to(dev)
    tex = torch.rand((B, f.shape[0], 4, 4, 4, 3), generator=torch.Generator().manual_seed(1)).to(dev)
    g = torch.randn((B, 3, 128, 128), generator=torch.Generator().manual_seed(2)).to(dev)
    results = []
    for fused in (False, True):
        r = nr.Renderer()
        r.image_size = 128
        r.fill_back = fill_back
        r.fused = fused
        r.eye = nr.get_points_from_angles(2.732, 30, 40)
        r.light_direction = [0.3, 1.0, -0.2]
        r.light_color_directional = [1.0, 0.8, 0.6]
        va = vertices.clone().requires_grad_(True)
        ta = tex.clone().requires_grad_(True)
        img = r.render(va, faces_idx, ta)
        (img * g).sum().backward()
        results.append((img.detach(), va.grad, ta.grad))
    (img0, gv0, gt0), (img1, gv1, gt1) = results
    assert rel_err(img1.cpu(), img0.cpu()) <= 1e-6  # the light factors differ by fp32 rounding (fused normalisation)
    assert rel_err(gt1.cpu(), gt0.cpu()) <= 1e-5
    assert rel_err(gv1.cpu(), gv0.cpu()) <= 1e-4


def test_face_light_and_fill_back_vs_reference_kernels():
    """rasterize(face_light=..., textures_fill_back=True) against the reference's own kernels fed the materialised
    tensors (bit-exact colours; texture / light gradients through the chain rule of the materialisation)."""
    import neural_renderer as nr
    from neural_renderer_b200 import synthetic
    from refgolden import RefGolden
    from test_gpu_parity import _reference
    dev = torch.device("cuda")
    B, F2 = 3, 100
    half = synthetic.triangle_soup(B, F2, seed=11)
    faces = torch.from_numpy(np.concatenate([half, half[:, :, ::-1].copy()], axis=1)).to(dev)  # reversed copies
    tex = torch.from_numpy(synthetic.random_textures(B, F2, 4, seed=12)).to(dev)
    light = (torch.rand((B, 2 * F2, 3), generator=torch.Generator().manual_seed(13)) * 1.5).to(dev)
    g = torch.randn((B, 3, 64, 64), generator=torch.Generator().manual_seed(14)).to(dev)
    gold = RefGolden("glue_face_light_fill_back")
    if gold.recording:
        tex_a = tex.clone().requires_grad_(True)
        light_a = light.clone().requires_grad_(True)
        full = torch.cat((tex_a, tex_a.permute(0, 1, 4, 3, 2, 5)), dim=1) * light_a[:, :, None, None, None, :]
        ref = _reference(gold, faces, full.detach().contiguous(), 64, False, 0.1, 100, 1e-4, [0.1, 0.2, 0.3], (1, 0, 0))
        gf_ref, gfull_ref = ref.backward(g, None, None)
        full.backward(gfull_ref)
        gold.put("grad_faces", gf_ref)
        gold.put("grad_tex", tex_a.grad)
        gold.put("grad_light", light_a.grad)
        gold.save()
    fa = faces.clone().requires_grad_(True)
    tb = tex.clone().requires_grad_(True)
    lb = light.clone().requires_grad_(True)
    img = nr.rasterize(fa, tb, 64, False, 0.1, 100, 1e-4, [0.1, 0.2, 0.3], face_light=lb, textures_fill_back=True)
    (img * g).sum().backward()
    assert gold.equal("rgb", img)
    assert gold.rel_err("grad_faces", fa.grad) <= 1e-4
    assert gold.rel_err("grad_tex", tb.grad) <= 1e-5
    assert gold.rel_err("grad_light", lb.grad) <= 1e-5


def test_face_lighting_kernels(teapot):
    """nr_b200_face_lighting* against lighting.py's op-by-op formulation (float64 on the CPU), values and gradients."""
    from neural_renderer_b200 import functional as F
    dev = torch.device("cuda")
    v, f = teapot
    vertices = torch.from_numpy(np.stack([v, v[:, [2, 0, 1]].copy()]))
    faces = torch.from_numpy(np.stack([f, f]))
    faces = torch.cat((faces, faces.flip(2)), dim=1)
    g = torch.randn((2, faces.shape[1], 3), generator=torch.Generator().manual_seed(3))
    args = (0.3, 0.7, [1.0, 0.9, 0.8], [0.5, 1.0, 0.25], [0.2, 0.9, -0.4])
    v_ref = vertices.double().requires_grad_(True)
    ref = F.face_light(F.vertices_to_faces(v_ref, faces), *args)
    (ref * g.double()).sum().backward()
    v_gpu = vertices.to(dev).requires_grad_(True)
    out = F.face_light_from_vertices(v_gpu, faces.to(dev), *args)
    (out * g.to(dev)).sum().backward()
    assert rel_err(out.detach().cpu(), ref.detach()) <= 2e-6
    assert rel_err(v_gpu.grad.cpu(), v_ref.grad) <= 1e-4


def test_renderer_step_in_cuda_graph(teapot):
    """A whole Renderer.render forward + backward (camera, lighting, gather, rasterizer and their backward kernels)
    only enqueues work on the current stream: it can be captured once and replayed."""
    import neural_renderer as nr
    dev = torch.device("cuda")
    v, f = teapot
    vertices = torch.from_numpy(np.stack([v, v])).to(dev).requires_grad_(True)
    faces_idx = torch.from_numpy(np.stack([f, f])).to(dev)
    tex = torch.rand((2, f.shape[0], 2, 2, 2, 3), generator=torch.Generator().manual_seed(1)).to(dev).requires_grad_(True)
    g = torch.randn((2, 3, 64, 64), generator=torch.Generator().manual_seed(2)).to(dev)
    r = nr.Renderer()
    r.image_size = 64
    r.eye = nr.get_points_from_angles(2.732, 30, 40)

    def step():
        vertices.grad = None
        tex.grad = None
        img = r.render(vertices, faces_idx, tex)
        img.backward(g)
        return img.detach().clone(), vertices.grad.clone(), tex.grad.clone()

    ref = step()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    for t in out:
        t.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], ref[0])
    assert rel_err(out[1].cpu(), ref[1].cpu()) <= 1e-4 and rel_err(out[2].cpu(), ref[2].cpu()) <= 1e-5


def _bake_inputs(ts, H, W, F, seed):
    rng = np.random.default_rng(seed)
    img = rng.random((H, W, 3), dtype=np.float32)
    uv = rng.random((F, 3, 2), dtype=np.float32)
    uv[0] = [[0, 0], [1, 0], [1, 1]]        # exact corners: the one-past-the-edge taps of the reference
    uv[1] = [[1, 1], [0, 1], [1, 0]]
    upd = (rng.random(F) < 0.7).astype(np.int32)
    upd[:2] = 1
    tex = rng.random((F, ts, ts, ts, 3), dtype=np.float32)
    return img, uv, upd, tex


@pytest.mark.parametrize("cfg", [(4, 64, 48), (2, 64, 48), (6, 33, 57)])
def test_bake_textures_kernel_bit_exact(cfg):
    """nr_b200_bake_textures == the C oracle == the reference's own kernel string (load_obj.py:88-137), bit for bit,
    NaN texels included."""
    import nr_oracle as o
    from neural_renderer_b200 import io
    from refgolden import RefGolden
    ts, H, W = cfg
    img, uv, upd, tex = _bake_inputs(ts, H, W, 301, seed=ts * 100 + H)
    got = io.bake_textures(img, uv, upd, ts, tex)
    want = o.bake_textures(img, uv, upd, ts, tex.copy())
    # NaN payloads differ between x86 and the GPU; every other value must match bit for bit
    assert ((got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want))).all()
    assert np.isnan(got).sum() == 3 * int(upd.sum())
    assert np.array_equal(got[upd == 0], tex[upd == 0])
    # faces 0 and 1 have UVs of exactly 1: there the reference kernel reads one row past the image -- with weight
    # 0, or, when (int)(pos_y + 1) rounds up past (int)pos_y + 1, with weight ~1 (undefined in the reference); the
    # product addresses those taps inside the image, so only the in-bounds faces are compared
    gold = RefGolden("glue_bake_ts%d_%dx%d" % cfg)
    if gold.recording:
        import refbake
        assert refbake.available(ts, H, W), "reference bake kernel not built (oracle/build_ref.py)"
        dev = torch.device("cuda")
        ref = refbake.bake(torch.from_numpy(img).to(dev), torch.from_numpy(uv).to(dev), torch.from_numpy(upd).to(dev), ts,
                           torch.from_numpy(tex).to(dev)).cpu().numpy()
        gold.put("textures_in_bounds", ref[2:], exact_only=True)
        gold.save()
    assert gold.equal("textures_in_bounds", got[2:])  # bit for bit, every NaN texel read as one NaN


def test_load_obj_with_textures_and_render():
    """examples 1 / 4 call sequence on a textured OBJ: load_obj(load_texture=True) -> Renderer.render."""
    import os
    import neural_renderer as nr
    import nr_oracle as o
    from neural_renderer_b200 import io
    obj = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "textured", "quads.obj")
    v, f, tex = nr.load_obj(obj, texture_size=4, load_texture=True)
    # host composition with the oracle in place of the kernel
    uv, names = io.parse_texture_faces(obj)
    want = np.full((6, 4, 4, 4, 3), 0.5, dtype=np.float32)
    want[1:4] = np.float32([0.2, 0.4, 0.6])
    want[4:] = np.float32([0.9, 0.1, 0.3])
    img = io._read_image(os.path.join(os.path.dirname(obj), "pattern.png"))[::-1]
    want = o.bake_textures(img, uv, (np.array(names) == "painted").astype(np.int32), 4, want)
    assert ((tex.view(np.uint32) == want.view(np.uint32)) | (np.isnan(tex) & np.isnan(want))).all()
    dev = torch.device("cuda")
    r = nr.Renderer()
    r.image_size = 64
    r.eye = nr.get_points_from_angles(2.732, 20, 30)
    image = r.render(torch.from_numpy(v)[None].to(dev), torch.from_numpy(f)[None].to(dev), torch.from_numpy(tex)[None].to(dev))
    assert image.shape == (1, 3, 64, 64) and torch.isfinite(image).all()  # texel (0,0,0) (NaN) is never sampled at ts = 4
    assert float(image.max()) > 0.1


# ---------------------------------------------------------------------- ABI 3: geometry and textures without copies
def _indexed_case(B, nv_scale=1.0, seed=0):
    from neural_renderer_b200 import synthetic
    v_np, f_np = synthetic.sphere_mesh(1800)
    rng = np.random.default_rng(seed)
    vs = []
    for b in range(B):
        v = (v_np * 0.7) @ synthetic._rotation(rng).T
        v[:, 2] += 2.6
        vs.append(v.astype(np.float32))
    return np.stack(vs), f_np


@pytest.mark.parametrize("flags", [(1, 1, 1), (0, 1, 0), (0, 0, 1)], ids=["rgb_alpha_depth", "alpha", "depth"])
@pytest.mark.parametrize("shared_idx", [False, True], ids=["idx_per_item", "idx_shared"])
def test_indexed_geometry_matches_materialised_faces(flags, shared_idx):
    """NR_FACES_INDEXED: rasterize(indices, ..., vertices=v) == rasterize(vertices_to_faces(v, indices), ...): the maps
    bit for bit (the same floats reach the same expressions), d loss / d vertices up to the order of the atomics --
    vertices_to_faces.py:16-21 and its get_item backward folded into the kernels (SURVEY.md 8(f)-1)."""
    import importlib
    import neural_renderer as nr
    R = importlib.import_module("neural_renderer_b200.rasterize")
    dev = torch.device("cuda")
    B = 3
    v_np, f_np = _indexed_case(B, seed=4)
    idx = torch.from_numpy(f_np).to(dev)
    idx_b = idx[None].expand(B, -1, -1).contiguous()
    tex = torch.rand((B, f_np.shape[0], 2, 2, 2, 3), generator=torch.Generator().manual_seed(1)).to(dev)
    bg = (0.2, 0.1, 0.3)

    def run(indexed):
        v = torch.from_numpy(v_np).to(dev).requires_grad_(True)
        t = tex.clone().requires_grad_(True)
        if indexed:
            out = R._run(idx if shared_idx else idx_b, t if flags[0] else None, 64, False, 0.1, 100, 1e-4, bg, *flags, vertices=v)
        else:
            out = R._run(nr.vertices_to_faces(v, idx_b), t if flags[0] else None, 64, False, 0.1, 100, 1e-4, bg, *flags)
        gen = torch.Generator().manual_seed(9)
        loss = 0
        for o in out[:3]:
            if o is not None:
                loss = loss + (o * torch.randn(o.shape, generator=gen).to(dev)).sum()
        loss.backward()
        return out, v.grad, t.grad

    a, gva, gta = run(True)
    b, gvb, gtb = run(False)
    for x, y in zip(a, b):
        assert (x is None) == (y is None)
        if x is not None:
            assert torch.equal(x, y)
    assert rel_err(gva.cpu(), gvb.cpu()) <= 1e-5
    if flags[0]:
        assert rel_err(gta.cpu(), gtb.cpu()) <= 1e-6


def test_indexed_geometry_out_of_range_indices_read_zero_vertices():
    """like nr_b200_vertices_to_faces: an index outside [0, Nv) gathers a vertex of zeros and receives no gradient"""
    import importlib
    R = importlib.import_module("neural_renderer_b200.rasterize")
    dev = torch.device("cuda")
    v_np, f_np = _indexed_case(1, seed=5)
    f_bad = f_np.copy()
    f_bad[::7, 1] = v_np.shape[1] + 5
    f_bad[3::11, 0] = -1
    v = torch.from_numpy(v_np).to(dev).requires_grad_(True)
    out = R._run(torch.from_numpy(f_bad).to(dev), None, 64, False, 0.1, 100, 1e-4, None, False, True, False, vertices=v)
    faces = torch.zeros((1, f_bad.shape[0], 3, 3), device=dev)
    ok = (f_bad >= 0) & (f_bad < v_np.shape[1])
    gathered = v.detach()[0][torch.from_numpy(np.where(ok, f_bad, 0)).to(dev).long()]
    faces[0] = torch.where(torch.from_numpy(ok).to(dev)[..., None], gathered, torch.zeros((), device=dev))
    ref = R._run(faces, None, 64, False, 0.1, 100, 1e-4, None, False, True, False)
    assert torch.equal(out[1], ref[1]) and torch.equal(out[3], ref[3])
    (out[1] * torch.randn(out[1].shape, generator=torch.Generator().manual_seed(2)).to(dev)).sum().backward()
    assert torch.isfinite(v.grad).all()


@pytest.mark.parametrize("fill_back", [False, True])
def test_shared_textures_match_expanded_copy(fill_back):
    """NR_TEX_SHARED: textures [1,F,...] (or an expanded stride-0 batch) sampled in place == the materialised
    [B,F,...] copy; the gradient is the sum over the batch items (Mesh.get_batch's broadcast backward, mesh.py:29-34)."""
    import importlib
    R = importlib.import_module("neural_renderer_b200.rasterize")
    dev = torch.device("cuda")
    B = 4
    v_np, f_np = _indexed_case(B, seed=6)
    idx = torch.from_numpy(f_np).to(dev)
    if fill_back:
        idx = torch.cat((idx, idx.flip(1)), dim=0)
    ncube = f_np.shape[0]
    base = torch.rand((ncube, 2, 2, 2, 3), generator=torch.Generator().manual_seed(3)).to(dev)
    g = torch.randn((B, 3, 64, 64), generator=torch.Generator().manual_seed(4)).to(dev)
    light = torch.rand((B, idx.shape[0], 3), generator=torch.Generator().manual_seed(5)).to(dev)
    res = {}
    for kind in ("copy", "batch1", "expanded"):
        t0 = base.clone().requires_grad_(True)
        if kind == "copy":
            t = t0[None].expand(B, -1, -1, -1, -1, -1).contiguous()
        elif kind == "batch1":
            t = t0[None]
        else:
            t = t0[None].expand(B, -1, -1, -1, -1, -1)
        v = torch.from_numpy(v_np).to(dev).requires_grad_(True)
        out = R._run(idx, t, 64, False, 0.1, 100, 1e-3, (0, 0, 0), True, False, False, face_light=light,
                     textures_fill_back=fill_back, vertices=v)
        (out[0] * g).sum().backward()
        res[kind] = (out[0].detach(), t0.grad, v.grad)
    for kind in ("batch1", "expanded"):
        assert torch.equal(res[kind][0], res["copy"][0])
        assert rel_err(res[kind][1].cpu(), res["copy"][1].cpu()) <= 1e-5
        assert rel_err(res[kind][2].cpu(), res["copy"][2].cpu()) <= 1e-5


def test_backward_in_two_parts_with_texture_hook():
    """NR_BWD_PART_TEXTURES / NR_BWD_PART_FACES: the hook sees the finished texture gradient before the edge scan is
    enqueued, and the two halves add up to exactly what the single call computes."""
    import importlib
    R = importlib.import_module("neural_renderer_b200.rasterize")
    from neural_renderer_b200 import synthetic
    dev = torch.device("cuda")
    faces_np = synthetic.sphere_faces(2, 800, seed=3)
    tex_np = synthetic.random_textures(2, 800, 2, seed=4)
    g = torch.randn((2, 3, 64, 64), generator=torch.Generator().manual_seed(1)).to(dev)

    def run():
        f = torch.from_numpy(faces_np).to(dev).requires_grad_(True)
        t = torch.from_numpy(tex_np).to(dev).requires_grad_(True)
        (R._run(f, t, 64, False, 0.1, 100, 1e-4, (0, 0, 0), True, False, False)[0] * g).sum().backward()
        return f.grad, t.grad

    gf0, gt0 = run()
    seen = {}

    class Pending:
        def wait(self):
            seen["waited"] = True

    def hook(grad_textures):
        seen["tex"] = grad_textures.clone()  # stream-ordered: the edge scan has not been enqueued yet
        return Pending()

    prev = R.set_texture_grad_hook(hook)
    try:
        gf1, gt1 = run()
    finally:
        R.set_texture_grad_hook(prev)
    assert seen.get("waited") and torch.equal(seen["tex"], gt1)
    assert rel_err(gt1.cpu(), gt0.cpu()) <= 1e-6
    assert rel_err(gf1.cpu(), gf0.cpu()) <= 1e-5


def test_renderer_fused_path_has_no_face_tensor(teapot):
    """Renderer.render* with the fused path: gradients reach the vertices through the indexed rasterizer and agree
    with the op-by-op formulation (vertices_to_faces + lighting + doubled textures)."""
    import neural_renderer as nr
    dev = torch.device("cuda")
    v, f = teapot
    B = 2
    faces_idx = torch.from_numpy(np.stack([f] * B)).to(dev)
    tex0 = torch.rand((B, f.shape[0], 2, 2, 2, 3), generator=torch.Generator().manual_seed(1)).to(dev)
    out = {}
    for fused in (True, False):
        vert = torch.from_numpy(np.stack([v, v * 0.9])).to(dev).requires_grad_(True)
        tex = tex0.clone().requires_grad_(True)
        r = nr.Renderer()
        r.fused = fused
        r.image_size = 64
        r.eye = nr.get_points_from_angles(2.732, 20, 50)
        imgs = (r.render(vert, faces_idx, tex), r.render_silhouettes(vert, faces_idx), r.render_depth(vert, faces_idx))
        gen = torch.Generator().manual_seed(7)
        loss = sum((im * torch.randn(im.shape, generator=gen).to(dev)).sum() for im in imgs)
        loss.backward()
        out[fused] = (imgs, vert.grad, tex.grad)
    for a, b in zip(out[True][0], out[False][0]):
        assert rel_err(a.detach().cpu(), b.detach().cpu()) <= 1e-5
    assert rel_err(out[True][1].cpu(), out[False][1].cpu()) <= 1e-4
    assert rel_err(out[True][2].cpu(), out[False][2].cpu()) <= 1e-4


@pytest.mark.parametrize("ts,fill_back,lit", [(4, False, False), (2, True, True), (3, False, False)])
def test_staged_texture_path_renders_the_same_pixels(ts, fill_back, lit):
    """NR_FWD_STAGE_TEXTURES: texture cubes staged per pixel row in shared memory with cp.async.bulk (TMA) -- bit-identical
    images to the direct gather (ts = 3: cubes of 324 bytes cannot be bulk-copied, the flag falls back silently)."""
    import importlib
    R = importlib.import_module("neural_renderer_b200.rasterize")
    from neural_renderer_b200 import synthetic
    dev = torch.device("cuda")
    B, F, S = 3, 3000, 320  # 320: a second, partial column chunk per row
    faces = torch.from_numpy(synthetic.sphere_faces(B, F, seed=9)).to(dev)
    ncube = F // 2 if fill_back else F
    tex = torch.from_numpy(synthetic.random_textures(B, ncube, ts, seed=10)).to(dev)
    light = torch.rand((B, F, 3), generator=torch.Generator().manual_seed(2)).to(dev) if lit else None
    out = {}
    for staged in (False, True):
        R.set_stage_textures(staged)
        try:
            out[staged] = R._run(faces, tex, S, False, 0.1, 100, 1e-4, (0.3, 0.2, 0.1), True, True, False, face_light=light,
                                 textures_fill_back=fill_back)
        finally:
            R.set_stage_textures(False)
    for a, b in zip(out[False], out[True]):
        if a is not None:
            assert torch.equal(a, b)
    assert float((out[True][3] >= 0).float().mean()) > 0.2
