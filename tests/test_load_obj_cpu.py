"""CPU tests of the OBJ / MTL loader and of the texture-bake oracle (SURVEY.md section 8(f) row 4; reference
load_obj.py:8-197).  The fixture under tests/golden/textured is synthetic (tests/golden/make_textured_fixture.py)."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "tests", "golden", "textured", "quads.obj")


def test_geometry_and_fan_triangulation():
    from neural_renderer_b200 import io
    v, f = io.load_obj(OBJ, normalization=False)
    assert v.shape == (7, 3) and v.dtype == np.float32
    # triangle + quad (2) + triangle + quad (2)
    assert f.shape == (6, 3) and f.dtype == np.int32
    assert f.min() == 0 and f.max() == 6
    assert f[1].tolist() == [0, 1, 2] and f[2].tolist() == [0, 2, 3]  # fan around the first vertex (load_obj.py:171-175)
    vn, _ = io.load_obj(OBJ)  # load_obj.py:188-192
    assert abs(np.abs(vn).max() - 1.0) < 1e-6 or np.abs(vn).max() <= 1.0 + 1e-6
    assert np.allclose(vn.max(0) + vn.min(0), 0, atol=1e-6)


def test_uv_parsing_materials_and_wrap():
    from neural_renderer_b200 import io
    uv, names = io.parse_texture_faces(OBJ)
    assert uv.shape == (6, 3, 2)
    assert names == ['', 'painted', 'painted', 'painted', 'flat', 'flat']
    # faces without vt indices use index 0 - 1 = -1 = the LAST vt (reference quirk, load_obj.py:44-64), wrapped
    assert np.allclose(uv[0], np.array([[0.5, 0.4]] * 3, dtype=np.float32))
    assert np.allclose(uv[1], [[0, 0], [1, 0], [1, 1]])           # exactly 1 stays 1 (`1 < x` is strict, :66)
    assert np.allclose(uv[3], [[0.31, 0.77], [0.6, 0.25], [0.5, 0.4]], atol=1e-6)  # 1.6 -> 0.6, 2.4 -> 0.4
    colors, files = io.load_mtl(os.path.join(os.path.dirname(OBJ), "quads.mtl"))
    assert list(colors) == ['painted', 'flat'] and files == {'painted': 'pattern.png'}
    assert np.allclose(colors['flat'], [0.9, 0.1, 0.3])


def test_bake_oracle_known_answers():
    import nr_oracle as o
    rng = np.random.default_rng(0)
    H, W, ts = 9, 7, 4
    img = rng.random((H, W, 3), dtype=np.float32)
    # UVs on exact pixel centres: the three cube corners sample exactly those pixels
    uv = np.array([[[0, 0], [1, 0], [0.5, 1.0]], [[2 / 6, 3 / 8], [4 / 6, 1 / 8], [1 / 6, 5 / 8]]], dtype=np.float32)
    tex = o.bake_textures(img, uv, np.array([1, 0], dtype=np.int32), ts)
    assert np.isnan(tex[0, 0, 0, 0]).all() and np.isnan(tex[0]).sum() == 3      # texel (0,0,0): 0/0 like the reference
    assert np.array_equal(tex[1], np.full((ts, ts, ts, 3), 0.5, dtype=np.float32))  # is_update == 0: untouched
    assert np.allclose(tex[0, ts - 1, 0, 0], img[0, 0], atol=1e-6)               # dims (1,0,0) -> uv0
    assert np.allclose(tex[0, 0, ts - 1, 0], img[0, W - 1], atol=1e-6)           # dims (0,1,0) -> uv1
    assert np.allclose(tex[0, 0, 0, ts - 1], img[H - 1, 3], atol=1e-6)           # dims (0,0,1) -> uv2 (x = 0.5 * 6 = 3)
    tex = o.bake_textures(img, uv, None, ts)
    assert np.allclose(tex[1, ts - 1, 0, 0], img[3, 2], atol=1e-5)
    # a constant image bakes to that constant everywhere but the NaN texel
    const = np.full((H, W, 3), 0.25, dtype=np.float32)
    t2 = o.bake_textures(const, uv, None, ts)
    assert np.nanmin(t2) == 0.25 and np.nanmax(t2) == 0.25 and np.isnan(t2).sum() == 6


def test_load_textures_composition_with_oracle(monkeypatch):
    """load_textures: 0.5 grey, then Kd, then the bake for map_Kd materials -- with the CPU oracle standing in for
    the GPU kernel (this is the host logic; the kernel itself is covered by the -m gpu tests)."""
    import nr_oracle as o
    from neural_renderer_b200 import io
    monkeypatch.setattr(io, "bake_textures", lambda image, uv, upd, ts, tex: o.bake_textures(image, uv, upd, ts, tex))
    v, f, tex = io.load_obj(OBJ, texture_size=4, load_texture=True)
    assert tex.shape == (6, 4, 4, 4, 3) and tex.dtype == np.float32
    assert np.array_equal(tex[0], np.full((4, 4, 4, 3), 0.5, dtype=np.float32))          # no material
    assert np.allclose(tex[4], np.broadcast_to(np.float32([0.9, 0.1, 0.3]), (4, 4, 4, 3)))  # Kd only
    assert np.isnan(tex[1, 0, 0, 0]).all() and np.isfinite(tex[1].reshape(-1, 3)[1:]).all()
    img = io._read_image(os.path.join(os.path.dirname(OBJ), "pattern.png"))[::-1]
    assert np.allclose(tex[1, 3, 0, 0], img[0, 0], atol=1e-6)   # uv (0,0) of the flipped image = bottom-left pixel


def test_textured_model_renders_like_the_reference_snapshot(monkeypatch):
    """The reference's own textured test model (test_load_obj.py:55-62: 3644 faces, 7 materials, 2 texture images,
    texture_size 16) through THIS loader (OBJ / MTL parsing, image flip, UV wrap, Kd fill, bilinear bake) and the CPU
    oracle's Renderer, against the display.png the reference's test writes for it.  The snapshot is 8-bit and was
    min-max scaled by scipy.misc.toimage, so the comparison is on that scale; the model files are the re-serialised
    copy tests/golden/make_golden.py wrote (tests/golden/display)."""
    import nr_oracle as o
    from neural_renderer_b200 import io
    d = os.path.join(ROOT, "tests", "golden", "display")
    monkeypatch.setattr(io, "bake_textures", lambda image, uv, upd, ts, tex: o.bake_textures(image, uv, upd, ts, tex))
    v, f, tex = io.load_obj(os.path.join(d, "model.obj"), load_texture=True, texture_size=16)
    assert v.shape == (921, 3) and f.shape == (3644, 3) and tex.shape == (3644, 16, 16, 16, 3)
    r = o.Renderer()
    r.eye = o.get_points_from_angles(2, 15, -90)
    img = np.asarray(r.render(v[None], f[None], tex[None])["rgb"])[0].transpose(1, 2, 0)
    assert np.isfinite(img).all()                      # the NaN texel (0,0,0) of baked cubes is never sampled at ts = 16
    mine = (img - img.min()) / (img.max() - img.min()) * 255.0
    ref = np.load(os.path.join(d, "display_u8.npz"))["display_u8"].astype(np.float32)[..., :3]
    diff = np.abs(mine - ref)
    assert diff.mean() < 0.5 and diff.max() < 16.0, (diff.mean(), diff.max())   # observed 0.13 / 4.4 grey levels

