"""GPU parity tests proper (-m gpu): this repo's CUDA path, called through the public Python API -> torch
binding -> C ABI, against
  * the UNMODIFIED reference CUDA extension (oracle/_ref, where a build for that feature width is present),
  * the CPU oracle (oracle/) for every case small enough, and
  * stored records (tests/golden/records, tests/make_records.py) for the full-size configs 2-5,
on identical seeded inputs.  Bars (BASELINE.json north_star): bit-exact tile/key indexing (radii,
num_rendered, point_list, ranges, n_contrib); RGB/feature/depth/gradients within 1e-4 relative
(parity.RTOL + ATOL_REL floor).  On top of the bar, colour / depth / final_T are asserted BIT-identical to
the reference build (same fp32 operation sequence), the feature map to 5e-6 of its scale.
Nothing here reads /root/reference.
"""
import copy
import os

import numpy as np
import pytest

import parity
import scenegen

pytestmark = pytest.mark.gpu


def _ref_available(C):
    from oracle import ref_wrapper as rw

    return rw.available(C)


def _check_record(ours, name):
    """Against the stored record of a full-size case (tests/make_records.py, parity.check_record): bit-exact digests of
    the indices and of colour / depth / final_T, and the CPU oracle's block and channel sums for every float array."""
    rec = np.load(os.path.join(os.path.dirname(__file__), "golden", "records", name + ".npz"))
    bad = parity.check_record(ours, rec)
    assert not bad, f"vs stored record {name} ({rec['gpu']}):\n  " + "\n  ".join(bad)


def _check(sc, cam, with_grads=True, vs_ref=True, vs_oracle=True, exact_vs_ref=True, record=None, **kw):
    grads = scenegen.upstream_grads(cam.image_height, cam.image_width, sc.C) if with_grads else None
    ours = parity.run_ours(sc, cam, grads=grads, **kw)
    n = 0
    if record is not None:
        _check_record(ours, record)
        n += 1
    if vs_ref and _ref_available(sc.C) and not kw:
        ref = parity.run_ref(sc, cam, grads=grads)
        rep = parity.compare(ours, ref)
        assert rep["ok"], "vs reference CUDA:\n" + parity.format_report(rep)
        if exact_vs_ref:
            for k in ("color", "depth", "final_T"):
                assert np.array_equal(ours[k], ref[k]), f"{k} not bit-identical to the reference build"
            if sc.C:
                # fp32-pipe kernel: <= 2e-6 of scale; tensor-core path (C > 64, compensated 3xTF32): <= 5e-6 of scale.
                # Both are ~20-50x inside the 1e-4 bar checked by parity.compare above.
                assert rep["feature_map"]["max_abs_err"] <= 5e-6 * max(rep["feature_map"]["scale"], 1e-6)
        n += 1
    if vs_oracle:
        okw = {k: v for k, v in kw.items() if k in ("colors_precomp", "cov3D_precomp")}
        orc = parity.run_oracle(sc, cam, grads=grads, threads=1, **okw)
        gk = tuple(k for k in ("means3D", "means2D", "sh", "semantic_feature", "opacities", "scales", "rotations",
                               "colors_precomp", "cov3D_precomp") if grads is not None and k in ours["grads"])
        rep = parity.compare(ours, orc, grad_keys=gk, tie_tolerant=True)
        assert rep["ok"], "vs CPU oracle:\n" + parity.format_report(rep)
        n += 1
    assert n > 0
    return ours


# ------------------------------------------------------------------------------------------- configs
@pytest.mark.parametrize("name", ["tiny", "small", "c1"])
def test_small_configs_vs_reference_and_oracle(name):
    sc = scenegen.make_config(name)
    _check(sc, sc.cameras[0])


def test_c2_vs_reference():
    sc = scenegen.make_config("c2")
    _check(sc, sc.cameras[0], vs_oracle=False, record="c2")


def test_golden_fixtures_match_gpu():
    """The committed golden vectors (reference outputs from an earlier B200 run) against today's GPU result."""
    import glob
    import os

    for path in sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))):
        g = np.load(path)
        sc = scenegen.make_config(str(g["config"]), seed=int(g["seed"]))
        cam = sc.cameras[0]
        ours = parity.run_ours(sc, cam, grads=scenegen.upstream_grads(cam.image_height, cam.image_width, sc.C))
        for k in ("radii", "point_list", "ranges", "n_contrib"):
            assert np.array_equal(np.asarray(ours[k]).astype(np.int64), g[k].astype(np.int64)), (path, k)
        for k in ("color", "depth", "final_T"):
            assert np.array_equal(ours[k], g[k]), (path, k)
        assert parity.float_mismatch(ours["feature_map"], g["feature_map"])[0] <= 1.0
        for k in ("means3D", "means2D", "sh", "semantic_feature", "opacities", "scales", "rotations"):
            assert parity.float_mismatch(ours["grads"][k], g["grad_" + k])[0] <= 1.0, (path, k)


# ------------------------------------------------------------------------------------------- feature widths
@pytest.mark.parametrize("C", [0, 1, 3, 4, 5, 8, 16, 31, 32, 33, 64, 100, 128, 129, 160, 256, 300])
def test_feature_widths(C):
    """Run-time feature width incl. widths that are not a multiple of 4 (no bulk-copy path), padding inside a
    128-channel chunk and multi-chunk widths (> 128)."""
    sc = scenegen.make_scene(P=1500, W=96, H=64, C=C, sh_degree=1, seed=100 + C)
    _check(sc, sc.cameras[0])


# ------------------------------------------------------------------------------------------- image shapes
@pytest.mark.parametrize("W,H", [(83, 61), (100, 40), (16, 16), (17, 33), (250, 10), (8, 8)])
def test_image_shapes_not_multiple_of_tile_or_vector(W, H):
    sc = scenegen.make_scene(P=800, W=W, H=H, C=8, sh_degree=2, seed=W * 1000 + H, target_radius_px=4.0)
    _check(sc, sc.cameras[0])


# ------------------------------------------------------------------------------------------- option matrix
@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_sh_degrees(deg):
    sc = scenegen.make_scene(P=1200, W=80, H=64, C=8, sh_degree=deg, seed=20 + deg)
    _check(sc, sc.cameras[0])


def test_background_and_scale_modifier():
    sc = scenegen.make_scene(P=1200, W=80, H=64, C=8, sh_degree=3, seed=31)
    sc.bg = np.array([0.3, 0.7, 0.1], np.float32)
    _check(sc, sc.cameras[0])


def test_colors_precomp_and_cov3d_precomp():
    sc = scenegen.make_scene(P=1200, W=80, H=64, C=8, sh_degree=3, seed=32)
    cam = sc.cameras[0]
    import oracle

    f = oracle.forward(sc, cam)
    rng = np.random.Generator(np.random.PCG64(5))
    colors = rng.uniform(0, 1, size=(sc.P, 3)).astype(np.float32)
    _check(sc, cam, vs_ref=False, colors_precomp=colors)
    _check(sc, cam, vs_ref=False, cov3D_precomp=f["cov3D"].copy())
    _check(sc, cam, vs_ref=False, colors_precomp=colors, cov3D_precomp=f["cov3D"].copy())


def test_debug_mode_synchronises_and_matches():
    sc = scenegen.make_config("tiny")
    a = parity.run_ours(sc, sc.cameras[0], debug=True)
    b = parity.run_ours(sc, sc.cameras[0], debug=False)
    for k in ("color", "feature_map", "depth", "n_contrib", "point_list"):
        assert np.array_equal(a[k], b[k])


# ------------------------------------------------------------------------------------------- edge cases
def test_empty_cloud_returns_zeros_like_reference():
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer

    sc = scenegen.make_scene(P=1, W=32, H=32, C=4, seed=1)
    rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(sc, sc.cameras[0], "cuda"))
    z = lambda *s: torch.zeros(*s, device="cuda")  # noqa: E731
    color, feat, radii, depth = GaussianRasterizer(rs)(means3D=z(0, 3), means2D=z(0, 3), opacities=z(0, 1),
                                                       shs=z(0, 16, 3), semantic_feature=z(0, 1, 4),
                                                       scales=z(0, 3), rotations=z(0, 4))
    assert color.shape == (3, 32, 32) and feat.shape == (4, 32, 32) and radii.shape == (0,)
    assert float(color.abs().sum()) == 0 and float(feat.abs().sum()) == 0 and float(depth.abs().sum()) == 0


def test_everything_culled_renders_background():
    sc = scenegen.make_scene(P=500, W=64, H=48, C=8, seed=3)
    sc.means3D = sc.means3D + np.array([100.0, 0, 0], np.float32)  # far off to the side, still in front
    sc.means3D[:250] = sc.cameras[0].campos * 2.0                 # behind the camera (it looks at the origin)
    sc.bg = np.array([0.2, 0.4, 0.6], np.float32)
    ours = _check(sc, sc.cameras[0], vs_ref=True)
    assert int(ours["num_rendered"]) == 0 or int(ours["num_rendered"]) > 0  # either way parity held
    behind = ours["radii"][:250]
    assert (behind == 0).all()
    g = ours["grads"]
    for k in ("means3D", "scales", "rotations", "opacities", "sh", "semantic_feature"):
        assert np.abs(g[k][:250]).max() == 0, k


def test_single_gaussian():
    sc = scenegen.make_scene(P=1, W=48, H=48, C=4, seed=4, target_radius_px=10.0)
    sc.means3D[:] = 0
    sc.opacities[:] = 0.9
    _check(sc, sc.cameras[0], vs_ref=False)


def test_huge_splats_cover_many_tiles():
    """Rectangles of hundreds of tiles: exercises the warp-cooperative key emission and long per-tile lists."""
    sc = scenegen.make_scene(P=300, W=320, H=240, C=16, sh_degree=1, seed=6, target_radius_px=120.0)
    ours = _check(sc, sc.cameras[0])
    assert int(ours["num_rendered"]) > 20 * 300


def test_opaque_dense_scene_terminates_early():
    """Near-opaque splats: most pixels saturate (T < 1e-4) long before their list ends."""
    sc = scenegen.make_scene(P=6000, W=96, H=96, C=32, sh_degree=0, seed=8, target_radius_px=25.0)
    sc.opacities[:] = 0.995
    ours = _check(sc, sc.cameras[0])
    ranges = ours["ranges"]
    longest = int((ranges[:, 1] - ranges[:, 0]).max())
    assert ours["n_contrib"].max() < longest  # early termination actually happened
    assert (ours["final_T"] < 1e-3).mean() > 0.3


def test_low_opacity_never_contributes():
    sc = scenegen.make_scene(P=1000, W=64, H=64, C=8, seed=9)
    sc.opacities[:500] = 1.0 / 512  # < 1/255: alpha can never pass the threshold
    ours = _check(sc, sc.cameras[0])
    assert np.abs(ours["grads"]["semantic_feature"][:500]).max() == 0


def test_noncontiguous_inputs_are_accepted():
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer

    sc = scenegen.make_config("tiny")
    cam = sc.cameras[0]
    t = scenegen.to_torch(sc, "cuda")
    rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(sc, cam, "cuda"))
    base = GaussianRasterizer(rs)(means3D=t["means3D"], means2D=torch.zeros_like(t["means3D"]),
                                  opacities=t["opacities"], shs=t["shs"], semantic_feature=t["semantic_feature"],
                                  scales=t["scales"], rotations=t["rotations"])
    m_nc = t["means3D"].t().contiguous().t()          # same values, column-major strides
    f_nc = t["semantic_feature"].transpose(1, 2).contiguous().transpose(1, 2)
    out = GaussianRasterizer(rs)(means3D=m_nc, means2D=torch.zeros_like(t["means3D"]), opacities=t["opacities"],
                                 shs=t["shs"], semantic_feature=f_nc, scales=t["scales"], rotations=t["rotations"])
    assert not m_nc.is_contiguous()
    for a, b in zip(base, out):
        assert torch.equal(a, b)


def test_runs_on_the_current_stream_and_is_deterministic_forward():
    import torch

    sc = scenegen.make_config("small")
    a = parity.run_ours(sc, sc.cameras[0])
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        b = parity.run_ours(sc, sc.cameras[0])
    s.synchronize()
    for k in ("color", "feature_map", "depth", "final_T", "n_contrib", "point_list", "ranges", "radii"):
        assert np.array_equal(a[k], b[k]), k


def test_forward_bit_identical_over_many_runs_c2():
    """Race regression (round 1): the persistent composite hands tiles out through a global atomic counter, so which
    tiles share a CTA - and how far its producer warp runs ahead - changes from run to run.  The forward has no
    atomics in its data path, so its outputs must not: 40 runs of config 2 (300k Gaussians, 800x800, C=16; this
    caught early-termination flags of two in-flight tiles aliasing) and the backward must agree within a fraction
    of the parity tolerance (its float atomics may reorder)."""
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer

    sc = scenegen.make_config("c2")
    cam = sc.cameras[0]
    t = scenegen.to_torch(sc, "cuda", requires_grad=True)
    rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(sc, cam, "cuda"))
    gc, gf, gd = [torch.from_numpy(g).cuda() for g in scenegen.upstream_grads(cam.image_height, cam.image_width, sc.C)]
    base = gbase = None
    for it in range(40):
        m2 = torch.zeros_like(t["means3D"], requires_grad=True)
        color, feat, radii, depth = GaussianRasterizer(rs)(
            means3D=t["means3D"], means2D=m2, opacities=t["opacities"], shs=t["shs"],
            semantic_feature=t["semantic_feature"], scales=t["scales"], rotations=t["rotations"])
        torch.autograd.backward([color, depth, feat], [gc, gd, gf])
        cur = [color.detach().clone(), feat.detach().clone(), depth.detach().clone(), radii.clone()]
        g = {k: t[k].grad.clone() for k in t if t[k].grad is not None}
        g["means2D"] = m2.grad.clone()
        for k in t:
            t[k].grad = None
        if base is None:
            base, gbase = cur, g
            continue
        for a, b, k in zip(cur, base, ("color", "feature_map", "depth", "radii")):
            assert torch.equal(a, b), (it, k, int((a != b).sum()))
        for k in g:
            b = gbase[k].double()
            tol = parity.RTOL * b.abs() + parity.GRAD_ATOL_REL * b.abs().max()
            assert float(((g[k].double() - b).abs() / tol).max()) <= 0.5, (it, k)


def test_mark_visible_matches_oracle():
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    import oracle

    sc = scenegen.make_scene(P=5000, W=64, H=64, C=0, seed=12)
    sc.means3D *= 4.0  # some behind the camera
    cam = sc.cameras[0]
    rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(sc, cam, "cuda"))
    vis = GaussianRasterizer(rs).markVisible(torch.from_numpy(sc.means3D).cuda())
    assert vis.dtype == torch.bool
    ref = oracle.mark_visible(sc.means3D, cam.viewmatrix)
    assert np.array_equal(vis.cpu().numpy(), ref) and 0 < ref.sum() < sc.P


def test_cpu_tensor_on_gpu_box_still_fails_loudly():
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer

    sc = scenegen.make_config("tiny")
    rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(sc, sc.cameras[0], "cuda"))
    t = scenegen.to_torch(sc, "cpu")
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        GaussianRasterizer(rs)(means3D=t["means3D"], means2D=torch.zeros_like(t["means3D"]), opacities=t["opacities"],
                               shs=t["shs"], semantic_feature=t["semantic_feature"], scales=t["scales"],
                               rotations=t["rotations"])


# ------------------------------------------------------------------------------------------- full-size properties
@pytest.fixture(scope="module")
def c3_scene():
    return scenegen.make_config("c3")


def _full_size_vs_reference(sc, with_grads, label):
    """One full-size view against its stored record and, where a reference build for this width is present, device-side
    against the reference build; the latter prints the worst violation ratio (|a-b| / tolerance, <= 1 passes) of every
    float tensor so the margin is on record in the test log."""
    import torch
    from oracle import ref_wrapper as rw

    cam = sc.cameras[0]
    grads = scenegen.upstream_grads(cam.image_height, cam.image_width, sc.C) if with_grads else None
    ours = parity.run_ours(sc, cam, grads=grads)
    _check_record(ours, label)
    if not rw.available(sc.C):
        return
    ref = parity.run_ref(sc, cam, grads=grads)
    for k in ("radii", "point_list", "ranges", "n_contrib"):
        assert np.array_equal(ours[k], ref[k]), k
    assert int(ours["num_rendered"]) == int(ref["num_rendered"])
    for k in ("color", "depth", "final_T"):
        assert np.array_equal(ours[k], ref[k]), k

    def viol(a, b, atol):
        a, b = torch.from_numpy(a).cuda().double(), torch.from_numpy(b).cuda().double()
        tol = parity.RTOL * b.abs() + atol * b.abs().max()
        return float(((a - b).abs() / tol).max())

    worst = {}
    if sc.C:
        worst["feature_map"] = viol(ours["feature_map"], ref["feature_map"], parity.ATOL_REL)
    if with_grads:
        for k in ("means3D", "means2D", "sh", "semantic_feature", "opacities", "scales", "rotations"):
            if k in ours["grads"]:
                worst["grad_" + k] = viol(ours["grads"][k], ref["grads"][k], parity.GRAD_ATOL_REL)
    print(f"[{label}] V={int((ours['radii'] > 0).sum())} R={int(ours['num_rendered'])} worst viol per tensor: "
          + ", ".join(f"{k}={v:.3g}" for k, v in worst.items()))
    for k, v in worst.items():
        assert v <= 1.0, (k, v)


def test_c3_full_size_vs_reference(c3_scene):
    """BASELINE.json's metric configuration itself: 1M Gaussians, 1080p, C=128 (device-side comparison)."""
    _full_size_vs_reference(c3_scene, True, "c3")


def test_c4_full_size_vs_reference():
    """BASELINE.json configs[3]: 1M Gaussians, 1080p, C=256 (two 128-channel chunks per tile), forward + backward."""
    _full_size_vs_reference(scenegen.make_config("c4", views=1), True, "c4")


def test_c5_forward_vs_reference():
    """BASELINE.json configs[4]: 5M Gaussians, 3840x2160, C=64, forward only (R ~ 16M instances, 47-bit sort keys)."""
    _full_size_vs_reference(scenegen.make_config("c5"), False, "c5")


def test_c3_structural_properties(c3_scene):
    """Size-independent properties at the full BASELINE size."""
    sc = c3_scene
    cam = sc.cameras[0]
    ours = parity.run_ours(sc, cam)
    R = int(ours["num_rendered"])
    ranges, pl = ours["ranges"], ours["point_list"]
    # ranges partition [0, R) in tile order; empty tiles are (0, 0)
    nz = ranges[(ranges[:, 1] - ranges[:, 0]) > 0]
    assert nz[0, 0] == 0 and nz[-1, 1] == R and np.array_equal(nz[1:, 0], nz[:-1, 1])
    # within a tile the list is depth sorted (ties broken by index = stable sort)
    depth = ours["rec"][:, 11]
    d = depth[pl]
    same_tile = np.ones(R - 1, bool)
    same_tile[nz[:-1, 1] - 1] = False
    assert (np.diff(d)[same_tile] >= 0).all()
    ties = same_tile & (np.diff(d) == 0)
    assert (np.diff(pl)[ties] > 0).all()
    # every visible Gaussian appears exactly tiles_touched times
    counts = np.bincount(pl, minlength=sc.P)
    assert ((counts > 0) == (ours["radii"] > 0)).all()
    # n_contrib never exceeds the tile's list length; T in (0, 1]
    gx = (cam.image_width + 15) // 16
    ty, tx = np.divmod(np.arange(cam.image_height * cam.image_width), cam.image_width)
    tile = (ty // 16) * gx + (tx // 16)
    lens = (ranges[:, 1] - ranges[:, 0])[tile].reshape(cam.image_height, cam.image_width)
    assert (ours["n_contrib"] <= lens).all()
    assert (ours["final_T"] > 0).all() and (ours["final_T"] <= 1).all()


def test_c3_feature_linearity_and_width_independence(c3_scene):
    """feature_map is linear in the features (blend weights do not depend on them): F(2f) == 2 F(f) bit for bit,
    and colour / depth / indices are bit-identical for C = 0 and C = 128."""
    sc = c3_scene
    cam = sc.cameras[0]
    a = parity.run_ours(sc, cam)
    sc2 = copy.copy(sc)
    sc2.features = sc.features * 2.0
    b = parity.run_ours(sc2, cam)
    assert np.array_equal(b["feature_map"], 2.0 * a["feature_map"])
    sc0 = copy.copy(sc)
    sc0.features = np.zeros((sc.P, 1, 0), np.float32)
    c = parity.run_ours(sc0, cam)
    for k in ("color", "depth", "final_T", "n_contrib", "point_list", "ranges", "radii"):
        assert np.array_equal(a[k], c[k]), k


# ------------------------------------------------------------------------------------------- view batches
@pytest.mark.parametrize("name", ["tiny", "small"])
def test_view_batch_accumulates_like_autograd(name):
    """ViewBatch (f3dgs_backward_accum: gradients ADDED in-kernel into one flat buffer, densification statistics folded
    in) against the sum over views of the per-view gradients from the reference-compatible autograd API."""
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    from diff_gaussian_rasterization.parallel import ViewBatch

    sc = scenegen.make_config(name, views=3)
    dev = "cuda"
    t = scenegen.to_torch(sc, dev, requires_grad=True)
    cam0 = sc.cameras[0]
    ups = [[torch.from_numpy(g).to(dev) for g in scenegen.upstream_grads(cam0.image_height, cam0.image_width, sc.C, seed=50 + v)]
           for v in range(3)]
    names = ("means3D", "scales", "rotations", "opacities", "shs", "semantic_feature")
    want = {k: torch.zeros_like(t[k]) for k in names}
    accum, denom = torch.zeros(sc.P, device=dev), torch.zeros(sc.P, device=dev)
    outs = []
    for v, cam in enumerate(sc.cameras):
        rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(sc, cam, dev))
        m2 = torch.zeros_like(t["means3D"], requires_grad=True)
        color, feat, radii, depth = GaussianRasterizer(rs)(
            means3D=t["means3D"], means2D=m2, opacities=t["opacities"], shs=t["shs"],
            semantic_feature=t["semantic_feature"], scales=t["scales"], rotations=t["rotations"])
        torch.autograd.backward([color, depth, feat], [ups[v][0], ups[v][2], ups[v][1]])
        for k in names:
            want[k] += t[k].grad
            t[k].grad = None
        vis = radii > 0
        accum[vis] += m2.grad[vis, :2].norm(dim=-1)   # scene/gaussian_model.py:436-438
        denom[vis] += 1
        outs.append((color.detach(), feat.detach(), depth.detach(), m2.grad.clone()))

    vb = ViewBatch({k: t[k].detach() for k in names})
    vb.zero_()
    for v, cam in enumerate(sc.cameras):
        rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(sc, cam, dev))
        color, feat, radii, depth, ctx = vb.forward(rs)
        assert torch.equal(color, outs[v][0]) and torch.equal(depth, outs[v][2]) and torch.equal(feat, outs[v][1])
        m2 = torch.empty(sc.P, 3, device=dev)
        vb.backward(ctx, ups[v][0], ups[v][1], ups[v][2], means2D_out=m2, last=(v == 2))
        assert parity.float_mismatch(m2.cpu().numpy(), outs[v][3].cpu().numpy(), atol_rel=parity.GRAD_ATOL_REL)[0] <= 1.0
    vb.all_reduce()  # no process group: a no-op that must leave the buffer intact
    for k in names:
        r = parity.float_mismatch(vb.grads[k].cpu().numpy(), want[k].cpu().numpy(), atol_rel=parity.GRAD_ATOL_REL)[0]
        assert r <= 1.0, (k, r)
    assert torch.equal(vb.denom, denom)
    assert parity.float_mismatch(vb.grad_accum.cpu().numpy(), accum.cpu().numpy(), atol_rel=parity.GRAD_ATOL_REL)[0] <= 1.0


# ------------------------------------------------------------------------------------------- per-process overrides
@pytest.mark.parametrize("env", [{"F3DGS_TC": "0"}, {"F3DGS_BWD2": "0"}, {"F3DGS_TC": "0", "F3DGS_BWD2": "0"},
                                 {"F3DGS_TC_MIN_C": "16"}, {"F3DGS_FBWD_TC": "1"}])
def test_kernel_selection_overrides_keep_parity(env):
    """F3DGS_TC / F3DGS_BWD2 / F3DGS_TC_MIN_C / F3DGS_FBWD_TC are read once per process, so each setting runs in its own
    interpreter: the fp32-pipe forward, the fused single-kernel backward, the tensor-core path at narrow widths and the
    opt-in tensor-core feature-gradient kernel must all pass the same parity checks as the defaults."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys; sys.path[:0] = [%r, %r, %r]\n"
        "import scenegen, parity\n"
        "from test_gpu_parity import _check\n"
        "for name in ('small', 'small128', 'small200'):\n"
        "    sc = scenegen.make_config(name); _check(sc, sc.cameras[0], vs_ref=(name == 'small'))\n"
        "print('OVERRIDE OK')\n" % (root, os.path.join(root, "feature-3dgs_b200"), os.path.join(root, "tests")))
    r = subprocess.run([sys.executable, "-c", code], env={**os.environ, **env}, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "OVERRIDE OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
