"""Shared parity harness: run one view through (a) this repo's CUDA path via the public Python API,
(b) the reference CUDA extension (oracle/_ref) or (c) the CPU oracle, and compare.

Tolerances (BASELINE.json north_star): bit-exact on tile/key indexing (radii, num_rendered,
point_list, ranges, n_contrib); float tensors within 1e-4 relative, implemented elementwise as
    images:     |a-b| <= 1e-4*|b| + 1e-5*max|b|
    gradients:  |a-b| <= 1e-4*|b| + 5e-5*max|b|
The absolute floor keeps near-cancelling entries from dominating: every gradient entry is a sum of thousands of
signed fp32 terms; the reference adds them with order-nondeterministic atomics (its own run-to-run spread is
~1e-6 of max|b|), we add them in a different (hierarchical) order.  Worst case over the test-suite so far:
1.4e-5 of max|b| (grad_scales with a non-zero background), i.e. 7x inside the 1e-4 bound.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "feature-3dgs_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import scenegen  # noqa: E402

RTOL = 1e-4
ATOL_REL = 1e-5
GRAD_ATOL_REL = 5e-5

INT_KEYS = ("radii", "num_rendered", "point_list", "ranges", "n_contrib")
FWD_FLOAT_KEYS = ("color", "feature_map", "depth", "final_T")
GRAD_KEYS = ("means3D", "means2D", "sh", "semantic_feature", "opacities", "scales", "rotations")


def _np(t):
    return t.detach().cpu().numpy()


def run_ours(scene, cam, device="cuda", grads=None, debug=False, colors_precomp=None, cov3D_precomp=None):
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer, _C

    t = scenegen.to_torch(scene, device, requires_grad=grads is not None)
    rs = GaussianRasterizationSettings(**scenegen.settings_kwargs(scene, cam, device, debug=debug))
    means2D = torch.zeros_like(t["means3D"], requires_grad=grads is not None)
    kw = dict(means3D=t["means3D"], means2D=means2D, opacities=t["opacities"],
              semantic_feature=t["semantic_feature"] if scene.C > 0 else None)
    if colors_precomp is None:
        kw["shs"] = t["shs"]
    else:
        kw["colors_precomp"] = torch.from_numpy(colors_precomp).to(device).requires_grad_(grads is not None)
    if cov3D_precomp is None:
        kw.update(scales=t["scales"], rotations=t["rotations"])
    else:
        kw["cov3D_precomp"] = torch.from_numpy(cov3D_precomp).to(device).requires_grad_(grads is not None)
    # direct _C call first to expose the internal buffers (same kernels as the autograd path)
    e = torch.Tensor([])
    sf = t["semantic_feature"] if scene.C > 0 else torch.empty(0, device=device)
    raw = _C.rasterize_gaussians(
        rs.bg, t["means3D"].detach(), e if colors_precomp is None else kw["colors_precomp"].detach(), sf.detach(),
        t["opacities"].detach(), e if cov3D_precomp is not None else t["scales"].detach(),
        e if cov3D_precomp is not None else t["rotations"].detach(), rs.scale_modifier,
        e if cov3D_precomp is None else kw["cov3D_precomp"].detach(), rs.viewmatrix, rs.projmatrix, rs.tanfovx,
        rs.tanfovy, rs.image_height, rs.image_width, e if colors_precomp is not None else t["shs"].detach(),
        rs.sh_degree, rs.campos, rs.prefiltered, rs.debug)
    R, color, feat, depth, radii, geom, binning, img = raw
    pl, ranges, ncontrib, final_T, rec = _C.debug_views(geom, binning, img, scene.P, cam.image_width,
                                                         cam.image_height, R)
    out = dict(num_rendered=np.int64(R), color=_np(color), feature_map=_np(feat), depth=_np(depth),
               radii=_np(radii), point_list=_np(pl).astype(np.int64), ranges=_np(ranges).astype(np.int64),
               n_contrib=_np(ncontrib).astype(np.int64), final_T=_np(final_T), rec=_np(rec))
    if grads is not None:
        color, feat, radii2, depth = GaussianRasterizer(rs)(**kw)
        gc, gf, gd = [torch.from_numpy(g).to(device) for g in grads]
        outs, gos = [color, depth], [gc, gd]
        if scene.C > 0:
            outs.append(feat)
            gos.append(gf)
        torch.autograd.backward(outs, gos)
        g = dict(means3D=_np(t["means3D"].grad), means2D=_np(means2D.grad), opacities=_np(t["opacities"].grad))
        if colors_precomp is None:
            g["sh"] = _np(t["shs"].grad)
        else:
            g["colors_precomp"] = _np(kw["colors_precomp"].grad)
        if cov3D_precomp is None:
            g["scales"], g["rotations"] = _np(t["scales"].grad), _np(t["rotations"].grad)
        else:
            g["cov3D_precomp"] = _np(kw["cov3D_precomp"].grad)
        if scene.C > 0:
            g["semantic_feature"] = _np(t["semantic_feature"].grad)
        out["grads"] = g
        out["color_autograd"] = _np(color)
    return out


def run_ref(scene, cam, device="cuda", grads=None):
    """Reference CUDA extension (oracle/_ref) on the same inputs."""
    import torch
    from oracle import ref_wrapper as rw

    C = scene.C
    t = scenegen.to_torch(scene, device, requires_grad=grads is not None)
    rs = scenegen.settings_kwargs(scene, cam, device)
    mod = rw.load(C)
    e = torch.Tensor([])
    sf = t["semantic_feature"] if C > 0 else torch.zeros(scene.P, 1, 1, device=device)
    raw = mod.rasterize_gaussians(rs["bg"], t["means3D"].detach(), e, sf.detach(), t["opacities"].detach(),
                                  t["scales"].detach(), t["rotations"].detach(), 1.0, e, rs["viewmatrix"],
                                  rs["projmatrix"], rs["tanfovx"], rs["tanfovy"], rs["image_height"],
                                  rs["image_width"], t["shs"].detach(), rs["sh_degree"], rs["campos"], False, False)
    R, color, feat, depth, radii, geom, binning, img = raw
    final_T, ncontrib, ranges = rw.parse_image_buffer(img, cam.image_width, cam.image_height)
    pl = rw.parse_binning_buffer(binning, R)
    out = dict(num_rendered=np.int64(R), color=_np(color), feature_map=_np(feat)[:C], depth=_np(depth),
               radii=_np(radii), point_list=_np(pl).astype(np.int64), ranges=_np(ranges).astype(np.int64),
               n_contrib=_np(ncontrib).astype(np.int64), final_T=_np(final_T))
    out["geom"] = {k: _np(v) for k, v in rw.parse_geom_buffer(geom, scene.P, C).items()}
    if grads is not None:
        means2D = torch.zeros_like(t["means3D"], requires_grad=True)
        rr = rw.RefRasterizer(rs, C)
        color, feat, _, depth = rr(means3D=t["means3D"], means2D=means2D, opacities=t["opacities"], shs=t["shs"],
                                   semantic_feature=t["semantic_feature"] if C > 0 else None, scales=t["scales"],
                                   rotations=t["rotations"])
        gc, gf, gd = [torch.from_numpy(g).to(device) for g in grads]
        outs, gos = [color, depth], [gc, gd]
        if C > 0:
            outs.append(feat)
            gos.append(gf)
        torch.autograd.backward(outs, gos)
        g = dict(means3D=_np(t["means3D"].grad), means2D=_np(means2D.grad), opacities=_np(t["opacities"].grad),
                 sh=_np(t["shs"].grad), scales=_np(t["scales"].grad), rotations=_np(t["rotations"].grad))
        if C > 0:
            g["semantic_feature"] = _np(t["semantic_feature"].grad)
        out["grads"] = g
    return out


def run_oracle(scene, cam, grads=None, threads=None, **kw):
    import oracle

    if threads:
        oracle.set_threads(threads)
    f = oracle.forward(scene, cam, **kw)
    out = dict(num_rendered=np.int64(f["num_rendered"]), color=f["color"], feature_map=f["feature_map"],
               depth=f["depth"], radii=f["radii"], point_list=f["point_list"].astype(np.int64),
               ranges=f["ranges"].astype(np.int64), n_contrib=f["n_contrib"].astype(np.int64),
               final_T=f["final_T"], fwd=f)
    if grads is not None:
        g = oracle.backward(scene, cam, f, *grads, **{k: v for k, v in kw.items() if k != "render"})
        out["grads"] = dict(means3D=g["means3D"], means2D=g["means2D"], opacities=g["opacities"], sh=g["sh"],
                            scales=g["scales"], rotations=g["rotations"], semantic_feature=g["semantic_feature"],
                            colors_precomp=g["colors"], cov3D_precomp=g["cov3D"])
    return out


def float_mismatch(a, b, rtol=RTOL, atol_rel=ATOL_REL):
    """-> (max violation ratio, max abs err, scale).  ratio <= 1 means within tolerance."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    if a.shape != b.shape:
        return float("inf"), float("inf"), 0.0
    if a.size == 0:
        return 0.0, 0.0, 0.0
    scale = float(np.max(np.abs(b)))
    err = np.abs(a - b)
    tol = rtol * np.abs(b) + atol_rel * scale + 1e-30
    bad = ~np.isfinite(a) | ~np.isfinite(b)
    ratio = float(np.max(np.where(bad, np.inf, err / tol)))
    return ratio, float(np.max(np.where(bad, np.inf, err))), scale


def compare(ours, ref, int_keys=INT_KEYS, float_keys=FWD_FLOAT_KEYS, grad_keys=GRAD_KEYS, rtol=RTOL,
            atol_rel=ATOL_REL, tie_tolerant=False):
    """-> dict report; report['ok'] is the overall verdict.

    tie_tolerant (CPU-oracle comparisons only): libm's expf differs from CUDA's by <= 2 ulp, so a pixel whose
    alpha or T lands within an ulp of the 1/255 or 1e-4 threshold can blend one Gaussian more or less.  Up to
    max(2, 1e-4 * pixels) such n_contrib mismatches are accepted; those pixels are masked out of the image
    comparison and, if any occurred, the gradient tolerance is widened 50x (a single flipped blend shows up in a
    few Gaussians' gradients).  The comparison against the reference CUDA build never uses this."""
    rep, ok = {}, True
    tie_mask, ties = None, 0
    for k in int_keys:
        a, b = np.asarray(ours[k]), np.asarray(ref[k])
        same = a.shape == b.shape and bool(np.array_equal(a, b))
        n_bad = int(np.sum(a != b)) if a.shape == b.shape else -1
        rep[k] = dict(exact=same, mismatches=n_bad, size=int(b.size))
        if k == "n_contrib" and tie_tolerant and not same and 0 < n_bad <= max(2, int(1e-4 * b.size)):
            tie_mask, ties = (a != b), n_bad
            rep[k]["accepted_ties"] = n_bad
            continue
        ok &= same
    for k in float_keys:
        a, b = np.asarray(ours[k]), np.asarray(ref[k])
        if tie_mask is not None and a.shape == b.shape and a.shape[-2:] == tie_mask.shape:
            a = np.where(tie_mask, b, a)
        r, e, s = float_mismatch(a, b, rtol, atol_rel)
        rep[k] = dict(ratio=r, max_abs_err=e, scale=s, bit_exact=bool(np.array_equal(ours[k], ref[k])))
        ok &= r <= 1.0
    if "grads" in ours and "grads" in ref:
        widen = 50.0 if ties else 1.0
        for k in grad_keys:
            if k in ours["grads"] and k in ref["grads"]:
                r, e, s = float_mismatch(ours["grads"][k], ref["grads"][k], rtol * widen, GRAD_ATOL_REL * widen)
                rep["grad_" + k] = dict(ratio=r, max_abs_err=e, scale=s)
                ok &= r <= 1.0
    rep["ok"] = bool(ok)
    return rep


RECORD_EXACT_KEYS = ("color", "depth", "final_T")  # bit-identical to the reference build
PIX_BLOCK = 64      # image moments: per 64 x 64-pixel block over all channels, and per channel over all pixels
GAUSS_BLOCK = 4096  # gradient moments: per block of 4096 Gaussians over all components, and per component


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _record_arrays(out):
    """name -> (array in its canonical dtype, is_float, absolute-tolerance floor) of one run_ours()/run_oracle() result."""
    arrs = {k: (np.asarray(out[k]).astype(np.int64), False, None) for k in INT_KEYS}
    arrs.update({k: (np.asarray(out[k], np.float32), True, ATOL_REL) for k in FWD_FLOAT_KEYS})
    for k, v in out.get("grads", {}).items():
        if k in GRAD_KEYS:
            arrs["grad_" + k] = (np.asarray(v, np.float32), True, GRAD_ATOL_REL)
    return arrs


def _moments(k, a):
    """float64 (count, sum x, sum |x|, sum x^2) of `a` in two groupings that each cover every element: images ([C,H,W] or
    [H,W]) per PIX_BLOCK x PIX_BLOCK pixels over all channels ("blk") and per channel over all pixels ("ch"); gradients
    ([P, ...]) per GAUSS_BLOCK Gaussians over all components ("blk") and per component over all Gaussians ("ch").
    -> {"blk": [4, blocks], "ch": [4, channels]}"""
    def four(v):
        return [np.ones_like(v), v, np.abs(v), v * v]

    if k.startswith("grad_"):
        x = a.reshape(a.shape[0], -1)
        starts = range(0, x.shape[0], GAUSS_BLOCK)
        blk, ch = np.zeros((4, len(starts))), np.zeros((4, x.shape[1]))
        for i, r in enumerate(starts):
            v = x[r:r + GAUSS_BLOCK].astype(np.float64)
            sums = np.stack([m.sum(axis=0) for m in four(v)])
            blk[:, i] = sums.sum(axis=1)
            ch += sums
        return {"blk": blk, "ch": ch}
    x = a.reshape((-1,) + a.shape[-2:])
    rows, cols = np.arange(0, x.shape[1], PIX_BLOCK), np.arange(0, x.shape[2], PIX_BLOCK)
    blk, ch = np.zeros((4, len(rows), len(cols))), np.zeros((4, x.shape[0]))
    for c in range(x.shape[0]):
        for j, m in enumerate(four(x[c].astype(np.float64))):
            blk[j] += np.add.reduceat(np.add.reduceat(m, rows, axis=0), cols, axis=1)
            ch[j, c] = m.sum()
    return {"blk": blk.reshape(4, -1), "ch": ch}


def make_record(ours, orc):
    """Compact stand-in for a full-size result.  From `ours` (this project's CUDA path, whose integer arrays and
    RECORD_EXACT_KEYS were asserted bit-identical to the reference build): the shape and SHA-256 of every array (integer
    arrays as int64, float arrays as float32).  From `orc` (the CPU oracle, the reference algorithm restated; see
    run_oracle): for every float array, max |b| over the whole array and the _moments() sums (float32)."""
    rec, bars = {}, _record_arrays(orc)
    for k, (a, is_float, _) in _record_arrays(ours).items():
        rec["shape_" + k] = np.asarray(a.shape, np.int64)
        rec["sha256_" + k] = np.asarray(_digest(a))
        if is_float and a.size:
            b = bars[k][0]
            assert b.shape == a.shape, (k, b.shape, a.shape)
            rec["scale_" + k] = np.float64(np.max(np.abs(b)))
            for g, m in _moments(k, b).items():
                rec[f"{g}_{k}"] = m[1:].astype(np.float32)
    return rec


def check_record(ours, rec):
    """Compare one run_ours() result with a make_record() record.  Integer arrays and RECORD_EXACT_KEYS must have the
    recorded digest (bit-identical over the whole array).  Every float array must satisfy, in every block and channel of
    _moments(), the bounds that the elementwise bar of compare(), |a-b| <= r|b| + q with r = RTOL and q = floor * max|b|,
    implies for sums over the n elements of a block:
        |sum a - sum b|, |sum |a| - sum |b||  <=  r sum|b| + n q
        |sum a^2 - sum b^2|                   <=  (2r + r^2) sum b^2 + 2 (1 + r) q sum|b| + n q^2
    (each widened by 2^-23 of its recorded magnitude for the float32 storage), so a result within the elementwise bar
    always passes, while a wrong tile, channel or block of Gaussians shows up in its sums.
    -> list of failure messages (empty: pass)."""
    bad = []
    arrs = _record_arrays(ours)
    for k in (n[len("shape_"):] for n in rec.files if n.startswith("shape_")):
        if k not in arrs:
            bad.append(f"{k}: missing from the result")
            continue
        a, is_float, atol_rel = arrs[k]
        want_shape = tuple(int(s) for s in rec["shape_" + k])
        if a.shape != want_shape:
            bad.append(f"{k}: shape {a.shape} != recorded {want_shape}")
            continue
        if (not is_float or k in RECORD_EXACT_KEYS) and _digest(a) != str(rec["sha256_" + k]):
            bad.append(f"{k}: not bit-identical to the record")
        if not (is_float and ("blk_" + k) in rec.files):
            continue
        r, q, eps = RTOL, atol_rel * float(rec["scale_" + k]), 2.0 ** -23
        for g, (n, s1, sa, s2) in _moments(k, a).items():
            b1, ba, b2 = rec[f"{g}_{k}"].astype(np.float64)
            t1 = r * ba + n * q + eps * ba + 1e-30
            t2 = (2 * r + r * r) * b2 + 2 * (1 + r) * q * ba + n * q * q + eps * b2 + 1e-30
            viol = np.max(np.stack([np.abs(s1 - b1) / t1, np.abs(sa - ba) / t1, np.abs(s2 - b2) / t2]), axis=0)
            worst = int(np.argmax(np.where(np.isfinite(viol), viol, np.inf)))
            if not np.all(np.isfinite(viol)) or viol[worst] > 1.0:
                bad.append(f"{k}: {g} sums outside the bar, worst {float(viol[worst]):.3g} at {g} {worst} of {viol.size}")
    return bad


def format_report(rep):
    lines = []
    for k, v in rep.items():
        if k == "ok":
            continue
        if "exact" in v:
            t = f" (accepted threshold ties: {v['accepted_ties']})" if "accepted_ties" in v else ""
            lines.append(f"  {k:22s} exact={v['exact']} mismatches={v['mismatches']}/{v['size']}{t}")
        else:
            extra = f" bit_exact={v['bit_exact']}" if "bit_exact" in v else ""
            lines.append(f"  {k:22s} viol={v['ratio']:.3g} max_abs_err={v['max_abs_err']:.3g} scale={v['scale']:.3g}{extra}")
    lines.append(f"  OK={rep['ok']}")
    return "\n".join(lines)
