"""GPU tests of the binning at every image size whose code path differs, and of every render variant per Gaussian.

  * Binning (test_binning_shape_sweep): one synthetic cloud at image sizes chosen by the branch of tile_binning.cu /
    binning.cu they take -- 1 tile (single radix pass, plain copy), 2-3 tiles (1-bit digits), a tall 1 x 260 grid,
    the largest grid whose 2-D prefix fits shared memory and the first one that needs the global scratch, UHD (8+7
    bit digits, 2 difference-array replicas), 256 x 255 tiles (8+8 bits, 1 replica), 65536 tiles (CUB with 32-bit
    keys) and 32-bit keys forced on a mid-size frame. tiles_touched, R, ranges and point_list must equal
    tests/util.bin_reference (a numpy restatement, itself checked against the CPU oracle in test_oracle_kat.py) bit
    for bit, for both binning implementations and both depth orders; forward variants 1-5 must be bit-identical to
    variant 0 (no sub-block culling); the default backward must agree with variant 0 per Gaussian.
  * Backward (test_backward_variants_per_gaussian): every render_bwd variant on an adversarial scene
    (util.adversarial_scene), per Gaussian against the fp64 CPU oracle and against variant 0.

Every test here runs with the options at their compiled defaults unless it sets one through util.kernel_options;
the module fixture asserts that on entry and on exit.
"""
import numpy as np
import pytest
import torch

from gaussianeditor_b200 import synth
from oracle import cpu_oracle
from util import (OPTION_DEFAULTS, adversarial_scene, axis_camera, bin_reference, get_option, kernel_options,
                  run_ours)

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, scope="module")
def options_at_compiled_defaults():
    """Earlier tests must not leak kernel options into these, and these must not leak any."""
    assert {k: get_option(k) for k in OPTION_DEFAULTS} == OPTION_DEFAULTS
    yield
    assert {k: get_option(k) for k in OPTION_DEFAULTS} == OPTION_DEFAULTS


# ---- per-row comparison ---------------------------------------------------------------------------------------
# Each check bounds the error of row i (one Gaussian's gradient) by
#     || g_i - want_i ||  <=  a * || f_i - e_i ||  +  b * || e_i ||  +  c * max_j || e_j ||
# with e the fp64 oracle and f the fp32 oracle (or, without an oracle, e = f = variant 0's result). (a, b, c) were
# calibrated on a B200 (1000 W power limit) with the unmodified kernels; the worst observed ratio of the left side to
# the right side is given with each. DIRECT are the gradients render_bwd produces (plus dsh, one linear step on);
# CHAIN = dmean3D, dscale, drot go through the 2-D -> 3-D chain rule, whose fp32 cancellation amplifies the order of the
# float atomics -- two runs of the SAME variant differ there by up to 0.4 % of the largest row.
DIRECT = ("dmean2D", "dopacity", "dcolor", "dsh")
TOL_FP64 = {"direct": (4.0, 1e-5, 1e-4),      # worst ratio 0.47 (after the allowed flips)
            "chain": (4.0, 1e-5, 1.2e-3)}     # worst ratio 0.56
TOL_VARIANT = {"direct": (4.0, 1e-5, 2e-7),   # worst ratio 0.65
               "chain": (4.0, 1e-5, 1e-2)}    # worst ratio 0.68
TOL_SELF = (0.0, 1e-5, 1e-4)                  # default vs variant 0 without an oracle, frames up to 4096^2: 0.34


def _tol(table, k):
    return table["direct" if k in DIRECT else "chain"]


def _rows(x):
    a = np.asarray(x.detach().cpu().numpy() if torch.is_tensor(x) else x, np.float64)
    return a.reshape(len(a), -1)


def row_terms(g, want, e, f):
    """(||g_i - want_i||, ||f_i - e_i||, ||e_i||, max_j ||e_j||) of row-major gradient arrays."""
    g, want, e, f = _rows(g), _rows(want), _rows(e), _rows(f)
    n = np.linalg.norm(e, axis=1)
    return np.linalg.norm(g - want, axis=1), np.linalg.norm(f - e, axis=1), n, float(n.max())


def failing_rows(terms, tol):
    d, ferr, n, nmax = terms
    a, b, c = tol
    return np.flatnonzero(d > a * ferr + b * n + c * nmax)


def signed_dL(H, W, seed):
    """Standard normal dL/dpixel with a zeroed block and channel 1 scaled by 10^3."""
    dL = np.random.default_rng(seed).standard_normal((3, H, W)).astype(np.float32)
    dL[:, H // 4:H // 2, W // 4:W // 2] = 0.0
    dL[1] *= 1e3
    return dL


GRADS_SH = ("dmean2D", "dopacity", "dsh", "dmean3D", "dscale", "drot")
GRADS_COLORS = ("dmean2D", "dopacity", "dcolor", "dmean3D", "dscale", "drot")


def _grad(out_grads, k):
    g = out_grads[k]
    return g[:, :2] if k == "dmean2D" else g


# ---- binning across image sizes -------------------------------------------------------------------------------
_CLOUD = {}


def sweep_cloud():
    if "c3" not in _CLOUD:
        _CLOUD["c3"] = synth.make_config("c3", P=150_000)[0]
    return _CLOUD["c3"]


def ours_binning(out):
    v = out["views"]
    u32 = lambda t: t.cpu().numpy().view(np.uint32)
    return dict(tiles_touched=u32(v["tiles_touched"]), R=out["R"], ranges=u32(v["ranges"]),
                point_list=u32(v["point_list"]))


def reference_binning(out, W, H):
    """util.bin_reference on this forward's own records: centres, radii and view-depth bit patterns."""
    rec = out["views"]["records"].cpu().numpy()
    return bin_reference(rec[:, 0:2], out["radii"].cpu().numpy(), rec[:, 6], W, H)


def assert_binning_equal(got, want, what):
    assert got["R"] == want["R"], (what, got["R"], want["R"])
    for k in ("tiles_touched", "ranges", "point_list"):
        assert got[k].shape == want[k].shape and np.array_equal(got[k], want[k]), (what, k)


# (W, H, options): the first size at which each branch is taken
SHAPES = [
    (1, 1, {}), (7, 5, {}), (16, 16, {}),   # one tile: a single 1-bit radix pass and the plain copy (bits2 == 0)
    (17, 16, {}), (48, 16, {}),             # 2 and 3 tiles: two 1-bit passes
    (64, 64, {}),                           # 16 tiles: 3 + 2 bits
    (16, 4160, {}),                         # one tile column, 260 rows
    (1600, 1600, {}),                       # (gx+1)(gy+1) = 10201: the last grid whose prefix fits shared memory
    (1616, 1600, {}),                       # 10302 entries: tile_prefix_kernel on the global scratch
    (3840, 2160, {}),                       # 32400 tiles: 8 + 7 bits, 2 difference-array replicas
    (4096, 4080, {}),                       # 65280 tiles: 8 + 8 bits, 1 replica
    (4096, 4096, {}),                       # 65536 tiles: CUB sort with 32-bit keys
    (640, 400, dict(tile_key_bits=32)),     # 32-bit keys forced
]


@pytest.mark.parametrize("W,H,opts", SHAPES, ids=[f"{w}x{h}{'-u32' if o else ''}" for w, h, o in SHAPES])
def test_binning_shape_sweep(W, H, opts):
    cloud = sweep_cloud()
    cam = synth.ring_cameras(8, 4.5, 15.0, W, H, 61.0)[3]
    bg = (0.3, 0.2, 0.1)
    with kernel_options(**opts):
        base = run_ours(cloud, cam, bg)
        want = reference_binning(base, W, H)
        assert want["R"] > 0
        assert_binning_equal(ours_binning(base), want, "default")
        for bv, dv in ((0, 0), (1, 1), (0, 1)):
            with kernel_options(binning_variant=bv, depth_sort_variant=dv):
                assert_binning_equal(ours_binning(run_ours(cloud, cam, bg)), want, ("binning", bv, "depth", dv))
        # forward variants: bit-identical to the CTA-per-tile kernel, which culls nothing per sub-block
        with kernel_options(render_fwd_variant=0):
            ref = run_ours(cloud, cam, bg)
        for fv in (1, 2, 3, 4, 5):
            with kernel_options(render_fwd_variant=fv):
                out = run_ours(cloud, cam, bg)
            for k in ("color", "depth"):
                assert torch.equal(out[k], ref[k]), (fv, k)
            for k in ("n_contrib", "final_T"):
                assert torch.equal(out["views"][k], ref["views"][k]), (fv, k)
        # backward: the default variant against variant 0, per Gaussian
        dL = signed_dL(H, W, seed=W * 7 + H)
        with kernel_options(render_bwd_variant=0):
            g0 = run_ours(cloud, cam, bg, dL=dL)["grads"]
        g = run_ours(cloud, cam, bg, dL=dL)["grads"]
        for k in GRADS_SH:
            e = _grad(g0, k)
            bad = failing_rows(row_terms(_grad(g, k), e, e, e), TOL_SELF)
            assert len(bad) == 0, (k, bad[:10])


def test_speculative_binning_at_uhd():
    """At 3840x2160 (the 8+7-bit radix passes) the sync-free forward gives the exact path's bits, with a good
    capacity guess and with a hopeless one that forces the redo."""
    import gaussianeditor_b200.rasterizer as RZ
    cloud = sweep_cloud()
    W, H = 3840, 2160
    cam = synth.ring_cameras(8, 4.5, 15.0, W, H, 61.0)[6]
    key = (0, cloud.means3D.shape[0], W, H)
    try:
        RZ.SPECULATIVE = False
        exact = run_ours(cloud, cam, (0.5, 0.5, 0.5))
        RZ.SPECULATIVE = True
        RZ._r_hint[key] = exact["R"]
        spec = run_ours(cloud, cam, (0.5, 0.5, 0.5))
        assert spec["state"].cap > spec["R"] == exact["R"]
        RZ._r_hint[key] = 10
        redo = run_ours(cloud, cam, (0.5, 0.5, 0.5))
        assert redo["state"].cap == redo["R"] == exact["R"]
        assert_binning_equal(ours_binning(exact), reference_binning(exact, W, H), "exact")
        for other in (spec, redo):
            assert torch.equal(other["color"], exact["color"]) and torch.equal(other["depth"], exact["depth"])
            for k in ("point_list", "ranges", "n_contrib", "final_T"):
                assert torch.equal(other["views"][k], exact["views"][k]), k
    finally:
        RZ.SPECULATIVE = True
        RZ._r_hint.pop(key, None)


# ---- every backward variant, per Gaussian, on an adversarial scene ----------------------------------------------
BWD_VARIANTS = list(range(15))
BG = (0.3, 0.6, 0.1)


def adversarial_case(W, H, path):
    cloud, cls = adversarial_scene()
    cam = axis_camera(W, H)
    cp = None
    if path == "colors":
        cp = np.random.default_rng(5).uniform(-0.2, 1.2, (cloud.means3D.shape[0], 3)).astype(np.float32)
    return cloud, cls, cam, cp, signed_dL(H, W, seed=11)


def oracle_grads(cloud, cam, cp, dL, f32):
    f = cpu_oracle.forward_from(cloud, cam, BG, f32=f32, colors_precomp=cp)
    g = f.backward(dL)
    f.close()
    return g


def assert_classes_present(out, cls, W, H):
    """Each splat class of the adversarial scene is on screen, in the form it was made for."""
    radii = out["radii"].cpu().numpy()
    rec = out["views"]["records"].cpu().numpy().astype(np.float64)
    vis = radii > 0
    A, B, C = rec[:, 2], rec[:, 3], rec[:, 4]
    tr, det = A + C, A * C - B * B
    disc = np.sqrt(np.maximum(tr * tr / 4 - det, 0))
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.sqrt((tr / 2 + disc) / (tr / 2 - disc))        # axis ratio of the projected ellipse
    n = cls["needle"]
    assert np.sum(vis[n] & (ratio[n] >= 100)) >= 10 and radii[n].max() >= 100
    assert np.sum(radii[cls["huge"]] >= max(W, H) // 2) >= 3
    assert np.sum(vis[cls["subpixel"]]) >= 100
    o = cls["offscreen"]
    ndc = np.stack([(2 * rec[o, 0] + 1) / W - 1, (2 * rec[o, 1] + 1) / H - 1], 1)
    assert np.sum(vis[o] & (np.abs(ndc).max(1) > 1.15)) >= 20
    d = rec[cls["equal_depth"], 6][vis[cls["equal_depth"]]]
    assert len(d) - len(np.unique(d)) >= 50
    assert np.sum(vis[cls["opacity_1_255"]]) >= 50 and np.sum(vis[cls["opacity_high"]]) >= 50
    assert np.sum(out["views"]["clamped"].cpu().numpy()[cls["negative_colour"]] != 0) >= 100
    # the T < 1e-4 stop inside a tile: a saturated pixel next to an unsaturated one in the same 16x16 tile
    T = out["views"]["final_T"].cpu().numpy()
    Tp = np.pad(T, ((0, -H % 16), (0, -W % 16)), constant_values=np.nan).reshape(-(-H // 16), 16, -(-W // 16), 16)
    assert np.any((np.nanmin(Tp, axis=(1, 3)) < 1e-3) & (np.nanmax(Tp, axis=(1, 3)) > 0.05))


def variant_grads(cloud, cam, cp, dL, v, **opts):
    with kernel_options(render_bwd_variant=v, **opts):
        return run_ours(cloud, cam, BG, dL=dL, colors_precomp=cp)


@pytest.mark.parametrize("W,H", [(333, 201), (7, 5)])
@pytest.mark.parametrize("path", ["sh", "colors"])
def test_backward_variants_per_gaussian(W, H, path):
    """All 15 render_bwd variants, Gaussian by Gaussian, on util.adversarial_scene with a signed dL/dpixel (zeroed
    block, one channel x 10^3) and a nonzero background, through the SH path and the colors_precomp path (which
    exposes render_bwd's dL/dcolour directly).

    Against fp64 truth, with TOL_FP64: at most max(2, 1e-4 V) rows of V visible may fail -- a pixel whose alpha sits
    on the 1/255 or T contour can be decided differently with and without FMA contraction. Against variant 0, with
    TOL_VARIANT: no row may fail (all variants make the same hit decisions and differ in summation order only).
    preprocess_variant 0 (plain loads of the SH rows) must give the same records bit for bit, and the gradients
    within TOL_VARIANT of the default.

    Calibration (B200, unmodified kernels, all four cases, 15 variants, 6 gradient arrays): the constants and the worst
    observed ratios are listed with TOL_FP64 / TOL_VARIANT. At most one row per array exceeded the fp64 bound (the
    allowance is 2)."""
    cloud, cls, cam, cp, dL = adversarial_case(W, H, path)
    names = GRADS_SH if path == "sh" else GRADS_COLORS
    e = oracle_grads(cloud, cam, cp, dL, f32=False)
    f = oracle_grads(cloud, cam, cp, dL, f32=True)
    outs = {v: variant_grads(cloud, cam, cp, dL, v) for v in BWD_VARIANTS}
    if path == "sh" and W == 333:
        assert_classes_present(outs[14], cls, W, H)
    V = int((outs[14]["radii"] > 0).sum())
    assert V > 0
    allowed = max(2, int(1e-4 * V))
    report = []
    for v in BWD_VARIANTS:
        g = outs[v]["grads"]
        for k in names:
            ek, fk = e[k], f[k]
            if k == "dmean2D":
                ek, fk = ek[:, :2], fk[:, :2]
            bad = failing_rows(row_terms(_grad(g, k), ek, ek, fk), _tol(TOL_FP64, k))
            report.append((v, k, bad.tolist()))
            assert len(bad) <= allowed, (v, k, bad[:20])
            bad0 = failing_rows(row_terms(_grad(g, k), _grad(outs[0]["grads"], k), ek, fk), _tol(TOL_VARIANT, k))
            assert len(bad0) == 0, (v, k, bad0[:20])
    flips = sorted({i for _, _, b in report for i in b})
    print(f"{W}x{H} {path}: {len(flips)} rows off the fp64 bound in some variant: {flips[:20]}")
    # preprocess_variant 0 against the default (1)
    p0 = variant_grads(cloud, cam, cp, dL, OPTION_DEFAULTS["render_bwd_variant"], preprocess_variant=0)
    p1 = outs[OPTION_DEFAULTS["render_bwd_variant"]]
    vis = p1["radii"] > 0        # a culled record defines nothing but its radius
    assert torch.equal(p0["radii"], p1["radii"]) and torch.equal(p0["views"]["records"][vis], p1["views"]["records"][vis])
    assert torch.equal(p0["color"], p1["color"])
    for k in names:
        ek, fk = e[k], f[k]
        if k == "dmean2D":
            ek, fk = ek[:, :2], fk[:, :2]
        bad = failing_rows(row_terms(_grad(p0["grads"], k), _grad(p1["grads"], k), ek, fk), _tol(TOL_VARIANT, k))
        assert len(bad) == 0, ("preprocess_variant 0", k, bad[:20])
