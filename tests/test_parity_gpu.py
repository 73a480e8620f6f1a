"""GPU parity tests (run on the B200 box: ``pytest -m gpu``). Everything goes through the public
GaussianRasterizer API -> ctypes -> C ABI (include/gsr_b200.h) -> sm_100a kernels.

Checkers (test infrastructure only):
  * the reference's own CUDA sources compiled unmodified (oracle/_ref/libdgr_ref.so): integer outputs
    (radii, R, tile ranges, sorted point list, n_contrib) must be BIT-EXACT, images bit-exact, gradients to
    tolerance (the reference's float atomics are themselves order-dependent). What each test compares against is
    stored under tests/golden/reference/ (see RefGolden), so the tests need no reference build;
  * oracle/liboracle_cpu.so -- the CPU restatement (fp32 mirror and fp64 truth).
Tolerances are the ones SURVEY.md 8(a) fixes.

Re-recording the stored reference outputs (GPU, oracle/_ref built with `make -C oracle ref REF=<reference's
diff-gaussian-rasterization directory>`):
    GSR_RECORD_REFERENCE_DIR=<dir> python -m pytest -m gpu tests/test_parity_gpu.py
compares every test with the live reference and writes <dir>/<case>.npz; copy those to tests/golden/reference/.
"""
import hashlib
import os
import zlib

import numpy as np
import pytest
import torch

from gaussianeditor_b200 import synth, _lib
from oracle import cpu_oracle, ref_cuda
from util import run_ours, rel_l2, cloud_tensors, settings_from, kernel_options

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RECORD_DIR = os.environ.get("GSR_RECORD_REFERENCE_DIR")


def _canon(x):
    """Array in a dtype-independent canonical form: integers as int64, float32 with -0.0 folded into +0.0 (the
    comparison is torch.equal's, which treats them as equal)."""
    a = np.asarray(x.detach().cpu().numpy() if torch.is_tensor(x) else x)
    if a.dtype.kind in "biu":
        return np.ascontiguousarray(a, np.int64)
    assert a.dtype == np.float32, a.dtype
    return np.ascontiguousarray(a + np.float32(0.0))


def _digest(a):
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).digest()


def _f64(x):
    return np.asarray(x.detach().cpu().numpy() if torch.is_tensor(x) else x, np.float64)


class RefGolden:
    """What the reference's own CUDA build produced for one test case.

    Recording (GSR_RECORD_REFERENCE_DIR set): `run()` executes oracle/_ref, each comparison is made against that live
    result, and what it compared against is written to <dir>/<case>.npz. Otherwise the stored values are read from
    tests/golden/reference/<case>.npz: bit-exact arrays as SHA-256 digests, tolerance-compared arrays as ROWS rows
    (seeded, among the rows where the reference is nonzero), small values in full. The `ref` arguments below map the
    live outputs to the value compared; they are only called while recording."""
    ROWS = 64

    def __init__(self, case, run):
        self.case = case
        if RECORD_DIR:
            self.live, self.z = run(), {}
        else:
            path = os.path.join(GOLDEN_DIR, case + ".npz")
            assert os.path.exists(path), f"{path} missing: record it as the module docstring says"
            with np.load(path) as z:
                self.live, self.z = None, dict(z)

    def same(self, key, ours, ref):
        """Bit-exact equality of `ours` with the reference's value."""
        a = _canon(ours)
        if self.live is not None:
            want = _canon(ref(self.live))
            assert a.shape == want.shape and np.array_equal(a, want), (self.case, key)
            self.z[key] = np.frombuffer(_digest(want), np.uint8)
        assert _digest(a) == self.z[key].tobytes(), (self.case, key)

    def rows(self, key, ours, ref):
        """(ours, reference) in float64 on the stored rows of the first axis, each row flattened."""
        if self.live is not None:
            want = _f64(ref(self.live))
            want = want.reshape(len(want), -1)
            nz = np.flatnonzero(np.abs(want).sum(1) > 0)
            rng = np.random.default_rng(zlib.crc32(key.encode()))
            idx = np.sort(rng.choice(nz, min(len(nz), self.ROWS), replace=False))
            self.z[key + "@rows"] = idx.astype(np.int32)
            self.z[key] = want[idx].astype(np.float32)
        a = _f64(ours)
        a = a.reshape(len(a), -1)[self.z[key + "@rows"]]
        assert a.shape == self.z[key].shape, (self.case, key)
        return a, self.z[key].astype(np.float64)

    def value(self, key, ref):
        """A small value (scalar or array) stored in full."""
        if self.live is not None:
            v = ref(self.live)
            self.z[key] = np.asarray(v.detach().cpu().numpy() if torch.is_tensor(v) else v)
        return self.z[key]

    def save(self):
        os.makedirs(RECORD_DIR, exist_ok=True)
        np.savez_compressed(os.path.join(RECORD_DIR, self.case + ".npz"), **self.z)


@pytest.fixture
def reference():
    made = []

    def make(case, run):
        made.append(RefGolden(case, run))
        return made[-1]
    yield make
    if RECORD_DIR:
        for g in made:
            g.save()


def _ref_run(cloud, cam, bg, dL=None, colors_precomp=None, scale_modifier=1.0):
    dev = "cuda"
    ct = cloud_tensors(cloud, dev)
    rs = settings_from(cam, bg, cloud.sh_degree, dev, scale_modifier)
    R = ref_cuda.ReferenceRasterizer()
    cp = None if colors_precomp is None else torch.from_numpy(colors_precomp).to(dev)
    common = dict(means3D=ct["means3D"], shs=None if cp is not None else ct["shs"], colors_precomp=cp,
                  scales=ct["scales"], rotations=ct["rotations"], cov3D_precomp=None, bg=rs.bg,
                  viewmatrix=rs.viewmatrix, projmatrix=rs.projmatrix, campos=rs.campos, tanfovx=rs.tanfovx,
                  tanfovy=rs.tanfovy, sh_degree=cloud.sh_degree, scale_modifier=scale_modifier)
    color, radii, depth, nr = R.forward(opacities=ct["opacities"], image_height=cam.image_height,
                                        image_width=cam.image_width, **common)
    out = dict(color=color, radii=radii, depth=depth, R=nr, state=R.state())
    if dL is not None:
        out["grads"] = R.backward(dL_dcolor=torch.from_numpy(dL).to(dev), radii=radii, R=nr, **common)
    torch.cuda.synchronize()
    return out


def _small_cases():
    c1, cams1 = synth.make_config("c1")
    c3, cams3 = synth.make_config("c3", P=60_000)
    cam3 = synth.ring_cameras(8, 4.5, 15.0, 400, 304, 61.0)[2]   # H not a multiple of 16*? 304 = 19*16; W 400 = 25*16
    cam_odd = synth.ring_cameras(8, 4.5, 15.0, 333, 201, 61.0)[5]  # partial last tile row and column
    return [("c1", c1, cams1[0], (0.0, 0.0, 0.0)), ("c3s", c3, cam3, (1.0, 1.0, 1.0)),
            ("c3odd", c3, cam_odd, (0.2, 0.5, 0.7))]


@pytest.mark.parametrize("fwd_variant", [0, 1, 2, 3, 4, 5])
def test_forward_matches_reference_cuda_bit_exact(fwd_variant, reference):
    with kernel_options(render_fwd_variant=fwd_variant):
        for name, cloud, cam, bg in _small_cases():
            ours = run_ours(cloud, cam, bg)
            ref = reference("forward_" + name, lambda: _ref_run(cloud, cam, bg))
            v = ours["views"]
            ref.same("R", ours["R"], lambda L: L["R"])
            ref.same("radii", ours["radii"], lambda L: L["radii"])
            for k in ("tiles_touched", "ranges", "point_list", "n_contrib", "final_T"):
                ref.same(k, v[k], lambda L: L["state"][k])
            ref.same("color", ours["color"], lambda L: L["color"])
            ref.same("depth", ours["depth"], lambda L: L["depth"])
            vis = ours["radii"] > 0
            rec = v["records"][vis]
            ref.same("means2D", rec[:, 0:2], lambda L: L["state"]["means2D"][vis])
            ref.same("conic_opacity", rec[:, [2, 3, 4, 5]], lambda L: L["state"]["conic_opacity"][vis])
            ref.same("depths", rec[:, 6], lambda L: L["state"]["depths"][vis])
            ref.same("rgb", rec[:, 8:11], lambda L: L["state"]["rgb"][vis])


@pytest.mark.parametrize("bwd_variant", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14])
def test_backward_matches_reference_cuda(bwd_variant, reference):
    with kernel_options(render_bwd_variant=bwd_variant):
        for name, cloud, cam, bg in _small_cases():
            rng = np.random.default_rng(7)
            dL = rng.uniform(size=(3, cam.image_height, cam.image_width)).astype(np.float32)
            ours = run_ours(cloud, cam, bg, dL=dL)
            # two runs: the second gives the reference's own run-to-run noise floor
            ref = reference("backward_" + name, lambda: [_ref_run(cloud, cam, bg, dL=dL) for _ in range(2)])
            pairs = [("dmean3D", "dL_dmeans3D"), ("dmean2D", "dL_dmeans2D"), ("dopacity", "dL_dopacity"),
                     ("dscale", "dL_dscales"), ("drot", "dL_drotations"), ("dsh", "dL_dsh")]
            for a, b in pairs:
                g, r = ref.rows(b, ours["grads"][a], lambda L: L[0]["grads"][b])
                noise = float(ref.value(b + "_noise", lambda L: rel_l2(_f64(L[1]["grads"][b]), _f64(L[0]["grads"][b]))))
                r_max = float(ref.value(b + "_absmax", lambda L: float(L[0]["grads"][b].abs().max())))
                err = rel_l2(g, r)
                assert err <= 1e-4 + 10 * noise, (name, a, err, noise)
                assert np.abs(g - r).max() <= 1e-3 * r_max + 1e-12, (name, a)


def test_forward_backward_vs_cpu_oracle():
    for name, cloud, cam, bg in _small_cases()[:2]:
        rng = np.random.default_rng(3)
        dL = rng.uniform(size=(3, cam.image_height, cam.image_width)).astype(np.float32)
        ours = run_ours(cloud, cam, bg, dL=dL)
        f = cpu_oracle.forward_from(cloud, cam, bg)
        radii = ours["radii"].cpu().numpy()
        # FMA contraction on the GPU vs none on the CPU: allow <= 1e-4 of the Gaussians to differ by a radius step
        assert (radii != f.radii).mean() <= 1e-4, name
        tiles = ours["views"]["tiles_touched"].cpu().numpy().astype(np.uint32)
        assert (tiles != f.tiles_touched).mean() <= 1e-4, name
        if np.array_equal(radii, f.radii) and np.array_equal(tiles, f.tiles_touched):
            assert ours["R"] == f.num_rendered
            assert np.array_equal(ours["views"]["ranges"].cpu().numpy().astype(np.uint32), f.ranges)
        col = ours["color"].cpu().numpy()
        assert np.mean(np.abs(col - f.color) > 1e-5 + 1e-4 * np.abs(f.color)) <= 1e-4, name
        g = f.backward(dL)
        for a, b in [("dmean3D", "dmean3D"), ("dmean2D", "dmean2D"), ("dopacity", "dopacity"), ("dscale", "dscale"),
                     ("drot", "drot"), ("dsh", "dsh")]:
            assert rel_l2(ours["grads"][a].cpu().numpy(), g[b]) <= 2e-4, (name, a)
        f.close()


def test_precomputed_colors_and_scale_modifier(reference):
    cloud, cams = synth.make_config("c2", P=20_000)
    cam = synth.look_at_camera((0, 0, -3.5), (0, 0, 0), (0, -1, 0), 320, 240, fovy_deg=50.0)
    rng = np.random.default_rng(11)
    cp = rng.uniform(size=(cloud.means3D.shape[0], 3)).astype(np.float32)
    dL = rng.uniform(size=(3, 240, 320)).astype(np.float32)
    ours = run_ours(cloud, cam, (0, 0, 0), dL=dL, colors_precomp=cp, scale_modifier=0.7)
    ref = reference("colors_precomp_c2",
                    lambda: _ref_run(cloud, cam, (0, 0, 0), dL=dL, colors_precomp=cp, scale_modifier=0.7))
    ref.same("radii", ours["radii"], lambda L: L["radii"])
    ref.same("color", ours["color"], lambda L: L["color"])
    assert rel_l2(*ref.rows("dL_dcolors", ours["grads"]["dcolor"], lambda L: L["grads"]["dL_dcolors"])) <= 1e-4
    assert rel_l2(*ref.rows("dL_dmeans3D", ours["grads"]["dmean3D"], lambda L: L["grads"]["dL_dmeans3D"])) <= 1e-4


def test_edge_cases_empty_and_all_culled():
    dev = "cuda"
    cam = synth.look_at_camera((0, 0, -3.5), (0, 0, 0), (0, -1, 0), 64, 48, fovy_deg=50.0)
    empty = synth.Cloud(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 4), np.float32),
                        np.zeros((0, 1), np.float32), np.zeros((0, 1, 3), np.float32), 0)
    out = run_ours(empty, cam, (0.3, 0.2, 0.1))
    assert out["R"] == 0 and out["color"].abs().sum().item() == 0.0  # rasterize_points.cu:72: outputs stay zero
    # every Gaussian behind the camera -> background only, zero gradients
    c, _ = synth.make_config("c1", P=500)
    c.means3D[:, 2] = -10.0
    dL = np.ones((3, 48, 64), np.float32)
    out = run_ours(c, cam, (0.3, 0.2, 0.1), dL=dL)
    assert out["R"] == 0 and int((out["radii"] > 0).sum()) == 0
    assert torch.allclose(out["color"][0], torch.full((48, 64), 0.3, device=dev))
    for k, g in out["grads"].items():
        if g is not None:
            assert float(g.abs().sum()) == 0.0, k


def _ref_apply_weights(ct, rs, mask, CH):
    P = ct["means3D"].shape[0]
    H, W = mask.shape[1:]
    w = torch.zeros(P, CH, device="cuda"); c = torch.zeros(P, 1, dtype=torch.int32, device="cuda")
    ref_cuda.ReferenceRasterizer().apply_weights(
        means3D=ct["means3D"], opacities=ct["opacities"], scales=ct["scales"], rotations=ct["rotations"], weights=w,
        cnt=c, image_weights=mask, bg=rs.bg, viewmatrix=rs.viewmatrix, projmatrix=rs.projmatrix, campos=rs.campos,
        tanfovx=rs.tanfovx, tanfovy=rs.tanfovy, image_height=H, image_width=W)
    torch.cuda.synchronize()
    return dict(weights=w, cnt=c)


def test_mark_visible_and_apply_weights_match_reference(reference):
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    dev = "cuda"
    cloud, cams = synth.make_config("c3", P=30_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 256, 192, 61.0)[1]
    ct = cloud_tensors(cloud, dev)
    rs = settings_from(cam, (0, 0, 0), 0, dev)
    rast = GaussianRasterizer(rs)
    vis = rast.markVisible(ct["means3D"])
    P = ct["means3D"].shape[0]
    rng = np.random.default_rng(5)
    mask = torch.from_numpy((rng.uniform(size=(1, 192, 256)) > 0.5).astype(np.float32)).to(dev)
    w1 = torch.zeros(P, 1, device=dev); c1 = torch.zeros(P, 1, dtype=torch.int32, device=dev)
    rast.apply_weights(ct["means3D"], None, ct["opacities"], None, w1, ct["scales"], ct["rotations"], None, c1, mask)
    torch.cuda.synchronize()
    ref = reference("mark_visible_apply_weights", lambda: dict(
        visible=ref_cuda.ReferenceRasterizer().mark_visible(ct["means3D"], rs.viewmatrix, rs.projmatrix),
        **_ref_apply_weights(ct, rs, mask, 1)))
    ref.same("visible", vis, lambda L: L["visible"])
    ref.same("cnt", c1, lambda L: L["cnt"])
    ref.same("weights", w1, lambda L: L["weights"])  # mask values are 0/1 -> sums are exact integers in fp32


@pytest.mark.parametrize("CH,binary", [(1, False), (2, True), (2, False), (3, True), (3, False)])
def test_apply_weights_channels_and_float_masks(CH, binary, reference):
    """apply_weights for CH = 1..3 (cuda_rasterizer/apply_weights.cu:365-380) and non-binary masks: `cnt` advances by
    CH per (pixel, splat) hit (:331-334) and must be EXACT; `weights` are float sums in a different order than the
    reference's per-hit atomics: exact for 0/1 masks (integer sums), <= 1e-5 relative for float masks."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    dev = "cuda"
    cloud, _ = synth.make_config("c3", P=25_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 333, 201, 61.0)[CH]      # partial last tile row and column
    H, W = cam.image_height, cam.image_width
    ct = cloud_tensors(cloud, dev)
    rs = settings_from(cam, (0, 0, 0), 0, dev)
    P = ct["means3D"].shape[0]
    rng = np.random.default_rng(17 + CH)
    m = rng.uniform(size=(CH, H, W)).astype(np.float32)
    if binary:
        m = (m > 0.4).astype(np.float32)
    mask = torch.from_numpy(m).to(dev)
    w1 = torch.zeros(P, CH, device=dev); c1 = torch.zeros(P, 1, dtype=torch.int32, device=dev)
    GaussianRasterizer(rs).apply_weights(ct["means3D"], None, ct["opacities"], None, w1, ct["scales"], ct["rotations"],
                                         None, c1, mask)
    torch.cuda.synchronize()
    ref = reference(f"apply_weights_ch{CH}_{'binary' if binary else 'float'}", lambda: _ref_apply_weights(ct, rs, mask, CH))
    ref.same("cnt", c1, lambda L: L["cnt"])
    assert int(c1.sum()) > 0 and int(c1.sum()) % CH == 0
    if binary:
        ref.same("weights", w1, lambda L: L["weights"])
    else:
        w, w2 = ref.rows("weights", w1, lambda L: L["weights"])
        assert rel_l2(w, w2) <= 1e-5
        w2_max = float(ref.value("weights_absmax", lambda L: float(L["weights"].abs().max())))
        assert float(np.abs(w - w2).max()) <= 1e-4 * w2_max
    # a second call ACCUMULATES (the reference never zeroes weights / cnt: rasterize_points.cu:223-231)
    c_first = c1.clone()
    GaussianRasterizer(rs).apply_weights(ct["means3D"], None, ct["opacities"], None, w1, ct["scales"], ct["rotations"],
                                         None, c1, mask)
    assert torch.equal(c1, 2 * c_first)


def test_alpha_output_matches_reference_accum_alpha_and_is_differentiable(reference):
    """Opt-in alpha image (north star: RGB / depth / alpha): alpha = 1 - final_T must equal 1 - the reference's
    ImageState::accum_alpha bit for bit; its gradient is checked through the identity
        color_0 with bg = (-1, 0, 0)  ==  C_0 - T_final  ==  C_0 + alpha - 1,
    i.e. d/dtheta [ sum G*(color_0 | bg=0) + sum G*alpha ] == d/dtheta sum G*(color_0 | bg=(-1,0,0))."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    dev = "cuda"
    cloud, _ = synth.make_config("c3", P=40_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 333, 201, 61.0)[2]
    H, W = cam.image_height, cam.image_width
    G = torch.from_numpy(np.random.default_rng(23).uniform(size=(H, W)).astype(np.float32)).to(dev)

    def run(bg, with_alpha):
        ct = cloud_tensors(cloud, dev, requires_grad=True)
        m2 = torch.zeros_like(ct["means3D"], requires_grad=True)
        rs = settings_from(cam, bg, cloud.sh_degree, dev)
        out = GaussianRasterizer(rs, return_alpha=with_alpha)(means3D=ct["means3D"], means2D=m2, opacities=ct["opacities"],
                                                              shs=ct["shs"], scales=ct["scales"], rotations=ct["rotations"])
        loss = (out[0][0] * G).sum()
        if with_alpha:
            assert len(out) == 4 and out[3].shape == (1, H, W)
            loss = loss + (out[3][0] * G).sum()
        loss.backward()
        grads = {k: v.grad.detach().cpu().numpy() for k, v in ct.items()}
        grads["means2D"] = m2.grad.detach().cpu().numpy()
        return out, grads

    out_a, g_a = run((0.0, 0.0, 0.0), True)
    ref = reference("alpha_c3", lambda: _ref_run(cloud, cam, (0.0, 0.0, 0.0)))
    ref.same("alpha", out_a[3][0], lambda L: 1.0 - L["state"]["final_T"])
    ref.same("color", out_a[0], lambda L: L["color"])
    out_b, g_b = run((-1.0, 0.0, 0.0), False)
    assert len(out_b) == 3
    for k in g_a:
        assert rel_l2(g_a[k], g_b[k]) <= 2e-5, (k, rel_l2(g_a[k], g_b[k]))


def test_camera_gradients_match_the_fp64_oracle_chain_and_finite_differences():
    """North star: backward over {..., viewmatrix}. The reference has no camera gradient, so the check is first
    principles, in three layers:
      1. tests/test_camera_grad_math.py (CPU): the formulas equal autograd of the smooth per-Gaussian forward map (1e-9);
      2. here: the CUDA kernel equals those formulas evaluated in float64 on the fp64 CPU oracle's upstream gradients
         (dL/dmean2D, dL/dconic, dL/dcolour of the same scene and loss), rel. L2 <= 1e-3 for all three camera arrays;
      3. here: viewmatrix and campos also agree with CENTRAL FINITE DIFFERENCES of the oracle's forward within 6 %.
         The pipeline is discontinuous where a pixel crosses a splat's alpha = 1/255 contour, the T < 1e-4 cut or the
         3-sigma tile rectangle, and the analytic gradient (the reference's, for every parameter) ignores the motion of
         those edges while a finite difference integrates it: the fp64 differences themselves move by 2-7 % between
         step sizes for the view matrix, and by far more for the projection matrix (210 / 188 / 24 / 68 for entry
         [0,0] at h = 2^-7 / 2^-11 / 2^-13 / 2^-15 against 243.7 analytic), which is why projmatrix has no layer 3."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    from test_camera_grad_math import camera_grads_formulas
    dev = "cuda"
    cloud, _ = synth.make_config("c3", P=4000)
    cloud.shs = np.ascontiguousarray(cloud.shs[:, :4, :])      # degree 1: what camera_grads_formulas restates
    cloud.sh_degree = 1
    cam = synth.ring_cameras(8, 4.5, 15.0, 96, 64, 61.0)[3]
    H, W = cam.image_height, cam.image_width
    bg = (0.2, 0.1, 0.3)
    G = np.random.default_rng(31).uniform(0.5, 1.5, size=(3, H, W)).astype(np.float32)
    ct = cloud_tensors(cloud, dev)
    rs = settings_from(cam, bg, cloud.sh_degree, dev)
    view = rs.viewmatrix.clone().requires_grad_(True)
    proj = rs.projmatrix.clone().requires_grad_(True)
    cpos = rs.campos.clone().requires_grad_(True)
    rs = rs._replace(viewmatrix=view, projmatrix=proj, campos=cpos)
    out = GaussianRasterizer(rs, camera_grad=True)(means3D=ct["means3D"], means2D=torch.zeros_like(ct["means3D"]),
                                                   opacities=ct["opacities"], shs=ct["shs"], scales=ct["scales"],
                                                   rotations=ct["rotations"])
    (out[0] * torch.from_numpy(G).to(dev)).sum().backward()
    got = dict(viewmatrix=view.grad.cpu().numpy().astype(np.float64), projmatrix=proj.grad.cpu().numpy().astype(np.float64),
               campos=cpos.grad.cpu().numpy().astype(np.float64))
    assert np.all(got["viewmatrix"][:, 3] == 0) and np.all(got["projmatrix"][:, 2] == 0)   # entries the forward never reads

    # layer 2: the chain rule in float64 on the oracle's upstream gradients
    f = cpu_oracle.forward_from(cloud, cam, bg, f32=False)
    g = f.backward(G)
    vis = f.radii > 0
    hx, hy = W / (2 * cam.tanfovx), H / (2 * cam.tanfovy)
    t = (cloud.means3D[vis].astype(np.float64) @ cam.viewmatrix.astype(np.float64)[:3, :3]) + cam.viewmatrix.astype(np.float64)[3, :3]
    assert np.all(np.abs(t[:, 0] / t[:, 2]) < 1.3 * cam.tanfovx) and np.all(np.abs(t[:, 1] / t[:, 2]) < 1.3 * cam.tanfovy)  # nobody clamped
    g_conic = np.stack([g["dconic"][vis, 0, 0], g["dconic"][vis, 0, 1], g["dconic"][vis, 1, 1]], 1)
    g_col = g["dcolor"][vis] * (1.0 - f.clamped[vis].astype(np.float64))
    dv, dp, dc = camera_grads_formulas(cam.viewmatrix.astype(np.float64), cam.projmatrix.astype(np.float64),
                                       cam.campos.astype(np.float64), cloud.means3D[vis].astype(np.float64),
                                       f.cov3D[vis].astype(np.float64), cloud.shs[vis].astype(np.float64),
                                       g["dmean2D"][vis, :2], g_conic, g_col, hx, hy)
    f.close()
    for name, want in (("viewmatrix", dv), ("projmatrix", dp), ("campos", dc)):
        assert rel_l2(got[name], want) <= 1e-3, (name, rel_l2(got[name], want), got[name], want)

    # layer 3: finite differences of the fp64 forward (float32-representable steps) for the two stable arrays
    def loss(**over):
        ff = cpu_oracle.forward_from(cloud, cam, bg, f32=False, **over)
        v = float((ff.color * G).sum())
        ff.close()
        return v
    h = np.float32(2.0 ** -11)
    for name, arr in (("viewmatrix", cam.viewmatrix.astype(np.float32)), ("campos", cam.campos.astype(np.float32))):
        fd = np.zeros(arr.shape, np.float64)
        for idx in np.ndindex(arr.shape):
            if name == "viewmatrix" and idx[1] == 3:
                continue
            ap, am = arr.copy(), arr.copy()
            ap[idx] += h; am[idx] -= h
            fd[idx] = (loss(**{name: ap}) - loss(**{name: am})) / float(ap[idx] - am[idx])
        assert np.linalg.norm(fd) > 0 and rel_l2(got[name], fd) <= 6e-2, (name, rel_l2(got[name], fd), got[name], fd)


def test_full_size_properties_config3():
    """BASELINE config 3 (1M Gaussians, 1600x1200): size-independent properties at full size."""
    cloud, cams = synth.make_config("c3")
    cam = cams[0]
    dL = np.random.default_rng(1).uniform(size=(3, cam.image_height, cam.image_width)).astype(np.float32)
    out = run_ours(cloud, cam, (0, 0, 0), dL=dL)
    v = out["views"]
    R = out["R"]
    assert R == int(v["tiles_touched"].sum())
    ranges = v["ranges"].cpu().numpy().astype(np.int64)
    nz = ranges[ranges[:, 1] > ranges[:, 0]]
    assert nz[:, 1].max() == R and int((nz[:, 1] - nz[:, 0]).sum()) == R   # ranges tile the list exactly
    keys = v["tile_keys"].cpu().numpy()
    if keys.dtype == np.int16:
        keys = keys.view(np.uint16)
    assert np.all(np.diff(keys.astype(np.int64)) >= 0)                       # sorted by tile
    pl = v["point_list"].cpu().numpy()
    depth = v["records"][:, 6].cpu().numpy()
    d = depth[pl]
    same_tile = keys[1:] == keys[:-1]
    assert np.all(d[1:][same_tile] >= d[:-1][same_tile])                     # depth-sorted inside every tile
    tie = same_tile & (d[1:] == d[:-1])
    assert np.all(pl[1:][tie] > pl[:-1][tie])                                # stable: ties by Gaussian index
    assert np.array_equal(np.bincount(pl, minlength=cloud.means3D.shape[0]), v["tiles_touched"].cpu().numpy())
    col = out["color"]
    assert torch.isfinite(col).all() and float(col.min()) >= 0.0
    T = v["final_T"]
    assert float(T.min()) >= float(np.float32(1e-4)) and float(T.max()) <= 1.0
    vis = (out["radii"] > 0)
    for k, g in out["grads"].items():
        if g is None:
            continue
        assert torch.isfinite(g).all(), k
        assert float(g[~vis].abs().sum()) == 0.0, k                          # culled Gaussians get exact zeros
    # linearity of the backward in dL/dpixel
    out2 = run_ours(cloud, cam, (0, 0, 0), dL=2.0 * dL)
    a, b = out["grads"]["dmean3D"], out2["grads"]["dmean3D"]
    assert rel_l2((2 * a).cpu().numpy(), b.cpu().numpy()) <= 1e-4


def test_host_buffer_api():
    """C-ABI host-buffer entry points (gsr_host_*): same images as the tensor path, checksums of all gradients."""
    import ctypes as C
    lib = _lib.load()
    cloud, _ = synth.make_config("c3", P=50_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 320, 240, 61.0)[4]
    dL = np.random.default_rng(2).uniform(size=(3, 240, 320)).astype(np.float32)
    ref = run_ours(cloud, cam, (0.2, 0.3, 0.4), dL=dL)
    ctx = C.c_void_p(lib.gsr_host_create())
    assert ctx.value
    P, M = cloud.means3D.shape[0], cloud.shs.shape[1]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    arrs = [np.ascontiguousarray(x, np.float32) for x in (cloud.means3D, cloud.opacities, cloud.shs, cloud.scales, cloud.rotations)]
    _lib.check(lib.gsr_host_upload_cloud(ctx, P, M, *[p(a) for a in arrs]), "upload")
    bg = np.array([0.2, 0.3, 0.4], np.float32)
    s = _lib.Settings(240, 320, cam.tanfovx, cam.tanfovy, 1.0, 3, M, 0, 0, p(bg).value, p(cam.viewmatrix).value,
                      p(cam.projmatrix).value, p(cam.campos).value)
    color = np.zeros((3, 240, 320), np.float32); radii = np.zeros(P, np.int32); sums = np.zeros(8, np.float64)
    R = lib.gsr_host_step(ctx, C.byref(s), p(dL), p(color), p(radii), p(sums))
    lib.gsr_host_destroy(ctx)
    assert R == ref["R"]
    assert np.array_equal(color, ref["color"].cpu().numpy())
    assert np.array_equal(radii, ref["radii"].cpu().numpy())
    g = ref["grads"]
    want = [g["dmean3D"], g["dmean2D"], None, g["dopacity"], None, g["dsh"], g["dscale"], g["drot"]]
    for i, w in enumerate(want):
        if w is not None:
            ws = float(w.double().sum())
            scale = float(w.double().abs().sum()) + 1e-12
            assert abs(sums[i] - ws) <= 1e-5 * scale, (i, sums[i], ws)


def test_speculative_second_half_equals_exact_path():
    """The sync-free forward (capacity guessed from the previous frame) must give the same bits as the exact path,
    including when the guess is too small and the second half is redone."""
    import gaussianeditor_b200.rasterizer as RZ
    cloud, _ = synth.make_config("c3", P=40_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 320, 240, 61.0)[6]
    dL = np.random.default_rng(9).uniform(size=(3, 240, 320)).astype(np.float32)
    key = (0, cloud.means3D.shape[0], 320, 240)
    try:
        RZ.SPECULATIVE = False
        exact = run_ours(cloud, cam, (0.5, 0.5, 0.5), dL=dL)
        RZ.SPECULATIVE = True
        RZ._r_hint[key] = exact["R"]            # good guess -> speculative path
        spec = run_ours(cloud, cam, (0.5, 0.5, 0.5), dL=dL)
        assert spec["state"].cap > spec["R"] == exact["R"]
        RZ._r_hint[key] = 10                    # hopeless guess -> overflow -> redo with the exact size
        redo = run_ours(cloud, cam, (0.5, 0.5, 0.5), dL=dL)
        assert redo["state"].cap == redo["R"] == exact["R"]
        for other in (spec, redo):
            assert torch.equal(other["color"], exact["color"]) and torch.equal(other["depth"], exact["depth"])
            assert torch.equal(other["views"]["point_list"], exact["views"]["point_list"])
            assert torch.equal(other["views"]["ranges"], exact["views"]["ranges"])
            assert torch.equal(other["views"]["n_contrib"], exact["views"]["n_contrib"])
            for k in ("dmean3D", "dsh", "dopacity"):
                assert rel_l2(other["grads"][k].cpu().numpy(), exact["grads"][k].cpu().numpy()) <= 1e-5
    finally:
        RZ.SPECULATIVE = True


@pytest.mark.parametrize("variant,depth_variant", [(0, 0), (1, 1), (1, 0), (0, 1)])
def test_binning_variants_match_reference_lists(variant, depth_variant, reference):
    """Both binning implementations -- 0: emit kernel + CUB radix sort + tile_ranges (binning.cu), 1: difference-array
    ranges + two own radix passes with the emission fused in (tile_binning.cu, default) -- and both depth orders -- 0: CUB
    radix sort + CUB scan, 1: depth_sort.cu (default) -- must give the reference's point_list / ranges / R bit for bit,
    incl. a partial last tile row/column and a frame with > 256 tile columns."""
    with kernel_options(binning_variant=variant, depth_sort_variant=depth_variant):
        cloud, _ = synth.make_config("c3", P=80_000)
        for (W, H, k) in [(333, 201, 5), (4160, 48, 1), (1600, 1200, 2)]:
            cam = synth.ring_cameras(8, 4.5, 15.0, W, H, 61.0)[k]
            ours = run_ours(cloud, cam, (0.1, 0.2, 0.3))
            ref = reference(f"binning_{W}x{H}", lambda: _ref_run(cloud, cam, (0.1, 0.2, 0.3)))
            v = ours["views"]
            ref.same("R", ours["R"], lambda L: L["R"])
            ref.same("ranges", v["ranges"], lambda L: L["state"]["ranges"])
            ref.same("point_list", v["point_list"], lambda L: L["state"]["point_list"])
            ref.same("color", ours["color"], lambda L: L["color"])


def test_depth_order_and_offsets_equal_cub_at_full_size():
    """depth_sort.cu against the CUB sort + scan it replaces, at BASELINE config 3 size (1M keys, 39 % of them the
    culled key 0xFFFFFFFF, ties between equal depths): depth_order and the instance total must be identical."""
    from gaussianeditor_b200.rasterizer import forward_state_views
    cloud, cams = synth.make_config("c3")
    res = {}
    for v in (0, 1):
        with kernel_options(depth_sort_variant=v):
            out = run_ours(cloud, cams[2], (0, 0, 0))
        res[v] = (out["views"]["depth_order"].clone(), out["R"], out["views"]["point_list"].clone())
    vis = int((out["radii"] > 0).sum())
    assert torch.equal(res[0][0][:vis], res[1][0][:vis])       # among the culled (equal keys) both are index-ordered too:
    assert torch.equal(res[0][0], res[1][0])
    assert res[0][1] == res[1][1] and torch.equal(res[0][2], res[1][2])


def test_edit_loop_harness_runs_and_densifies():
    """Config-5 loop shape (2 forwards + 1 backward per step, densification changing P) on a small cloud."""
    from gaussianeditor_b200 import edit_loop
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    out = edit_loop.run_edit_loop(GaussianRasterizer, steps=8, P=20_000, densification_interval=3)
    assert out["P_last"] != out["P_first"] and 0.0 < out["render_fraction"] < 1.0
    assert np.isfinite(out["final_loss"])


def test_edit_loop_matches_the_reference_rasterizer_step_by_step(reference):
    """SURVEY 8(f-2): the SAME config-5-shaped loop (two renders + one backward per step, Adam, densify / prune
    changing P) driven once by this repository's rasterizer and once by the reference's own CUDA kernels
    (oracle/ref_torch.RefGaussianRasterizer) from identical seeds: the Gaussian count after every densification must be
    identical, the loss trajectories must agree to 1e-3, and the max_radii2D bookkeeping (what the reference's prune
    test reads) must be identical at the first densification and agree on >= 99.9 % of the Gaussians at the end."""
    from gaussianeditor_b200 import edit_loop
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    kw = dict(steps=20, P=20_000, densification_interval=5, seed=3)
    ours = edit_loop.run_edit_loop(GaussianRasterizer, **kw)

    def run_ref():
        from oracle.ref_torch import RefGaussianRasterizer
        return edit_loop.run_edit_loop(RefGaussianRasterizer, **kw)
    ref = reference("edit_loop", run_ref)
    ref_counts = ref.value("counts", lambda L: L["counts"]).tolist()
    assert ours["counts"] == ref_counts and len(set(ours["counts"])) >= 3       # P changed, identically
    lo, lr = np.array(ours["losses"]), ref.value("losses", lambda L: L["losses"])
    assert np.all(np.isfinite(lo)) and np.abs(lo - lr).max() <= 1e-3 * np.abs(lr).max(), np.abs(lo - lr).max()
    ref.same("max_radii2D_at_densify0", ours["max_radii2D_at_densify"][0], lambda L: L["max_radii2D_at_densify"][0])
    ref_radii = ref.value("max_radii2D", lambda L: L["max_radii2D"])
    assert ours["max_radii2D"].shape == ref_radii.shape
    same = float((ours["max_radii2D"].numpy() == ref_radii).mean())
    assert same >= 0.999, same
    # the fused-activation entry point must drive the same loop to the same counts
    fused = edit_loop.run_edit_loop(GaussianRasterizer, fused_activations=True, **kw)
    assert fused["counts"] == ref_counts
    assert np.abs(np.array(fused["losses"]) - lr).max() <= 1e-3 * np.abs(lr).max()


def _grad_close(ours, ref, pairs, name, tol=1e-4):
    for a, b in pairs:
        g = ours["grads"][a]
        if g is None:
            continue
        err = rel_l2(*ref.rows(b, g, lambda L: L["grads"][b]))
        assert err <= tol, (name, a, err)


@pytest.mark.parametrize("deg,M", [(0, 16), (1, 16), (2, 16), (3, 16), (1, 4), (2, 9), (0, 1)])
def test_sh_degrees_and_coefficient_counts(deg, M, reference):
    """Active degree below the allocated one (GaussianEditor ramps sh_degree up), M = 4 / 16 take the TMA row path,
    M = 1 / 9 the plain-load path; coefficients above the active degree must get exactly zero gradient."""
    cloud, _ = synth.make_config("c3", P=30_000)
    cloud.shs = np.ascontiguousarray(cloud.shs[:, :M, :])
    cloud.sh_degree = deg
    cam = synth.ring_cameras(8, 4.5, 15.0, 208, 160, 61.0)[3]
    dL = np.random.default_rng(deg * 7 + M).uniform(size=(3, 160, 208)).astype(np.float32)
    ours = run_ours(cloud, cam, (0.1, 0.1, 0.1), dL=dL)
    ref = reference(f"sh_deg{deg}_M{M}", lambda: _ref_run(cloud, cam, (0.1, 0.1, 0.1), dL=dL))
    ref.same("radii", ours["radii"], lambda L: L["radii"])
    ref.same("color", ours["color"], lambda L: L["color"])
    vis = ours["radii"] > 0
    ref.same("rgb", ours["views"]["records"][vis][:, 8:11], lambda L: L["state"]["rgb"][vis])

    def ref_clamped(L):
        rc = L["state"]["clamped"][vis]
        return (rc[:, 0] + 2 * rc[:, 1] + 4 * rc[:, 2]).to(torch.uint8)
    ref.same("clamped", ours["views"]["clamped"][vis], ref_clamped)
    _grad_close(ours, ref, [("dsh", "dL_dsh"), ("dmean3D", "dL_dmeans3D"), ("dopacity", "dL_dopacity")], (deg, M))
    nb = (deg + 1) ** 2
    assert float(ours["grads"]["dsh"][:, nb:, :].abs().sum()) == 0.0


def test_precomputed_covariance_path(reference):
    """cov3D_precomp instead of scale/rotation (unused by GaussianEditor but part of the API): forward bit-exact,
    dL/dcov3D to tolerance, scale/rotation gradients absent."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    dev = "cuda"
    cloud, _ = synth.make_config("c3", P=20_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 192, 144, 61.0)[5]
    f = cpu_oracle.forward_from(cloud, cam, render=False)          # cov3D from the oracle as the precomputed input
    cov = torch.from_numpy(f.cov3D.astype(np.float32)).to(dev).requires_grad_(True)
    f.close()
    ct = cloud_tensors(cloud, dev, requires_grad=True)
    rs = settings_from(cam, (0, 0, 0), 3, dev)
    m2 = torch.zeros_like(ct["means3D"], requires_grad=True)
    color, radii, depth = GaussianRasterizer(rs)(means3D=ct["means3D"], means2D=m2, opacities=ct["opacities"],
                                                 shs=ct["shs"], cov3D_precomp=cov)
    dL = torch.from_numpy(np.random.default_rng(13).uniform(size=(3, 144, 192)).astype(np.float32)).to(dev)
    (color * dL).sum().backward()

    def run_ref():
        R = ref_cuda.ReferenceRasterizer()
        common = dict(means3D=ct["means3D"].detach(), shs=ct["shs"].detach(), colors_precomp=None, scales=None,
                      rotations=None, cov3D_precomp=cov.detach(), bg=rs.bg, viewmatrix=rs.viewmatrix,
                      projmatrix=rs.projmatrix, campos=rs.campos, tanfovx=rs.tanfovx, tanfovy=rs.tanfovy, sh_degree=3)
        rc, rr, rd, n = R.forward(opacities=ct["opacities"].detach(), image_height=144, image_width=192, **common)
        return dict(color=rc, radii=rr, grads=R.backward(dL_dcolor=dL, radii=rr, R=n, **common))
    ref = reference("cov3D_precomp", run_ref)
    ref.same("radii", radii, lambda L: L["radii"])
    ref.same("color", color, lambda L: L["color"])
    assert rel_l2(*ref.rows("dL_dcov3D", cov.grad, lambda L: L["grads"]["dL_dcov3D"])) <= 1e-4
    assert rel_l2(*ref.rows("dL_dmeans3D", ct["means3D"].grad, lambda L: L["grads"]["dL_dmeans3D"])) <= 1e-4


def test_hd_frame_partial_tile_row_and_debug_flag(reference):
    """1920x1080: 1080 is not a multiple of 16 (68 tile rows, last partial); debug=True synchronises after each launch."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer, _RasterizeGaussians, forward_state_views
    dev = "cuda"
    cloud, _ = synth.make_config("c3", P=150_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 1920, 1080, 61.0)[1]
    ct = cloud_tensors(cloud, dev)
    rs = settings_from(cam, (0.3, 0.6, 0.9), 3, dev, debug=True)
    color, radii, depth = GaussianRasterizer(rs)(means3D=ct["means3D"], means2D=torch.zeros_like(ct["means3D"]),
                                                 opacities=ct["opacities"], shs=ct["shs"], scales=ct["scales"],
                                                 rotations=ct["rotations"])
    v = forward_state_views(_RasterizeGaussians.last_state)
    ref = reference("hd_1920x1080", lambda: _ref_run(cloud, cam, (0.3, 0.6, 0.9)))
    assert v["ranges"].shape[0] == 120 * 68
    ref.same("radii", radii, lambda L: L["radii"])
    ref.same("ranges", v["ranges"], lambda L: L["state"]["ranges"])
    ref.same("color", color, lambda L: L["color"])
    ref.same("depth", depth, lambda L: L["depth"])
    ref.same("n_contrib", v["n_contrib"], lambda L: L["state"]["n_contrib"])


def _check_forward_bit_exact(ours, ref):
    v = ours["views"]
    ref.same("R", ours["R"], lambda L: L[0]["R"])
    for k in ("radii", "color", "depth"):
        ref.same(k, ours[k], lambda L: L[0][k])
    for k in ("n_contrib", "final_T"):
        ref.same(k, v[k].flatten(), lambda L: L[0]["state"][k].flatten())
    ref.same("point_list", v["point_list"], lambda L: L[0]["state"]["point_list"])


@pytest.mark.parametrize("cfg", ["c2", "c3"])
def test_full_size_configs_match_reference_cuda(cfg, reference):
    """BASELINE configs 2 (100k, SH 0, 800x800) and 3 (1M, SH 3, 1600x1200) at FULL size against the reference's
    own CUDA build: forward bit-exact (images, radii, n_contrib, final_T, the complete sorted list).

    Gradients are judged against the fp64 CPU oracle (ground truth), because at full size the REFERENCE is the
    inaccurate one: its ~10^6 per-pixel fp32 atomics on the largest splats swamp small addends and under-count
    (config 3: reference 2.5e-4 .. 6.3e-4 relative L2 from fp64; this repo 1e-6 .. 1.3e-5, like the fp32 CPU oracle).
    So: ours vs fp64 <= 5e-5, and ours vs reference no further apart than the reference is from the truth."""
    cloud, cams = synth.make_config(cfg)
    cam = cams[-1]
    bg = (0.1, 0.2, 0.3)
    dL = np.random.default_rng(11).uniform(size=(3, cam.image_height, cam.image_width)).astype(np.float32)
    ours = run_ours(cloud, cam, bg, dL=dL)
    ref = reference("full_" + cfg, lambda: [_ref_run(cloud, cam, bg, dL=dL) for _ in range(2)])
    _check_forward_bit_exact(ours, ref)
    f64 = cpu_oracle.forward_from(cloud, cam, bg, f32=False)
    truth = f64.backward(dL)
    f64.close()
    for a, b in [("dmean3D", "dL_dmeans3D"), ("dmean2D", "dL_dmeans2D"), ("dopacity", "dL_dopacity"),
                 ("dscale", "dL_dscales"), ("drot", "dL_drotations"), ("dsh", "dL_dsh")]:
        g, t = ours["grads"][a].cpu().numpy(), truth[a]
        noise = float(ref.value(b + "_noise", lambda L: rel_l2(_f64(L[1]["grads"][b]), _f64(L[0]["grads"][b]))))
        ref_err = float(ref.value(b + "_err_vs_fp64", lambda L: rel_l2(_f64(L[0]["grads"][b]), t)))
        ours_err = rel_l2(g, t)
        assert ours_err <= 5e-5, (cfg, a, ours_err)
        # the reference's own distance from the truth must stay inside the band observed on B200 (<= 6.3e-4 at
        # config 3, profiles/README.md), so that a regression of OURS cannot hide behind a growing ref_err term
        assert ref_err <= 1.5e-3, (cfg, a, ref_err)
        g_rows, r_rows = ref.rows(b, g, lambda L: L[0]["grads"][b])
        err = rel_l2(g_rows, r_rows)
        assert err <= 1e-4 + 10 * noise + 1.5 * ref_err, (cfg, a, err, noise, ref_err)


def test_full_size_properties_config4():
    """BASELINE config 4 (5M Gaussians, 1920x1080) on one GPU: list invariants, determinism of the forward
    (bit-identical across two runs), finite gradients that vanish exactly for culled Gaussians."""
    cloud, cams = synth.make_config("c4")
    cam = cams[3]
    dL = np.random.default_rng(2).uniform(size=(3, cam.image_height, cam.image_width)).astype(np.float32)
    out = run_ours(cloud, cam, (0, 0, 0), dL=dL)
    v, R = out["views"], out["R"]
    assert R == int(v["tiles_touched"].to(torch.int64).sum())
    ranges = v["ranges"].to(torch.int64)
    lens = ranges[:, 1] - ranges[:, 0]
    assert int(lens.sum()) == R and int(lens.min()) >= 0 and int(ranges[:, 1].max()) == R
    keys = v["tile_keys"]
    keys = (keys.to(torch.int32) & 0xFFFF) if keys.dtype == torch.int16 else keys
    assert bool((keys[1:] >= keys[:-1]).all())
    pl = v["point_list"].to(torch.int64)
    d = v["records"][:, 6][pl]
    same = keys[1:] == keys[:-1]
    assert bool((d[1:][same] >= d[:-1][same]).all())
    tie = same & (d[1:] == d[:-1])
    assert bool((pl[1:][tie] > pl[:-1][tie]).all())
    assert float(v["final_T"].min()) >= float(np.float32(1e-4)) and float(v["final_T"].max()) <= 1.0
    vis = out["radii"] > 0
    for k, g in out["grads"].items():
        if g is not None:
            assert torch.isfinite(g).all(), k
            assert float(g[~vis].abs().sum()) == 0.0, k
    again = run_ours(cloud, cam, (0, 0, 0))
    assert torch.equal(again["color"], out["color"]) and torch.equal(again["radii"], out["radii"])
    assert torch.equal(again["views"]["point_list"], v["point_list"]) and again["R"] == R


def _raw_params(cloud, dev, seed=0):
    """Inverse activations of a synth.Cloud -> leaf tensors shaped like the scene model's raw parameters
    (scene/gaussian_model.py:_xyz, _features_dc, _features_rest, _opacity, _scaling, _rotation)."""
    g = torch.Generator().manual_seed(seed)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    op = t(cloud.opacities).clamp(1e-6, 1 - 1e-6)
    rot = t(cloud.rotations) * (0.25 + 3.0 * torch.rand(cloud.rotations.shape[0], 1, generator=g)).to(dev)  # unnormalised
    raw = dict(xyz=t(cloud.means3D), opacity=torch.log(op / (1 - op)), features_dc=t(cloud.shs[:, :1, :]),
               features_rest=t(cloud.shs[:, 1:, :]), scaling=torch.log(t(cloud.scales)), rotation=rot)
    return {k: v.contiguous().requires_grad_(True) for k, v in raw.items()}


@pytest.mark.parametrize("deg,M,P", [(3, 16, 60013), (3, 16, 4096), (1, 4, 20000), (0, 1, 5000)])
def test_fused_activations_match_pytorch_prologue(deg, M, P):
    """SURVEY 8(f-3): GaussianRasterizer.forward_raw (sigmoid / exp / normalize / SH concatenation inside the
    preprocess kernels) against the scene model's PyTorch prologue followed by the default rasterizer, forward and
    all raw-parameter gradients. P = 60013 ends in a partial block (plain-load fallback), 4096 is all bulk copies."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    dev = torch.device("cuda")
    cloud, cams = synth.make_config("c3", P=P)
    cloud.shs = np.ascontiguousarray(cloud.shs[:, :M, :])
    cloud.sh_degree = deg
    cam = synth.ring_cameras(8, 4.5, 15.0, 640, 400, 61.0)[1]
    rs = settings_from(cam, (0.3, 0.1, 0.2), deg, dev)
    dL = torch.from_numpy(np.random.default_rng(5).uniform(size=(3, cam.image_height, cam.image_width)).astype(np.float32)).to(dev)
    rast = GaussianRasterizer(rs)

    a = _raw_params(cloud, dev)
    m2a = torch.zeros_like(a["xyz"], requires_grad=True)
    col_a, rad_a, dep_a = rast(means3D=a["xyz"], means2D=m2a, opacities=torch.sigmoid(a["opacity"]),
                               shs=torch.cat((a["features_dc"], a["features_rest"]), dim=1),
                               scales=torch.exp(a["scaling"]), rotations=torch.nn.functional.normalize(a["rotation"]))
    (col_a * dL).sum().backward()

    b = _raw_params(cloud, dev)
    m2b = torch.zeros_like(b["xyz"], requires_grad=True)
    col_b, rad_b, dep_b = rast.forward_raw(means3D=b["xyz"], means2D=m2b, opacity_logits=b["opacity"],
                                           features_dc=b["features_dc"], features_rest=b["features_rest"],
                                           log_scales=b["scaling"], raw_rotations=b["rotation"])
    (col_b * dL).sum().backward()

    assert float((rad_a != rad_b).float().mean()) <= 1e-4           # activations round differently in rare cases
    ca, cb = col_a.detach().cpu().numpy(), col_b.detach().cpu().numpy()
    assert np.mean(np.abs(ca - cb) > 1e-5 + 1e-4 * np.abs(ca)) <= 1e-4
    assert rel_l2(dep_b.detach().cpu().numpy(), dep_a.detach().cpu().numpy()) <= 1e-5
    same = (rad_a == rad_b)
    for k in a:
        ga, gb = a[k].grad, b[k].grad
        assert gb is not None and gb.shape == ga.shape, k
        assert torch.isfinite(gb).all(), k
        assert rel_l2(gb[same].cpu().numpy(), ga[same].cpu().numpy()) <= 1e-4, (k, rel_l2(gb[same].cpu().numpy(), ga[same].cpu().numpy()))
    assert rel_l2(m2b.grad[same].cpu().numpy(), m2a.grad[same].cpu().numpy()) <= 1e-4
    assert float(b["features_rest"].grad[rad_b == 0].abs().sum()) == 0.0   # culled rows are written as exact zeros


def test_blending_weights_conserve_energy_at_full_size():
    """Size-independent property at BASELINE config 3 size: with precomputed colours and dL/dpixel = 1 on one channel,
    dL/dcolor_i is the total blending weight of splat i, and the weights of all splats plus the remaining
    transmittance of every pixel add up to the number of pixels (sum_i alpha_i T_i + T_final = 1 per pixel)."""
    cloud, cams = synth.make_config("c3")
    cam = cams[5]
    H, W = cam.image_height, cam.image_width
    dL = np.zeros((3, H, W), np.float32)
    dL[1] = 1.0
    cols = np.random.default_rng(4).random((cloud.means3D.shape[0], 3), dtype=np.float32)
    out = run_ours(cloud, cam, (0.0, 0.0, 0.0), dL=dL, colors_precomp=cols)
    w = out["grads"]["dcolor"].double()
    assert float(w.min()) >= 0.0 and float(w[:, 0].abs().sum()) == 0.0 and float(w[:, 2].abs().sum()) == 0.0
    total = float(w[:, 1].sum()) + float(out["views"]["final_T"].double().sum())
    assert abs(total - H * W) <= 2e-5 * H * W, (total, H * W)
