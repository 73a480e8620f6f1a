"""CPU-only checks of the drop-in boundary: the C-ABI library loads and exports every symbol the header declares,
argument validation mirrors the reference's messages, and the product path fails LOUDLY (never falls back to a
CPU implementation) when no CUDA device is available."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from gaussianeditor_b200 import _lib, synth
from gaussianeditor_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
from util import OPTION_DEFAULTS, get_option, kernel_options

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "gsr_b200.h")).read()
    return sorted(set(re.findall(r"GSR_API\s+[\w\s\*]+?\b(gsr_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/gsr_b200.h but not exported"
    assert sorted(_lib.SYMBOLS) == syms
    assert lib.gsr_abi_version() == 2


def test_library_contains_sm100a_code_and_tma():
    import shutil
    import subprocess
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass  # cp.async.bulk (TMA unit) in the preprocess kernels


def test_sizing_and_validation_without_gpu_semantics():
    lib = _lib.load()
    assert lib.gsr_image_bytes(1600, 1200) >= 1600 * 1200 * 8 + 7500 * 12
    assert lib.gsr_backward_scratch_bytes(1000) >= 1000 * 48
    s = _lib.Settings(16, 16, 1.0, 1.0, 1.0, 0, 1, 0, 0, None, None, None, None)
    dummy = C.c_void_p(256)
    host = (C.c_int32 * 1)()
    # both SHs and colours missing -> the reference's message (diff_gaussian_rasterization/__init__.py:271-276)
    c = _lib.Cloud(4, dummy, dummy, None, None, dummy, dummy, None)
    rc = lib.gsr_forward_preprocess(C.byref(s), C.byref(c), dummy, 1 << 20, dummy, host, None)
    assert rc == -1 and b"excatly one of either SHs or precomputed colors" in lib.gsr_last_error()
    # scale/rotation AND cov3D_precomp -> the reference's second message (:278-283)
    c = _lib.Cloud(4, dummy, dummy, dummy, None, dummy, dummy, dummy)
    rc = lib.gsr_forward_preprocess(C.byref(s), C.byref(c), dummy, 1 << 20, dummy, host, None)
    assert rc == -1 and b"scale/rotation pair or precomputed 3D covariance" in lib.gsr_last_error()
    # unknown option
    assert lib.gsr_set_option(b"no_such_option", 1) == -1
    with kernel_options(render_fwd_variant=2):
        assert lib.gsr_get_option(b"render_fwd_variant") == 2


def test_option_defaults_match_the_compiled_ones():
    """tests/util.OPTION_DEFAULTS (what kernel_options() and the shape/variant tests treat as "the default") is the
    Options struct of csrc/common.cuh, and kernel_options() restores what it changed."""
    text = open(os.path.join(ROOT, "gaussianeditor_b200", "csrc", "common.cuh")).read()
    body = re.search(r"struct Options \{(.*?)\};", text, re.S).group(1)
    compiled = {k: int(v) for k, v in re.findall(r"int (\w+) = (-?\d+);", body)}
    assert compiled == OPTION_DEFAULTS
    before = {k: get_option(k) for k in compiled}
    with kernel_options(render_bwd_variant=3, tile_key_bits=32):
        assert get_option("render_bwd_variant") == 3 and get_option("tile_key_bits") == 32
    assert {k: get_option(k) for k in compiled} == before


def _settings(device):
    cam = synth.look_at_camera((0, 0, -3.5), (0, 0, 0), (0, -1, 0), 32, 32, fovy_deg=50.0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
    return GaussianRasterizationSettings(32, 32, cam.tanfovx, cam.tanfovy, torch.zeros(3, device=device), 1.0,
                                         t(cam.viewmatrix), t(cam.projmatrix), 0, t(cam.campos), False, False)


def test_python_api_argument_errors_match_reference():
    rast = GaussianRasterizer(_settings("cpu"))
    P = 5
    m = torch.zeros(P, 3); o = torch.ones(P, 1); sh = torch.zeros(P, 1, 3); c = torch.zeros(P, 3)
    sc = torch.ones(P, 3); ro = torch.zeros(P, 4); cov = torch.zeros(P, 6)
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        rast(m, m, o, shs=None, colors_precomp=None, scales=sc, rotations=ro)
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        rast(m, m, o, shs=sh, colors_precomp=c, scales=sc, rotations=ro)
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        rast(m, m, o, shs=sh, scales=sc, rotations=ro, cov3D_precomp=cov)
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        rast(m, m, o, shs=sh, scales=sc)
    with pytest.raises(RuntimeError, match=r"dimensions \(num_points, 3\)"):
        rast(torch.zeros(P, 4), m, o, shs=sh, scales=sc, rotations=ro)


def test_no_cpu_fallback():
    """CPU tensors (or a box without a GPU) must raise -- the oracle is never on the product path."""
    rast = GaussianRasterizer(_settings("cpu"))
    P = 5
    m = torch.zeros(P, 3); o = torch.ones(P, 1); sh = torch.zeros(P, 1, 3)
    with pytest.raises(RuntimeError, match="no CPU path"):
        rast(m, m, o, shs=sh, scales=torch.ones(P, 3), rotations=torch.zeros(P, 4))
    import gaussianeditor_b200.rasterizer as R
    import gaussianeditor_b200._lib as L
    src = open(R.__file__).read() + open(L.__file__).read()
    assert "oracle" not in src.replace("CPU oracle under ``oracle/``", "").replace("The CPU oracle", "") or \
        "import oracle" not in src and "from oracle" not in src
    if not torch.cuda.is_available():
        assert _lib.load().gsr_geometry_bytes(1000) == 0          # CUB size query needs the driver: loud failure
        assert b"CUDA" in _lib.load().gsr_last_error()


def test_settings_namedtuple_matches_reference_field_order():
    assert GaussianRasterizationSettings._fields == (
        "image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix",
        "sh_degree", "campos", "prefiltered", "debug")   # diff_gaussian_rasterization/__init__.py:228-240
    import diff_gaussian_rasterization as D   # the import name GaussianEditor uses
    assert D.GaussianRasterizer is GaussianRasterizer


def test_synthetic_configs_are_deterministic():
    a, cams = synth.make_config("c3", P=5000)
    b, _ = synth.make_config("c3", P=5000)
    for f in ("means3D", "scales", "rotations", "opacities", "shs"):
        assert np.array_equal(getattr(a, f), getattr(b, f))
    assert a.shs.shape == (5000, 16, 3) and len(cams) == 8
    assert np.allclose(np.linalg.norm(a.rotations, axis=1), 1.0, atol=1e-6)
    # camera convention: transposed W2C, full projection = view @ P^T, camera centre consistent with the view matrix
    cam = cams[0]
    W2C = cam.viewmatrix.T
    centre = -W2C[:3, :3].T @ W2C[:3, 3]
    assert np.allclose(centre, cam.campos, atol=1e-5)
    assert abs(cam.tanfovx / cam.tanfovy - 1600 / 1200) < 1e-6


def test_shard_entry_points_validate_before_touching_the_device():
    """Gaussian-sharded C-ABI (gsr_shard_*): ownership and slice arguments are checked up front."""
    lib = _lib.load()
    dummy = C.c_void_p(256)
    host = (C.c_int32 * 1)()
    s = _lib.Settings(64, 64, 1.0, 1.0, 1.0, 0, 1, 0, 0, dummy, dummy, dummy, dummy)
    for stride, phase in [(0, 0), (2, 2), (3, -1)]:
        own = _lib.TileOwner(stride, phase)
        rc = lib.gsr_shard_order(C.byref(s), C.byref(own), 100, dummy, 1 << 20, dummy, host, None)
        assert rc == -1 and b"row_stride" in lib.gsr_last_error()
    shard = _lib.Cloud(10, dummy, dummy, dummy, None, dummy, dummy, None)
    # slice [95, 95+10) does not fit P_total = 100; slice shorter than the shard
    assert lib.gsr_shard_preprocess(C.byref(s), C.byref(shard), 100, 95, 10, dummy, 1 << 20, dummy, None) == -1
    assert b"does not fit" in lib.gsr_last_error()
    assert lib.gsr_shard_preprocess(C.byref(s), C.byref(shard), 100, 0, 5, dummy, 1 << 20, dummy, None) == -1
    peers = (C.c_void_p * 9)(*([256] * 9))
    assert lib.gsr_shard_preprocess_p2p(C.byref(s), C.byref(shard), 100, 0, 10, peers, 9, 0, 1 << 20, dummy, None) == -1
    assert b"world" in lib.gsr_last_error()
    assert lib.gsr_shard_preprocess_p2p(C.byref(s), C.byref(shard), 100, 0, 10, peers, 2, 2, 1 << 20, dummy, None) == -1
    ev = _lib.ExchangeView()
    assert lib.gsr_view_exchange(dummy, -1, C.byref(ev)) == -1


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_python_sh_colour_path_of_render_mirror(deg):
    """render()'s ``pipe.convert_SHs_python`` branch (gaussian_renderer.py:_python_sh_colors) against an independent
    restatement of the reference's eval_sh (tests/test_oracle_kat.py)."""
    from types import SimpleNamespace
    from gaussianeditor_b200 import gaussian_renderer as GR
    from test_oracle_kat import _eval_sh_numpy
    g = torch.Generator().manual_seed(deg)
    P = 40
    xyz = torch.randn(P, 3, generator=g, dtype=torch.float64)
    feats = torch.randn(P, 16, 3, generator=g, dtype=torch.float64)
    campos = torch.tensor([0.3, -1.0, 2.0], dtype=torch.float64)
    pc = SimpleNamespace(get_features=feats, get_xyz=xyz, active_sh_degree=deg)
    got = GR._python_sh_colors(pc, campos).numpy()
    d = (xyz - campos).numpy()
    d = d / np.linalg.norm(d, axis=1, keepdims=True)
    sh = feats.numpy().transpose(0, 2, 1)                                # [P, 3, M] like the reference's shs_view
    want = np.maximum(_eval_sh_numpy(deg, sh, d) + 0.5, 0.0)
    assert np.allclose(got, want, rtol=1e-12, atol=1e-12)


def test_product_package_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under gaussianeditor_b200/ or diff_gaussian_rasterization/ may
    import, load or execute it (no CPU fallback can hide behind the product path)."""
    bad = []
    for top in ("gaussianeditor_b200", "diff_gaussian_rasterization"):
        for dp, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                    text = open(os.path.join(dp, f), errors="replace").read()
                    if re.search(r"^\s*(from|import)\s+oracle\b|oracle/_ref|cpu_oracle|liboracle|libdgr_ref", text, re.M):
                        bad.append(os.path.join(dp, f))
    assert bad == []


@pytest.mark.parametrize("stride,phase", [(1, 0), (2, 1), (3, 0), (8, 5)])
def test_tile_count_difference_array_identities(stride, phase):
    """The arithmetic behind csrc/tile_binning.cu, restated in numpy: every visible Gaussian adds +1/-1/-1/+1 at the four
    corners of its tile rectangle; (a) the 2-D prefix sum of that array is the per-tile instance count, and (b) the total
    over the tiles of the owned rows (ty % stride == phase) is the plain weighted sum
    sum_entries diff[y][x] * (gx - x) * #owned rows >= y  -- which is how R reaches the host without any prefix pass."""
    rng = np.random.default_rng(stride * 10 + phase)
    gx, gy, n = 13, 11, 400
    x0 = rng.integers(0, gx, n); y0 = rng.integers(0, gy, n)
    x1 = np.minimum(gx, x0 + rng.integers(0, 5, n)); y1 = np.minimum(gy, y0 + rng.integers(0, 6, n))   # some empty rects
    diff = np.zeros((gy + 1, gx + 1), dtype=np.int64)
    brute = np.zeros((gy, gx), dtype=np.int64)
    for a, b, c, d in zip(x0, y0, x1, y1):
        if c > a and d > b:
            diff[b, a] += 1; diff[b, c] -= 1; diff[d, a] -= 1; diff[d, c] += 1
            brute[b:d, a:c] += 1
    counts = diff.cumsum(0).cumsum(1)[:gy, :gx]
    assert np.array_equal(counts, brute)
    owned = np.array([(ty % stride) == phase for ty in range(gy)])
    rows_from = np.array([owned[y:].sum() for y in range(gy + 1)])            # owned rows with ty >= y
    weights = rows_from[:, None] * (gx - np.arange(gx + 1))[None, :]
    assert int((diff * weights).sum()) == int(brute[owned].sum())
    # ranges: exclusive scan of the owned tiles' counts in row-major order, (0, 0) for empty tiles (the reference's memset)
    flat = np.where(owned[:, None], brute, 0).reshape(-1)
    excl = np.concatenate([[0], flat.cumsum()[:-1]])
    ranges = [(int(e), int(e + c)) if c else (0, 0) for e, c in zip(excl, flat)]
    assert ranges[-1][1] in (0, int(flat.sum())) and all(b - a == c for (a, b), c in zip(ranges, flat))
