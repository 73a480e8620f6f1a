"""The reference's OWN callers of the hot path (GaussianEditor's gaussiansplatting/gaussian_renderer/__init__.py and
scene/gaussian_model.py), against what they use and produce:

  * every name, positional slot and keyword the reference's renderer and scene model use on the rasterizer must exist
    in this repository's drop-in package (SURVEY 7.3-10 / 8(f-2));
  * the reference's optimizer surgery (scene/gaussian_model.py:553-641) and gaussianeditor_b200/optim_surgery.py give
    equal parameters and Adam state, bit for bit;
  * the vertex table the reference's ``save_ply`` (:410-445) hands to plyfile (field names, order, float32 values)
    serialises to exactly the bytes gaussianeditor_b200/ply_io.py writes behind the header (SURVEY 8(f-4)), and the
    reference's ``load_ply`` (:447-501) reads our file back to the same tensors.

What these checks compare against is stored under tests/golden/reference/callers_*. Recording it runs the reference's
code itself, imported unchanged, with ``diff_gaussian_rasterization`` resolving to this repository's drop-in package and
the two third-party modules it needs (``plyfile``, ``simple_knn``) stubbed:
    GSR_REFERENCE_ROOT=<GaussianEditor checkout> GSR_RECORD_REFERENCE_DIR=<dir> python -m pytest tests/test_reference_callers.py
then copy <dir>/callers_* to tests/golden/reference/.
"""
import ast
import inspect
import json
import os
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "reference")
REF = os.environ.get("GSR_REFERENCE_ROOT")
RECORD_DIR = os.environ.get("GSR_RECORD_REFERENCE_DIR")
RECORDING = bool(REF and RECORD_DIR)


def _stored_json(name, record):
    """The facts `record()` extracts from the reference's sources: computed while recording, read back otherwise."""
    if RECORDING:
        facts = record()
        os.makedirs(RECORD_DIR, exist_ok=True)
        with open(os.path.join(RECORD_DIR, name + ".json"), "w") as f:
            json.dump(facts, f, indent=1, sort_keys=True)
        return facts
    with open(os.path.join(GOLDEN_DIR, name + ".json")) as f:
        return json.load(f)


def _stored_arrays(name, record):
    """The arrays `record()` gets from running the reference's code: computed while recording, read back otherwise."""
    if RECORDING:
        arrays = {k: np.asarray(v) for k, v in record().items()}
        os.makedirs(RECORD_DIR, exist_ok=True)
        np.savez_compressed(os.path.join(RECORD_DIR, name + ".npz"), **arrays)
        return arrays
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        return dict(z)


class _Captured:
    def __init__(self, data, name):
        self.data, self.name = data, name


def _install_stubs():
    """plyfile: just enough to CAPTURE what the reference hands over / to serve what our reader parsed."""
    ply = types.ModuleType("plyfile")

    class PlyElement:
        @staticmethod
        def describe(data, name):
            return _Captured(data, name)

    class PlyData:
        last_written = None

        def __init__(self, elements):
            self.elements = elements

        def write(self, path):
            PlyData.last_written = (path, self.elements)

        @staticmethod
        def read(path):
            from gaussianeditor_b200 import ply_io
            cols = ply_io.read_vertex_table(path)
            names = list(cols)

            class _El:
                properties = [types.SimpleNamespace(name=n) for n in names]

                def __getitem__(self, k):
                    return cols[k]
            return types.SimpleNamespace(elements=[_El()])
    ply.PlyElement, ply.PlyData = PlyElement, PlyData
    knn = types.ModuleType("simple_knn")
    knn_c = types.ModuleType("simple_knn._C")
    knn_c.distCUDA2 = lambda pts: torch.full((pts.shape[0],), 1e-2)
    knn._C = knn_c
    sys.modules.setdefault("plyfile", ply)
    sys.modules.setdefault("simple_knn", knn)
    sys.modules.setdefault("simple_knn._C", knn_c)
    return sys.modules["plyfile"]


@pytest.fixture(scope="module")
def ref():
    """The reference's modules while recording, None otherwise."""
    if not RECORDING:
        return None
    for p in (ROOT, REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    ply = _install_stubs()
    import diff_gaussian_rasterization as dgr
    assert os.path.dirname(dgr.__file__).startswith(ROOT), "the reference must resolve the drop-in, not its own package"
    import gaussiansplatting.gaussian_renderer as GR
    import gaussiansplatting.scene.gaussian_model as GM
    return types.SimpleNamespace(GR=GR, GM=GM, ply=ply, dgr=dgr)


def _calls(tree, func_pred):
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and func_pred(node.func):
            yield dict(args=len(node.args), keywords=sorted(k.arg for k in node.keywords))


def _parse(rel):
    with open(os.path.join(REF, rel)) as f:
        src = f.read()
    return src, ast.parse(src)


def test_reference_render_uses_only_names_the_drop_in_has(ref):
    import diff_gaussian_rasterization as dgr
    import gaussianeditor_b200.rasterizer as RZ
    assert os.path.dirname(dgr.__file__).startswith(ROOT)

    def record():
        src, tree = _parse("gaussiansplatting/gaussian_renderer/__init__.py")
        assert ref.GR.GaussianRasterizer is RZ.GaussianRasterizer
        assert ref.GR.GaussianRasterizationSettings is RZ.GaussianRasterizationSettings
        return dict(
            imports=[a.name for n in ast.walk(tree) if isinstance(n, ast.ImportFrom)
                     and n.module == "diff_gaussian_rasterization" for a in n.names],
            settings_calls=list(_calls(tree, lambda f: isinstance(f, ast.Name) and f.id == "GaussianRasterizationSettings")),
            rasterizer_calls=list(_calls(tree, lambda f: isinstance(f, ast.Name) and f.id == "rasterizer")),
            unpacks_three_outputs="rendered_image, radii, depth = rasterizer(" in src)
    facts = _stored_json("callers_render", record)
    # the reference binds the drop-in's classes
    assert set(facts["imports"]) == {"GaussianRasterizationSettings", "GaussianRasterizer"}
    for name in facts["imports"]:
        assert getattr(dgr, name) is getattr(RZ, name), name
    # every GaussianRasterizationSettings(...) call: keywords == our NamedTuple fields (order irrelevant, all present)
    fields = set(RZ.GaussianRasterizationSettings._fields)
    assert len(facts["settings_calls"]) >= 2
    for c in facts["settings_calls"]:
        assert c["args"] == 0 and set(c["keywords"]) == fields, set(c["keywords"]) ^ fields
    # GaussianRasterizer(raster_settings=...) and the forward call rasterizer(means3D=..., ...)
    assert "raster_settings" in inspect.signature(RZ.GaussianRasterizer.__init__).parameters
    fwd = set(inspect.signature(RZ.GaussianRasterizer.forward).parameters) - {"self"}
    assert len(facts["rasterizer_calls"]) >= 1
    for c in facts["rasterizer_calls"]:
        kws = set(c["keywords"])
        assert kws <= fwd and {"means3D", "means2D", "opacities"} <= kws, kws - fwd
    # the reference unpacks exactly three outputs: rendered_image, radii, depth
    assert facts["unpacks_three_outputs"]


def test_reference_scene_model_calls_apply_weights_with_our_slot_order(ref):
    import gaussianeditor_b200.rasterizer as RZ
    from gaussianeditor_b200 import gaussian_renderer

    def record():
        _, tree = _parse("gaussiansplatting/scene/gaussian_model.py")
        _, dgr_tree = _parse("gaussiansplatting/submodules/diff-gaussian-rasterization/diff_gaussian_rasterization/"
                             "__init__.py")
        cls = next(n for n in ast.walk(dgr_tree) if isinstance(n, ast.ClassDef) and n.name == "GaussianRasterizer")
        assert callable(ref.GR.camera2rasterizer)
        return dict(
            apply_weights_calls=list(_calls(tree, lambda f: isinstance(f, ast.Attribute) and f.attr == "apply_weights"
                                            and isinstance(f.value, ast.Name) and f.value.id == "rasterizer")),
            rasterizer_methods={fn.name: [a.arg for a in fn.args.args if a.arg != "self"] for fn in cls.body
                                if isinstance(fn, ast.FunctionDef) and not fn.name.startswith("__")},
            camera2rasterizer_params=list(inspect.signature(ref.GR.camera2rasterizer).parameters))
    facts = _stored_json("callers_scene_model", record)
    calls = facts["apply_weights_calls"]
    assert len(calls) == 1 and calls[0]["args"] == 10 and not calls[0]["keywords"]
    # positional slots of scene/gaussian_model.py:821-832 -> our parameter names
    ours = [p for p in inspect.signature(RZ.GaussianRasterizer.apply_weights).parameters if p != "self"]
    assert ours == ["means3D", "means2D", "opacities", "shs", "weights", "scales", "rotations", "cov3Ds_precomp", "cnt",
                    "image_weights"]
    # same as the reference package's own signature (DGR/diff_gaussian_rasterization/__init__.py:311-322)
    assert "apply_weights" in facts["rasterizer_methods"]
    for name, theirs in facts["rasterizer_methods"].items():
        assert hasattr(RZ.GaussianRasterizer, name), name
        mine = [p for p in inspect.signature(getattr(RZ.GaussianRasterizer, name)).parameters if p != "self"]
        assert mine[:len(theirs)] == theirs, (name, mine, theirs)
    # camera2rasterizer(camera, bg, sh_degree), which the scene model imports from the renderer module
    assert list(inspect.signature(gaussian_renderer.camera2rasterizer).parameters) == facts["camera2rasterizer_params"]


def _bare_params(P=13, deg=2, seed=0):
    """Seeded parameters and an Adam optimizer with non-trivial state, laid out like the scene model's."""
    g = torch.Generator().manual_seed(seed)
    K = (deg + 1) ** 2 - 1
    r = lambda *s: torch.nn.Parameter(torch.randn(*s, generator=g))
    p = dict(_xyz=r(P, 3), _features_dc=r(P, 1, 3), _features_rest=r(P, K, 3), _opacity=r(P, 1), _scaling=r(P, 3),
             _rotation=r(P, 4))
    groups = [("xyz", p["_xyz"], 1.6e-4), ("f_dc", p["_features_dc"], 2.5e-3), ("f_rest", p["_features_rest"], 1.25e-4),
              ("opacity", p["_opacity"], 0.05), ("scaling", p["_scaling"], 5e-3), ("rotation", p["_rotation"], 1e-3)]
    opt = torch.optim.Adam([{"params": [t], "lr": lr, "name": n} for n, t, lr in groups], lr=0.0, eps=1e-15)
    for step in range(3):   # build non-trivial Adam state
        opt.zero_grad()
        sum((t * (i + 1 + step)).sum() + (t ** 2).sum() for i, (_, t, _) in enumerate(groups)).backward()
        opt.step()
    return p, opt


def _bare_model(ref, P=13, deg=2, seed=0):
    """A reference GaussianModel on CPU tensors (its __init__ hard-codes device='cuda': bypassed with __new__)."""
    m = ref.GM.GaussianModel.__new__(ref.GM.GaussianModel)
    m.setup_functions()
    m.active_sh_degree = m.max_sh_degree = deg
    p, m.optimizer = _bare_params(P, deg, seed)
    for k, v in p.items():
        setattr(m, k, v)
    return m


def _snapshot(opt, prefix):
    out = {}
    for gr in opt.param_groups:
        p = gr["params"][0]
        out[f"{prefix}/{gr['name']}/param"] = p.detach().numpy().copy()
        for k, v in opt.state.get(p, {}).items():
            out[f"{prefix}/{gr['name']}/{k}"] = v.numpy().copy() if torch.is_tensor(v) else np.asarray(v)
    return out


def _assert_same(ours, stored):
    assert ours.keys() == stored.keys(), set(ours) ^ set(stored)
    for k in ours:
        assert ours[k].dtype == stored[k].dtype and np.array_equal(ours[k], stored[k]), k


def test_optimizer_surgery_equals_the_reference_functions(ref):
    from gaussianeditor_b200 import optim_surgery as OS

    def stages(prune, cat, replace, opt):
        """The three surgeries in sequence (prune, densification_postfix's cat :643-660, reset_opacity's replace),
        then one more Adam step; returns a snapshot after each and the tensors each surgery returns."""
        g = torch.Generator().manual_seed(5)
        out = {}
        keep = torch.rand(13, generator=g) > 0.4
        out.update({f"prune_ret/{k}": v.detach().numpy().copy() for k, v in prune(keep).items()})
        out.update(_snapshot(opt, "prune"))
        ext = {"xyz": torch.randn(4, 3, generator=g), "f_dc": torch.randn(4, 1, 3, generator=g),
               "f_rest": torch.randn(4, 8, 3, generator=g), "opacity": torch.randn(4, 1, generator=g),
               "scaling": torch.randn(4, 3, generator=g), "rotation": torch.randn(4, 4, generator=g)}
        out.update({f"cat_ret/{k}": v.detach().numpy().copy() for k, v in cat(ext).items()})
        out.update(_snapshot(opt, "cat"))
        new_op = torch.randn(opt.param_groups[3]["params"][0].shape, generator=g)
        out.update({f"replace_ret/{k}": v.detach().numpy().copy() for k, v in replace(new_op, "opacity").items()})
        out.update(_snapshot(opt, "replace"))
        opt.zero_grad()
        sum((gr["params"][0] ** 2).sum() for gr in opt.param_groups).backward()
        opt.step()
        out.update(_snapshot(opt, "step"))
        return out

    def record():
        a = _bare_model(ref)
        return stages(lambda keep: a._prune_optimizer(keep),
                      lambda ext: a.cat_tensors_to_optimizer({k: v.clone() for k, v in ext.items()}),
                      lambda t, name: a.replace_tensor_to_optimizer(t.clone(), name), a.optimizer)
    stored = _stored_arrays("callers_optimizer_surgery", record)
    _, opt = _bare_params()
    returned = {}

    def keep_returned(kind, res):
        returned[kind] = res
        return res
    ours = stages(lambda keep: keep_returned("prune", OS.prune_optimizer(opt, keep)),
                  lambda ext: OS.cat_tensors_to_optimizer(opt, {k: v.clone() for k, v in ext.items()}),
                  lambda t, name: OS.replace_tensor_to_optimizer(opt, t.clone(), name), opt)
    _assert_same(ours, stored)
    assert all(isinstance(v, torch.nn.Parameter) and v.requires_grad for v in returned["prune"].values())
    assert {k.split("/")[1] for k in stored if k.startswith("replace_ret/")} == {"opacity"}


@pytest.mark.parametrize("deg", [0, 1, 3])
def test_ply_bytes_equal_what_the_reference_writer_hands_to_plyfile(ref, tmp_path, deg):
    from gaussianeditor_b200 import ply_io
    p, _ = _bare_params(P=11, deg=deg, seed=deg)
    names = ("_xyz", "_features_dc", "_features_rest", "_opacity", "_scaling", "_rotation")
    ours = str(tmp_path / "ours.ply")
    ply_io.write_gaussian_ply(ours, xyz=p["_xyz"].detach().numpy(), features_dc=p["_features_dc"].detach().numpy(),
                              features_rest=p["_features_rest"].detach().numpy(), opacity=p["_opacity"].detach().numpy(),
                              scaling=p["_scaling"].detach().numpy(), rotation=p["_rotation"].detach().numpy())

    def record():
        m = _bare_model(ref, P=11, deg=deg, seed=deg)
        ref_path = str(tmp_path / "ref" / "point_cloud.ply")
        m.save_ply(ref_path)                                   # the REFERENCE's code builds the vertex table
        path, elements = ref.ply.PlyData.last_written
        assert path == ref_path and len(elements) == 1 and elements[0].name == "vertex"
        table = elements[0].data                               # numpy structured array, fields in the reference's order
        # the reference's load_ply (:447-501) on top of our reader (its .cuda() calls are redirected to CPU for the
        # duration of the call)
        m2 = ref.GM.GaussianModel.__new__(ref.GM.GaussianModel)
        m2.setup_functions()
        m2.max_sh_degree = deg
        fns = ["tensor", "zeros", "ones", "empty", "full"]
        orig = {n: getattr(torch, n) for n in fns}

        def on_cpu(fn):
            return lambda *a, **k: fn(*a, **({**k, "device": "cpu"} if k.get("device") == "cuda" else k))
        try:
            for n in fns:
                setattr(torch, n, on_cpu(orig[n]))
            m2.load_ply(ours)
        finally:
            for n in fns:
                setattr(torch, n, orig[n])
        return {"table_fields": np.array(table.dtype.names), "table_formats": np.array([table.dtype[n].str for n in table.dtype.names]),
                "table_bytes": np.frombuffer(table.tobytes(), np.uint8),
                **{"load_ply" + n: getattr(m2, n).detach().numpy() for n in names}}
    stored = _stored_arrays(f"callers_ply_deg{deg}", record)
    fields = [str(n) for n in stored["table_fields"]]
    assert all(f == "<f4" for f in stored["table_formats"])
    raw = open(ours, "rb").read()
    header = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\n" % 11 +
              "".join(f"property float {n}\n" for n in fields) + "end_header\n").encode()   # plyfile's header
    assert raw[:len(header)] == header
    assert raw[len(header):] == stored["table_bytes"].tobytes()   # body: bit for bit the reference's table
    # the reference's load_ply reconstructed the same tensors from our file
    for n in names:
        assert np.array_equal(stored["load_ply" + n], p[n].detach().numpy()), n
