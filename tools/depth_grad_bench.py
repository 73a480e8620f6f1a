"""What the depth-image gradient (GaussianRasterizer(..., depth_grad=True)) costs at BASELINE config 3.

    python tools/depth_grad_bench.py [--config c3] [--steps 40] [--regions 5] [--out FILE]

Two arms, the same forward + backward step as bench.py (activated leaf parameters, 8 ring cameras cycled):
  plain : depth_grad=False, loss = (color * G).sum()                               (bench.py's step)
  depth : depth_grad=True,  loss = (color * G).sum() + (depth * G_D).sum()          (gsr_backward_depth)
Both run in one process, region by region alternated; each arm's time is the median of the regions (CUDA events, a
synchronize before every region). Stage times (render_bwd, preprocess_bwd) come from the library's "profile" option in
a separate pass after the timed regions. The card's name and power limit are read in the same run. Prints one JSON line
(and writes it to --out).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from gaussianeditor_b200 import _lib, synth  # noqa: E402
from gaussianeditor_b200.rasterizer import GaussianRasterizer  # noqa: E402
from util import settings_from  # noqa: E402


def card():
    """Name, power limit and max SM clock of cuda:0 (read-only query)."""
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "--id=0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # the measurement stands, but say that the power limit is unknown
        info["power_limit"] = f"unknown ({e.__class__.__name__})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c3")
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--regions", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda")
    cloud, cams = synth.make_config(a.config)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev).requires_grad_(True)
    leaves = dict(means3D=t(cloud.means3D), opacities=t(cloud.opacities), shs=t(cloud.shs), scales=t(cloud.scales),
                  rotations=t(cloud.rotations))
    H, W = cams[0].image_height, cams[0].image_width
    gen = torch.Generator(device=dev).manual_seed(0)
    G = torch.rand(3, H, W, device=dev, generator=gen)
    G_D = torch.randn(H, W, device=dev, generator=gen)
    rasts = {arm: [GaussianRasterizer(settings_from(c, (0, 0, 0), cloud.sh_degree, dev), depth_grad=(arm == "depth"))
                   for c in cams] for arm in ("plain", "depth")}

    def step(i, arm):
        for v in leaves.values():
            v.grad = None
        m2 = torch.zeros_like(leaves["means3D"], requires_grad=True)
        color, _, depth = rasts[arm][i % len(cams)](means2D=m2, **leaves)
        loss = (color * G).sum()
        if arm == "depth":
            loss = loss + (depth[0] * G_D).sum()
        loss.backward()

    arms = ("plain", "depth")
    for arm in arms:
        for i in range(a.warmup):
            step(i, arm)
    torch.cuda.synchronize()
    region_ms = {arm: [] for arm in arms}
    for r in range(a.regions):
        for arm in (arms if r % 2 == 0 else arms[::-1]):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(a.steps):
                step(i, arm)
            e1.record()
            torch.cuda.synchronize()
            region_ms[arm].append(e0.elapsed_time(e1))
    stages = {}
    for arm in arms:
        _lib.set_option("profile", 1)
        _lib.profile_read()
        for i in range(a.steps):
            step(i, arm)
        prof = _lib.profile_read()
        _lib.set_option("profile", 0)
        stages[arm] = {k: prof[k][0] / max(prof[k][1], 1) for k in ("render_bwd", "preprocess_bwd")}
    ms = {arm: float(np.median(region_ms[arm])) / a.steps for arm in arms}
    out = {
        "metric": "fwd+bwd ms/step with and without depth_grad",
        "card": card(),
        "config": f"{a.config}: P={cloud.means3D.shape[0]}, SH degree {cloud.sh_degree}, {W}x{H}, "
                  f"{len(cams)} ring cameras cycled",
        "protocol": f"median of {a.regions} alternated regions of {a.steps} steps per arm, CUDA events",
        "ms_per_step": ms,
        "region_ms": region_ms,
        "spread_pct": {arm: 100.0 * (max(region_ms[arm]) - min(region_ms[arm])) / min(region_ms[arm]) for arm in arms},
        "step_increase_pct": 100.0 * (ms["depth"] / ms["plain"] - 1.0),
        "stages_ms_per_call": stages,
        "stage_increase_pct": {k: 100.0 * (stages["depth"][k] / stages["plain"][k] - 1.0)
                               for k in ("render_bwd", "preprocess_bwd")},
    }
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
