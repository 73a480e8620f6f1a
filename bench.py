#!/usr/bin/env python
"""bench.py -- forward+backward Mpixels/s of the differentiable Gaussian rasterizer on BASELINE config 3
(1M synthetic "bicycle-shaped" Gaussians, SH degree 3, 1600x1200), the metric BASELINE.json names.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c3] [--dump-outputs DIR]

One "step" = one pass of the hot path over one camera: GaussianRasterizer.forward (preprocess + tile-count
difference array -> R to the host -> depth order -> scan -> ranges -> two radix passes over tile ids (the first
generates the instances) -> blend, plus output/workspace allocation) + autograd backward of loss = (color * G).sum() with a fixed seeded G ~ U(0,1)[3,H,W]  (BASELINE.md timing
protocol).  The 8 ring cameras of the config are cycled step by step.

  value  : W*H*steps / t / 1e6 with every input resident in HBM before the timed region (CUDA events, max over
           ranks).  Inputs (236 MB of Gaussian parameters + 192 MB of SH gradients written) exceed the 126 MB
           L2, so no separate L2 flush is needed between iterations.
  e2e    : the same step through the public API with HOST buffers: each step copies the camera and the G image
           from pinned host memory (H2D; the 23 MB image on a side stream, overlapping the forward) and reads the
           loss back (D2H into pinned memory) inside the timed region. The read-back is asynchronous and the host
           consumes each step's loss while the NEXT step is already enqueued (what a training loop that logs its
           loss does); all K losses are on the host before the closing event is recorded. Both arms do the same.
  N > 1  : one process per GPU (torchrun), the cloud replicated, every rank renders its own camera stream --
           the path shards over views with no data-path collective ("weak" scaling); value = all ranks' pixels
           / max-over-ranks time.
  --impl reference : the reference's OWN CUDA path (oracle/_ref/libdgr_ref.so = its unmodified .cu files
           compiled for sm_100a) on the same workload; if that library is absent, the CPU oracle port.

  timing : the K timed steps run back to back (a barrier + synchronize on each side); CUDA events on the stream split
           them into 5 regions of about K/5 steps, every number is the MEDIAN of the regions' times per step, and the
           region times are reported under "timing".
  --dump-outputs DIR : after the timed steps, what the last timed step returned to its caller is written as
           DIR/<name>.npy (float32, float64 for the loss): the image and depth in full, and for the per-Gaussian arrays
           (radii and the gradients of all inputs) the rows of a fixed seeded sample of at most 65536 Gaussians, listed
           in gaussian_index.npy. The inputs depend only on the arguments, so two builds can be compared output by
           output.
  N > 1 also runs BASELINE config 4 (5M Gaussians, 1920x1080) through the Gaussian-sharded rasterizer over all N
           GPUs (strong scaling) and reports it under "sharded_c4": ms/step, Mpixels/s, ratio to the plain rasterizer
           on one GPU measured in the same run, bit-comparison of the 8 frames, per-phase times, exchange bytes.
           (--no-sharded skips it; a watchdog prints the headline line anyway if a rank fails inside that leg.)

Extra objects on the JSON line: "roofline" (dominant kernel, CUDA-event timed inside this script; "issue" = the
instruction-issue lens for the FP32-bound render kernels), "cpu_baseline" (CPU oracle on the host cores, rank 0, N=1
only), "stages_ms" (per-stage ms), "workload" descriptors (V, R, R/V, R/Ntile, mean n_contrib), "robustness" (the same
step on a non-saturating variant of config 3 and on config 2, and the miss rate of the speculative second half over
config 5's 48 cameras; --no-robustness skips it), "clocks", "gpu_launches". --option name=value sets a library
option (kernel variants) for A/B runs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

from gaussianeditor_b200 import synth


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                d = json.load(f)
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md recipe). NVML is polled from a thread every
    ~4 ms (a timed region of K steps lasts only K x 1.4 ms); if NVML is unavailable, `nvidia-smi -lms 100` is used."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self.nvml = None
        self.stop_flag = False

    def _nvml_loop(self):
        nv, h = self.nvml
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((float(sm), int(mask)))
            except Exception:
                break
            time.sleep(0.004)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.gpu]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.gpu
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.nvml = (nv, h)
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1.0)
            sm = [r[0] for r in self.rows]
            reasons = sorted(n for n, b in self.BITS.items() if any(r[1] & b for r in self.rows))
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def to_dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


class Workload:
    def __init__(self, name, dev, P=None, opacity_scale=1.0):
        self.name = name
        self.cloud, self.cams = synth.make_config(name, P=P)
        c = self.cloud
        if opacity_scale != 1.0:   # robustness leg: a scene that does not saturate (every list is walked to its end)
            c.opacities = (c.opacities * np.float32(opacity_scale)).astype(np.float32)
        self.dev = dev
        self.P = c.means3D.shape[0]
        self.W, self.H = self.cams[0].image_width, self.cams[0].image_height
        self.t = dict(means3D=to_dev(c.means3D, dev), opacities=to_dev(c.opacities, dev), shs=to_dev(c.shs, dev),
                      scales=to_dev(c.scales, dev), rotations=to_dev(c.rotations, dev))
        self.bg = torch.zeros(3, device=dev)
        rng = np.random.default_rng(1234)
        self.G_host = torch.from_numpy(rng.uniform(size=(3, self.H, self.W)).astype(np.float32)).pin_memory()
        self.G = self.G_host.to(dev)
        self.cam_host = []
        for cam in self.cams:
            blob = np.concatenate([cam.viewmatrix.ravel(), cam.projmatrix.ravel(), cam.campos.ravel(),
                                   np.zeros(1, np.float32)]).astype(np.float32)
            self.cam_host.append(torch.from_numpy(blob).pin_memory())
        self.cam_dev = [b.to(dev) for b in self.cam_host]
        self.copy_stream = torch.cuda.Stream(device=dev)

    def stage_host_inputs(self, k):
        """e2e leg: this step's inputs travel from pinned host memory inside the timed region. The camera (144 B) goes
        on the compute stream; the 23 MB G image is only needed by the loss, so it is copied on a side stream into one
        of two persistent device buffers and overlaps whatever the GPU is doing when the host issues it (the tail of
        the previous step and this step's forward); the compute stream waits for it right before the loss. The copy
        takes 0.42 ms at the measured 54 GB/s (`e2e.h2d_GBps_measured`). A buffer is reused only after the backward
        that read it (two steps earlier) has finished -- an event, not an allocation, guards it: per-step allocation
        of the image on the side stream made the caching allocator stall once the run got longer than ~50 steps."""
        cur = torch.cuda.current_stream(self.dev)
        blob = self.cam_host[k].to(self.dev, non_blocking=True)
        if not hasattr(self, "_G_dev"):
            self._G_dev = [torch.empty_like(self.G) for _ in range(2)]
            self._G_free = [None, None]
            self._slot = 0
        slot = self._slot
        self._slot ^= 1
        with torch.cuda.stream(self.copy_stream):
            if self._G_free[slot] is not None:
                self.copy_stream.wait_event(self._G_free[slot])
            self._G_dev[slot].copy_(self.G_host, non_blocking=True)
        self._cur_slot = slot
        return blob, self._G_dev[slot]

    def join_host_inputs(self):
        torch.cuda.current_stream(self.dev).wait_stream(self.copy_stream)

    def read_back(self, loss):
        """e2e leg: D2H of the step's result into pinned memory, asynchronously; returns a handle whose wait() gives
        the float once the copy has landed."""
        if not hasattr(self, "_loss_host"):
            self._loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
            self._loss_slot = 0
        buf = self._loss_host[self._loss_slot]
        self._loss_slot ^= 1
        buf.copy_(loss.detach().reshape(1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        self._G_free[self._cur_slot] = ev   # forward, loss and backward of this step are behind this event
        return PendingLoss(buf, ev)


class PendingLoss:
    def __init__(self, buf, ev):
        self.buf, self.ev = buf, ev

    def wait(self) -> float:
        self.ev.synchronize()
        return float(self.buf[0])


# ---------------------------------------------------------------------------------------------------------
# ours: through the public drop-in API
# ---------------------------------------------------------------------------------------------------------
class OursRunner:
    impl = "ours"

    def __init__(self, wl: Workload):
        from gaussianeditor_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
        self.GRS, self.GR = GaussianRasterizationSettings, GaussianRasterizer
        self.wl = wl
        self.leaf = {k: v.clone().requires_grad_(True) for k, v in wl.t.items()}
        self.means2D = torch.zeros_like(self.leaf["means3D"], requires_grad=True)

    def _settings(self, cam, blob):
        wl = self.wl
        return self.GRS(image_height=wl.H, image_width=wl.W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=wl.bg,
                        scale_modifier=1.0, viewmatrix=blob[0:16].view(4, 4), projmatrix=blob[16:32].view(4, 4),
                        sh_degree=wl.cloud.sh_degree, campos=blob[32:35], prefiltered=False, debug=False)

    def step(self, i, host=False):
        wl, L = self.wl, self.leaf
        k = i % len(wl.cams)
        if host:
            blob, G = wl.stage_host_inputs(k)
        else:
            blob, G = wl.cam_dev[k], wl.G
        rast = self.GR(self._settings(wl.cams[k], blob))
        for v in L.values():
            v.grad = None
        self.means2D.grad = None
        color, radii, depth = rast(means3D=L["means3D"], means2D=self.means2D, opacities=L["opacities"], shs=L["shs"],
                                   scales=L["scales"], rotations=L["rotations"])
        if host:
            wl.join_host_inputs()
        loss = (color * G).sum()
        loss.backward()
        self.last_out = (color, depth, radii, loss)
        if host:
            return wl.read_back(loss)
        return loss

    def outputs(self):
        """What the last step handed back to its caller: image, depth, radii, loss and the input gradients."""
        color, depth, radii, loss = self.last_out
        L = self.leaf
        return dict(color=color, depth=depth, radii=radii, loss=loss, grad_means3D=L["means3D"].grad,
                    grad_means2D=self.means2D.grad, grad_opacities=L["opacities"].grad, grad_shs=L["shs"].grad,
                    grad_scales=L["scales"].grad, grad_rotations=L["rotations"].grad)

    def describe(self):
        from gaussianeditor_b200.rasterizer import _RasterizeGaussians, forward_state_views
        st = _RasterizeGaussians.last_state
        v = forward_state_views(st)
        V = int((st.radii > 0).sum())
        ntile = v["ranges"].shape[0]
        return dict(P=st.P, V=V, R=st.num_rendered, R_per_V=st.num_rendered / max(V, 1),
                    R_per_tile=st.num_rendered / ntile, mean_n_contrib=float(v["n_contrib"].float().mean()),
                    Ntile=ntile)


# ---------------------------------------------------------------------------------------------------------
# reference: the reference's own CUDA sources (oracle/_ref) behind its glue restated in oracle/ref_cuda.py
# ---------------------------------------------------------------------------------------------------------
class ReferenceCudaRunner:
    impl = "reference"

    def __init__(self, wl: Workload):
        from oracle import ref_cuda
        self.R = ref_cuda.ReferenceRasterizer()
        self.wl = wl

    def step(self, i, host=False):
        wl = self.wl
        k = i % len(wl.cams)
        cam = wl.cams[k]
        if host:
            blob, G = wl.stage_host_inputs(k)
        else:
            blob, G = wl.cam_dev[k], wl.G
        common = dict(means3D=wl.t["means3D"], shs=wl.t["shs"], colors_precomp=None, scales=wl.t["scales"],
                      rotations=wl.t["rotations"], cov3D_precomp=None, bg=wl.bg, viewmatrix=blob[0:16],
                      projmatrix=blob[16:32], campos=blob[32:35], tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
                      sh_degree=wl.cloud.sh_degree)
        color, radii, depth, R = self.R.forward(opacities=wl.t["opacities"], image_height=wl.H, image_width=wl.W,
                                                **common)
        if host:
            wl.join_host_inputs()
        loss = (color * G).sum()
        # autograd of loss = (color*G).sum() hands dL/dcolor = G to the rasterizer's backward
        self.g = self.R.backward(dL_dcolor=G, radii=radii, R=R, **common)
        self.last = (radii, R)
        self.last_out = (color, depth, loss)
        if host:
            return wl.read_back(loss)
        return loss

    def outputs(self):
        color, depth, loss = self.last_out
        g = self.g
        return dict(color=color, depth=depth, radii=self.last[0], loss=loss, grad_means3D=g["dL_dmeans3D"],
                    grad_means2D=g["dL_dmeans2D"], grad_opacities=g["dL_dopacity"], grad_shs=g["dL_dsh"],
                    grad_scales=g["dL_dscales"], grad_rotations=g["dL_drotations"])

    def describe(self):
        radii, R = self.last
        V = int((radii > 0).sum())
        ntile = ((self.wl.W + 15) // 16) * ((self.wl.H + 15) // 16)
        return dict(P=self.wl.P, V=V, R=int(R), R_per_V=R / max(V, 1), R_per_tile=R / ntile, Ntile=ntile)


DUMP_ROWS = 65536


def dump_outputs(outs, P, out_dir):
    """Writes the arrays of `outs` as out_dir/<name>.npy: per-Gaussian arrays (first axis P) on a fixed seeded sample
    of DUMP_ROWS Gaussians (gaussian_index.npy), the rest in full; float32, the loss in float64. Returns bytes written."""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.arange(P) if P <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(P, DUMP_ROWS, replace=False))
    arrays = {"gaussian_index": idx.astype(np.float64)}
    for name, t in outs.items():
        a = t.detach().cpu().numpy()
        if name != "loss" and a.ndim and a.shape[0] == P:
            a = a[idx]
        arrays[name] = a.astype(np.float64 if name == "loss" else np.float32)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs would write {total} bytes"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def cpu_oracle_time(name, P=None, threads=None, budget_s=12.0, max_steps=8):
    """fwd+bwd steps of the workload (cameras cycled like the GPU arm) on the CPU oracle (oracle/liboracle_cpu.so,
    OpenMP, all host threads): one untimed warm-up step, then steps until ~budget_s of CPU work or max_steps.
    Returns (seconds per step, pixels per step, threads, steps timed)."""
    from oracle import cpu_oracle
    cloud, cams = synth.make_config(name, P=P)
    G = np.random.default_rng(1234).uniform(size=(3, cams[0].image_height, cams[0].image_width)).astype(np.float32)

    def one(k):
        f = cpu_oracle.forward_from(cloud, cams[k % len(cams)])
        f.backward(G)
        f.close()
    one(0)
    n, t0 = 0, time.perf_counter()
    while n < max_steps and (n == 0 or time.perf_counter() - t0 < budget_s):
        one(n)
        n += 1
    dt = (time.perf_counter() - t0) / n
    return dt, cams[0].image_width * cams[0].image_height, cpu_oracle.num_threads(), n


def alg_bytes(desc, M, Msh, W, H):
    """Compulsory HBM traffic per stage of OUR pipeline (DESIGN.md 'Algorithmic bytes'); bytes."""
    P, V, R, Nt = desc["P"], desc["V"], desc["R"], desc["Ntile"]
    npix = W * H
    return {
        # in: mean12+scale12+rot16+opacity4 for all P, SH rows only for z-visible; out: record48 (visible) + radii4+tiles4+clamped1+key4+ident4
        "preprocess_fwd": P * 44 + V * 12 * Msh + V * 48 + P * 17,
        "depth_order_scan": 4 * (8 + 8) * P + 4 * P + 8 * P + 4 * P,   # 4 radix passes r+w of (key,val) + hist + scan gather/write
        # binning_variant 0 (CUB): emit kernel + histogram + 2 passes over (u16 key, u32 val) + ranges from the sorted keys
        "emit_instances": P * 8 + V * (16 + 4 + 4) + 8 * R,
        # binning_variant 1 (tile_binning.cu): pass 1 generates (reads offsets/order/record/radius of the visible
        # Gaussians) and writes 6 B per instance, pass 2 reads 6 B and writes 6 B
        "tile_sort": 18 * R + 28 * V + 4 * P,
        # tile_count + tile_prefix: replicas of the difference array in, ranges out (no pass over the instances)
        "tile_ranges": 8 * Nt + 4 * 17 * (Nt + 200),
        "render_fwd": (4 + 48) * R + 8 * Nt + 24 * npix,                 # upper bound: whole lists; early-out reads less
        "render_bwd": (4 + 48) * R + 20 * npix + 36 * R + 48 * P,
        "preprocess_bwd": P * 5 + V * (48 + 44 + 12 * Msh) + P * (56 + 24 + 12 * M),
    }


def robustness_leg(impl, dev, steps=8):
    """Outside the headline: the same fwd+bwd step on two more workloads, so that the speed-up is not a property of one
    saturated scene. Each arm reports its own ms/step; the reader divides the two lines.
      c3_nonsaturating : config 3 with every opacity x 0.03 -> alpha <= 0.03, no pixel saturates, both render kernels of
                         both implementations walk every tile list to its end (mean n_contrib ~ list length)
      c2               : BASELINE config 2 (100k Gaussians, SH degree 0, 800x800)
    and, for this repository only, the miss rate of the speculative second half over config 5's 48 cameras."""
    out = {}
    for key, name, scale in (("c3_nonsaturating", "c3", 0.03), ("c2", "c2", 1.0)):
        wl = Workload(name, dev, opacity_scale=scale)
        r = OursRunner(wl) if impl == "ours" else ReferenceCudaRunner(wl)
        for i in range(3):
            r.step(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            r.step(i)
        b.record()
        torch.cuda.synchronize()
        d = r.describe()
        out[key] = {"ms_per_step": a.elapsed_time(b) / steps, "mpix_s": wl.W * wl.H * steps / (a.elapsed_time(b) * 1e-3) / 1e6,
                    "R_per_tile": d.get("R_per_tile"), "mean_n_contrib": d.get("mean_n_contrib")}
        del r, wl
        torch.cuda.empty_cache()
    if impl == "ours":
        import gaussianeditor_b200.rasterizer as RZ
        wl = Workload("c5", dev)
        r = OursRunner(wl)
        for i in range(len(wl.cams)):       # first visit of every camera (the hint is per (P, W, H), not per camera)
            r.step(i)
        RZ.SPEC_STATS.update(launched=0, missed=0)
        for i in range(2 * len(wl.cams)):
            r.step(i)
        torch.cuda.synchronize()
        out["speculative_second_half"] = {"workload": "config 5: 500k Gaussians, 512x512, 48 ring cameras cycled twice",
                                          **RZ.SPEC_STATS, "miss_rate": RZ.SPEC_STATS["missed"] / max(RZ.SPEC_STATS["launched"], 1)}
    return out


def sharded_config4(dist, dev, rank, world, steps, warmup, points=None):
    """BASELINE config 4 (5M Gaussians, SH degree 3, 1920x1080) through the Gaussian-sharded rasterizer on all `world`
    GPUs (sparse exchange when peer mappings are available), next to the plain single-GPU rasterizer on rank 0:
    fwd+bwd of loss = (color*G).sum(), 8 ring cameras cycled, CUDA events, max over ranks. Every frame of the timed
    cameras is compared BIT FOR BIT with the single-GPU frame on rank 0. Returns the "sharded_c4" object (rank 0)."""
    from gaussianeditor_b200 import sharded as S
    from gaussianeditor_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    cloud, cams = synth.make_config_cached("c4", P=points)
    P = cloud.means3D.shape[0]
    W, H = cams[0].image_width, cams[0].image_height
    bg = torch.zeros(3, device=dev)
    G = torch.from_numpy(np.random.default_rng(77).uniform(size=(3, H, W)).astype(np.float32)).to(dev)

    def settings(cam):
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        return GaussianRasterizationSettings(image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg,
                                             scale_modifier=1.0, viewmatrix=t(cam.viewmatrix), projmatrix=t(cam.projmatrix),
                                             sh_degree=cloud.sh_degree, campos=t(cam.campos), prefiltered=False, debug=False)
    rs = [settings(c) for c in cams]
    names = ["means3D", "opacities", "shs", "scales", "rotations"]
    rast = S.ShardedGaussianRasterizer(rs[0], P)
    plan = rast.plan
    loc = {k: torch.from_numpy(np.ascontiguousarray(getattr(cloud, k)[plan.base:plan.base + plan.count])).to(dev).requires_grad_(True)
           for k in names}
    lm2 = torch.zeros_like(loc["means3D"], requires_grad=True)

    def sharded_step(i, keep=False):
        rast.raster_settings = rs[i % len(rs)]
        for v in list(loc.values()) + [lm2]:
            v.grad = None
        color, radii, depth = rast(means3D=loc["means3D"], means2D=lm2, opacities=loc["opacities"], shs=loc["shs"],
                                   scales=loc["scales"], rotations=loc["rotations"])
        (color * G).sum().backward()
        return (color.detach(), depth.detach()) if keep else None

    def timed(fn, n, all_ranks=True):
        if all_ranks:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / n
        if all_ranks:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms

    for i in range(max(warmup, 3)):
        sharded_step(i)
    reps = sorted(timed(sharded_step, steps) for _ in range(3))
    ms_sharded = reps[1]
    frames = [sharded_step(i, keep=True) for i in range(len(rs))]
    # per-phase device time (CUDA events between the phases of the autograd path; separate pass, max over ranks)
    phases = None
    if rast.mode == "sparse":
        from gaussianeditor_b200 import sparse_sharded as SS
        acc = {}
        nph = 9
        for i in range(nph):
            dist.barrier()                       # align the ranks: a late starter would show up as barrier wait
            torch.cuda.synchronize()
            SS.TRACE = []
            sharded_step(i)
            torch.cuda.synchronize()
            tr = SS.TRACE
            for (n0, e0), (n1, e1) in zip(tr[:-1], tr[1:]):
                acc.setdefault(n1, []).append(e0.elapsed_time(e1))
        acc = {n: sorted(v)[len(v) // 2] for n, v in acc.items()}   # median over the traced steps
        SS.TRACE = None
        ph_names = list(acc.keys())
        t = torch.tensor([acc[n] for n in ph_names], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        phases = {n: round(float(v), 4) for n, v in zip(ph_names, t.tolist())}
    out = None
    # plain single-GPU rasterizer on the full cloud, rank 0 only (the others wait at the barrier below)
    if rank == 0:
        full = {k: torch.from_numpy(np.ascontiguousarray(getattr(cloud, k))).to(dev).requires_grad_(True) for k in names}
        m2 = torch.zeros_like(full["means3D"], requires_grad=True)
        plain = [GaussianRasterizer(r) for r in rs]

        def plain_step(i, keep=False):
            for v in list(full.values()) + [m2]:
                v.grad = None
            color, radii, depth = plain[i % len(plain)](means3D=full["means3D"], means2D=m2, opacities=full["opacities"],
                                                        shs=full["shs"], scales=full["scales"], rotations=full["rotations"])
            (color * G).sum().backward()
            return (color.detach(), depth.detach()) if keep else None
        for i in range(max(warmup, 3)):
            plain_step(i)
        ms_plain = sorted(timed(plain_step, steps, all_ranks=False) for _ in range(3))[1]
        same = True
        for i in range(len(rs)):
            c, d = plain_step(i, keep=True)
            same = same and torch.equal(c, frames[i][0]) and torch.equal(d, frames[i][1])
        # gradient agreement of rank 0's shard on the last camera (summation order differs: tolerance, not bits)
        sharded_step(len(rs) - 1)
        gerr = 0.0
        for k in names:
            a_, b_ = loc[k].grad.double(), full[k].grad[plan.base:plan.base + plan.count].double()
            gerr = max(gerr, float((a_ - b_).norm() / b_.norm().clamp_min(1e-30)))
        out = {"config": f"BASELINE config 4: P={P}, SH degree {cloud.sh_degree}, {W}x{H}, {len(rs)} ring cameras cycled",
               "n_gpus": world, "mode": rast.mode, "ms_per_step": ms_sharded, "mpix_s": W * H / (ms_sharded * 1e-3) / 1e6,
               "ms_per_step_runs": reps, "plain_1gpu_ms_per_step": ms_plain,
               "plain_1gpu_mpix_s": W * H / (ms_plain * 1e-3) / 1e6, "vs_1gpu_plain": ms_plain / ms_sharded,
               "image_equals_1gpu": bool(same), "frames_compared": len(rs), "grad_rel_l2_vs_1gpu_max": gerr,
               "scaling": "strong"}
        if phases:
            out["phase_ms_max_over_ranks"] = phases
        if rast.mode == "sparse":
            from gaussianeditor_b200 import sparse_sharded as SS
            last = SS._SparseShardedRasterize.last
            out.update(seg_cap=last["cap"], largest_segment=last["max_count"], candidates_per_rank=world * last["cap"],
                       redone_forwards=rast.sparse_pool.redo,
                       exchange_bytes_per_rank={"records_out~": 48 * world * last["max_count"], "frame_rows_out": 16 * W * H // world * (world - 1),
                                                "acc_rows_out~": 48 * world * last["max_count"]})
        del full, m2
    else:
        sharded_step(len(rs) - 1)
    dist.barrier()
    del frames
    import gc
    gc.collect()
    rast.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3")
    ap.add_argument("--points", type=int, default=None, help="override the Gaussian count (debug only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-robustness", action="store_true", help="skip the extra workloads of the robustness leg")
    ap.add_argument("--option", action="append", default=[], help="library tuning option k=v (A/B measurements only)")
    ap.add_argument("--no-sharded", action="store_true", help="skip the config-4 Gaussian-sharded leg at --gpus N > 1")
    ap.add_argument("--sharded-points", type=int, default=None, help="override config 4's Gaussian count (debug only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        # the sharded leg allocates large workspaces next to collectives on the compute stream (sharded.init_distributed)
        os.environ.setdefault("TORCH_NCCL_AVOID_RECORD_STREAMS", "1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    use_cpu_port = False
    if args.impl == "reference":
        from oracle import ref_cuda
        use_cpu_port = not (ref_cuda.available() and torch.cuda.is_available())

    name = args.config
    cfg = synth.CONFIGS[name]
    metric = "forward+backward Mpixels/s @1M Gaussians 1600x1200"
    config = {"workload": f"BASELINE config 3: 1M synthetic bicycle-shaped Gaussians, SH degree 3, 1600x1200, "
                          f"8 ring cameras cycled, loss=(color*G).sum()" if name == "c3" else f"config {name}",
              "P": args.points or cfg["P"], "sh_degree": cfg["sh_degree"], "image": [cfg["W"], cfg["H"]],
              "l2": "inputs (236 MB params + 192 MB SH grads) exceed the 126 MB L2; no explicit flush",
              "parallelism": f"replicas x{world} (one camera stream per GPU, no data-path collective)"}

    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if use_cpu_port:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs needs the GPU path (the CPU oracle port is not the timed path)")
        # reference arm without the compiled reference: the CPU oracle port, rank 0 only
        if rank != 0:
            return
        dt, npix, thr, nst = cpu_oracle_time(name, P=args.points, max_steps=max(1, min(args.steps, 8)))
        val = npix / dt / 1e6
        line = {"metric": metric, "value": val, "unit": "Mpixels/s", "n_gpus": 0, "steps": nst, "warmup": 1,
                "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "impl": "reference", "config": config,
                "cpu_baseline": {"value": val, "unit": "Mpixels/s", "cores": thr, "kind": "port",
                                 "sample": f"{nst} full steps (fwd+bwd, cameras cycled) of the workload"},
                "e2e": {"value": val, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the rasterizer has no CPU fallback "
                         "(use --impl reference for the CPU oracle port)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    wl = Workload(name, dev, P=args.points)
    runner = OursRunner(wl) if args.impl == "ours" else ReferenceCudaRunner(wl)
    from gaussianeditor_b200 import _lib
    for kv in args.option:
        k, v = kv.split("=")
        _lib.set_option(k, int(v))
    npix = wl.W * wl.H

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    REPEATS = 5

    def timed(n, host):
        """The n timed steps run back to back between a barrier + synchronize on each side; CUDA events recorded on
        the stream split them into REPEATS regions of about n / REPEATS steps, and the MEDIAN time per step over the
        regions (max over ranks) is reported, as the time of n steps: one host hiccup (GC, a page fault, a neighbour
        rank's launch burst) in a single region of 20 steps used to move the number by 10-20 %. Python's cyclic GC is
        paused during the steps for the same reason."""
        import gc
        sizes = [n // REPEATS + (1 if r < n % REPEATS else 0) for r in range(min(REPEATS, n))]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(sizes) + 1)]
        inner_ends = {int(e) - 1: r + 1 for r, e in enumerate(np.cumsum(sizes)[:-1])}   # last step of a region -> event
        gc.collect()
        gc.disable()
        try:
            barrier()
            ev[0].record()
            pending, losses = None, []
            for i in range(n):
                cur = runner.step(i + rank * 3, host=host)
                if host:  # consume step i-1's loss on the host while step i runs on the GPU
                    if pending is not None:
                        losses.append(pending.wait())
                    pending = cur
                if i in inner_ends:
                    ev[inner_ends[i]].record()
            if pending is not None:
                losses.append(pending.wait())
                assert len(losses) == n and all(np.isfinite(losses))
            ev[-1].record()
            barrier()
        finally:
            gc.enable()
        runs = torch.tensor([ev[r].elapsed_time(ev[r + 1]) for r in range(len(sizes))], device=dev)
        if dist is not None:
            dist.all_reduce(runs, op=dist.ReduceOp.MAX)
        runs = runs.tolist()
        return statistics.median(ms / k for ms, k in zip(runs, sizes)) * n, runs

    for i in range(max(args.warmup, 3)):
        runner.step(i + rank * 3)
    launches0 = _lib.launch_count() if args.impl == "ours" else 0
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, ms_runs = timed(args.steps, host=False)
    clocks = sampler.stop()
    launches = (_lib.launch_count() - launches0) if args.impl == "ours" else None
    dumped = dump_outputs(runner.outputs(), wl.P, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    for i in range(3):
        runner.step(i, host=True).wait()
    ms_e2e, ms_e2e_runs = timed(args.steps, host=True)
    desc = runner.describe()

    # host->device bandwidth of the G image copy alone (explains the e2e/value gap when the copy is the longer leg)
    ca, cb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ca.record()
    for _ in range(4):
        wl.G_host.to(dev, non_blocking=True)
    cb.record()
    torch.cuda.synchronize()
    h2d_gbps = 4 * wl.G_host.numel() * 4 / (ca.elapsed_time(cb) * 1e-3) / 1e9

    value = world * npix * args.steps / (ms * 1e-3) / 1e6
    e2e = world * npix * args.steps / (ms_e2e * 1e-3) / 1e6
    line = {"metric": metric, "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": args.impl,
            "config": config, "clocks": clocks,
            "timing": {"protocol": f"{args.steps} steps back to back (barrier + synchronize on each side), split by "
                                   f"CUDA events into {min(REPEATS, args.steps)} regions; median time per step over "
                                   "the regions, max over ranks",
                       "region_ms": [round(x, 4) for x in ms_runs], "e2e_region_ms": [round(x, 4) for x in ms_e2e_runs]},
            "e2e": {"value": e2e, "unit": "Mpixels/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": 3 * npix * 4 + 36 * 4, "d2h_bytes_per_step": 4,
                    "h2d_GBps_measured": round(h2d_gbps, 1)},
            "workload": desc}
    if dumped is not None:
        line["dump_outputs"] = {"dir": args.dump_outputs, "bytes": dumped}

    if args.impl == "ours":
        line["gpu_launches"] = int(launches)   # over the `steps` timed steps
        # per-stage CUDA-event timing (separate pass so the headline is not perturbed)
        _lib.set_option("profile", 1)
        _lib.profile_read()
        nprof = min(args.steps, 16)
        for i in range(nprof):
            runner.step(i)
        prof = _lib.profile_read()
        _lib.set_option("profile", 0)
        stages = {k: v[0] / max(v[1], 1) for k, v in prof.items() if v[1] > 0}
        line["stages_ms"] = {k: round(v, 4) for k, v in stages.items()}
        M = wl.cloud.shs.shape[1]
        ab = alg_bytes(desc, M, (wl.cloud.sh_degree + 1) ** 2, wl.W, wl.H)
        dom = max(stages, key=stages.get)
        peak, peak_src = measured_peaks()
        ach = ab[dom] / (stages[dom] * 1e-3) / 1e9
        traffic, issue = None, None
        try:  # DRAM bytes and instruction count per launch from the committed ncu --set full capture of the same command
            tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
            with open(tp if os.path.exists(tp) else os.path.join(ROOT, "profiles", "r01_traffic.json")) as f:
                kd = json.load(f)["kernels"][dom]
            traffic = kd["dram_bytes"]
            # second lens for the issue-bound render kernels: warp instructions per launch (ncu) / live kernel time,
            # against 148 SMs x 4 schedulers x 1 instruction per clock at the clock sampled during the timed region
            sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
            peak_inst = 148 * 4 * sm_mhz * 1e6
            issue = {"warp_inst_per_launch": kd["warp_inst"], "achieved_Ginst_s": kd["warp_inst"] / (stages[dom] * 1e-3) / 1e9,
                     "peak_Ginst_s": peak_inst / 1e9, "frac": kd["warp_inst"] / (stages[dom] * 1e-3) / peak_inst,
                     "ipc_per_sm_under_ncu": kd.get("ipc_per_sm")}
        except Exception:
            pass
        line["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                            "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                            "note": "the render kernels are FP32-issue bound, not HBM bound (DESIGN.md section 5): "
                                    "frac is the share of the HBM time the algorithmic bytes would need",
                            "alg_bytes": ab[dom], "kernel_ms": stages[dom], "issue": issue,
                            "all": {k: {"ms": round(stages[k], 4), "alg_GB": round(ab[k] / 1e9, 4),
                                        "GBps": round(ab[k] / (stages[k] * 1e-3) / 1e9, 1),
                                        "frac": round(ab[k] / (stages[k] * 1e-3) / 1e9 / peak, 4)}
                                    for k in stages if k in ab}}
    else:
        line["gpu_launches"] = None
        line["note"] = "reference CUDA kernels (oracle/_ref), torch glue restated in oracle/ref_cuda.py"

    if rank == 0 and world == 1 and not args.no_robustness and name == "c3" and args.points is None:
        try:
            line["robustness"] = robustness_leg(args.impl, dev)
        except Exception as ex:
            line["robustness"] = {"error": repr(ex)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            dt, npx, thr, nst = cpu_oracle_time(name, P=args.points)
            line["cpu_baseline"] = {"value": npx / dt / 1e6, "unit": "Mpixels/s", "cores": thr, "kind": "port",
                                    "sample": f"{nst} full steps (fwd+bwd, cameras cycled, after 1 warm-up step) of the "
                                              "workload on the CPU oracle",
                                    "seconds_per_step": dt}
        except Exception as ex:  # the oracle is a checker; never let it break the bench line
            line["cpu_baseline"] = {"value": None, "error": str(ex)}
    if dist is not None and args.impl == "ours" and not args.no_sharded:
        # BASELINE config 4 under the same clock: the cloud sharded by Gaussian index over all N GPUs (strong scaling)
        # A rank that fails inside this leg would leave the others blocked in a collective: a watchdog guarantees that the
        # headline line (already complete) is still printed and every process exits.
        def give_up():
            if rank == 0:
                line["sharded_c4"] = {"error": "timed out (a rank failed or hung inside the sharded leg)"}
                print(json.dumps(line), flush=True)
            os._exit(0)
        dog = threading.Timer(float(os.environ.get("GSR_SHARDED_TIMEOUT_S", "420")), give_up)
        dog.daemon = True
        dog.start()
        try:
            sh = sharded_config4(dist, dev, rank, world, steps=min(args.steps, 20), warmup=args.warmup,
                                 points=args.sharded_points)
            ok = torch.tensor([1], device=dev)
        except Exception as ex:
            sh = {"error": repr(ex)}
            ok = torch.tensor([0], device=dev)
        if rank == 0:
            line["sharded_c4"] = sh
        if int(ok[0]) == 0:   # do not enter further collectives after a local failure: let the watchdog end the job
            if rank == 0:
                print(json.dumps(line), flush=True)
            os._exit(0)
        dog.cancel()
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
