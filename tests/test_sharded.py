"""Gaussian-sharded multi-GPU path (gaussianeditor_b200/sharded.py, BASELINE config 4).

CPU (not gpu): shard plan arithmetic, the three collectives of the dense scheme under gloo (world_size 2), and the
protocol of the sparse exchange restated in numpy and run over gloo (world_size 2 and 3).
GPU: (a) the ownership logic of the kernels with VIRTUAL ranks on one device -- per-rank images must tile the
single-GPU image bit-exactly and the summed accumulators must reproduce its gradients; (b) the real thing, one
process per GPU over NCCL (needs >= 2 GPUs, skipped otherwise).
"""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gaussianeditor_b200 import sharded as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def test_shard_plan_partitions_indices_and_tile_rows():
    for P in (1, 7, 100, 1001, 5_000_000):
        for w in (1, 2, 3, 4, 8):
            plans = [S.ShardPlan(P, w, r) for r in range(w)]
            assert all(p.slice_len == plans[0].slice_len and p.P_pad == plans[0].P_pad for p in plans)
            assert plans[0].P_pad >= P and plans[0].P_pad - P < w
            covered = []
            for p in plans:
                assert 0 <= p.count <= p.slice_len
                covered += list(range(p.base, p.base + p.count)) if P <= 1001 else []
            assert sum(p.count for p in plans) == P
            if P <= 1001:
                assert covered == list(range(P))
            for H in (16, 17, 1080, 1200):
                rows = sorted(r for p in plans for r in p.owned_tile_rows(H))
                assert rows == list(range((H + 15) // 16))


def _gloo_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ex = S.Exchange()
        plan = S.ShardPlan(11, world, rank)
        n, Pp = plan.slice_len, plan.P_pad
        # all-gather in place: every rank fills its own slice of [P_pad, 48] bytes / [P_pad] keys
        rec = torch.zeros(Pp, 48, dtype=torch.uint8)
        rec[plan.base:plan.base + n] = (torch.arange(n * 48, dtype=torch.int64).view(n, 48) % 251 + rank).to(torch.uint8)
        ex.all_gather_inplace(rec)
        ok = True
        for r in range(world):
            want = (torch.arange(n * 48, dtype=torch.int64).view(n, 48) % 251 + r).to(torch.uint8)
            ok &= bool((rec[r * n:(r + 1) * n] == want).all())
        # frame all-reduce: every pixel has one writer (tile rows interleaved) -> sum == concatenation, bit for bit
        H, W = 40, 8
        g = torch.Generator().manual_seed(5)
        full = torch.randn(4, H, W, generator=g)
        frame = torch.zeros(4, H, W)
        for ty in plan.owned_tile_rows(H):
            frame[:, 16 * ty:16 * ty + 16] = full[:, 16 * ty:16 * ty + 16]
        ex.all_reduce_sum(frame)
        ok &= torch.equal(frame, full)
        # reduce-scatter of the accumulators
        acc = torch.full((Pp, S.ACC_STRIDE), float(rank + 1))
        mine = torch.empty(n, S.ACC_STRIDE)
        ex.reduce_scatter_sum(acc, mine)
        ok &= bool((mine == float(sum(range(1, world + 1)))).all())
        out[rank] = ok
    finally:
        dist.destroy_process_group()


def test_gloo_world2_exchange_collectives():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert [out[r] for r in range(world)] == [True] * world


# ---- sparse exchange: the protocol of csrc/sparse_exchange.cu restated in numpy and run over gloo ---------------------
# What the CUDA kernels do per rank (sparse_mask / sparse_scan / sparse_push / sparse_order / sparse_return /
# sparse_gather), with the peer stores replaced by gloo collectives: the claims under test are protocol claims --
# (1) concatenating the per-source segments in rank order keeps GLOBAL index order, so a stable sort of the candidates
#     by the 32-bit depth key alone equals the single-process (depth key, index) order of the Gaussians a rank blends;
# (2) holes (unused segment slots) sort behind every candidate; (3) the count matrix tells every rank alike whether
# a segment overflowed; (4) the return path brings every partial row back to its owner and adding them in ascending
# rank order is deterministic and complete.
CULLED_KEY = np.uint32(0xFFFFFFFF)


def _model_cloud(P, gy, seed=11):
    """Synthetic per-Gaussian facts the exchange depends on: visibility, tile-row span [ymin, ymax), depth key (with ties)."""
    rng = np.random.default_rng(seed)
    visible = rng.random(P) < 0.6
    ymin = rng.integers(0, gy, P)
    span = np.where(rng.random(P) < 0.05, rng.integers(1, gy + 1, P), rng.integers(1, 4, P))   # a few huge splats
    ymax = np.minimum(gy, ymin + span)
    key = rng.integers(0, 50, P).astype(np.uint32)            # few distinct depths: ties must fall back to the index
    return visible, ymin, ymax, key


def _dest_mask(visible, ymin, ymax, world):
    m = np.zeros(visible.shape[0], dtype=np.uint32)
    for i in np.nonzero(visible)[0]:
        if ymax[i] - ymin[i] >= world:
            m[i] = (1 << world) - 1
        else:
            for y in range(ymin[i], ymax[i]):
                m[i] |= 1 << (y % world)
    return m


def _sparse_model_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        P, gy = 1003, 9
        plan = S.ShardPlan(P, world, rank)
        visible, ymin, ymax, key = _model_cloud(P, gy)
        sl = slice(plan.base, plan.base + plan.count)
        mask = _dest_mask(visible[sl], ymin[sl], ymax[sl], world)          # owner side: sparse_mask
        ids = np.arange(plan.base, plan.base + plan.count)
        ok = True
        for cap in (plan.slice_len, None, 3):     # worst case, tight (set below from the matrix), overflowing
            # sparse_scan: slot of Gaussian i in the list for destination d = number of earlier own Gaussians with bit d
            slots = {d: np.cumsum((mask >> d) & 1) - ((mask >> d) & 1) for d in range(world)}
            row = torch.tensor([int(((mask >> d) & 1).sum()) for d in range(world)], dtype=torch.int64)
            rows = [torch.zeros(world, dtype=torch.int64) for _ in range(world)]
            dist.all_gather(rows, row)                                       # the count matrix (peer_barrier with_row)
            matrix = torch.stack(rows).numpy()                               # matrix[s, d] = n[s -> d]
            if cap is None:
                cap = int(matrix.max())
            overflow = int(matrix.max()) > cap
            # sparse_push: segment [src] of every destination's candidate arrays; unused slots = holes with the culled key
            seg_id = np.full((world, cap), -1, dtype=np.int64)
            seg_key = np.full((world, cap), CULLED_KEY, dtype=np.uint32)
            for d in range(world):
                sel = np.nonzero((mask >> d) & 1)[0]
                sel = sel[slots[d][sel] < cap]
                seg_id[d, slots[d][sel]] = ids[sel]
                seg_key[d, slots[d][sel]] = key[sl][sel]
            got_id = [torch.zeros(world, cap, dtype=torch.int64) for _ in range(world)]
            got_key = [torch.zeros(world, cap, dtype=torch.int64) for _ in range(world)]
            dist.all_gather(got_id, torch.from_numpy(seg_id))
            dist.all_gather(got_key, torch.from_numpy(seg_key.astype(np.int64)))
            cand_id = np.concatenate([got_id[s][rank].numpy() for s in range(world)])      # segments in rank order
            cand_key = np.concatenate([got_key[s][rank].numpy() for s in range(world)]).astype(np.uint32)
            ok &= overflow == (cap == 3)
            if overflow:
                continue                                                     # every rank sees it in the same matrix
            # sparse_order: stable sort by the 32-bit key alone
            order = np.argsort(cand_key, kind="stable")
            n_real = int(matrix[:, rank].sum())
            ok &= bool((cand_id[order[n_real:]] == -1).all())                # holes sort last
            full_mask = _dest_mask(visible, ymin, ymax, world)
            mine = np.nonzero((full_mask >> rank) & 1)[0]                    # what a single process would blend here
            want = mine[np.lexsort((mine, key[mine]))]                       # (depth key, global index)
            ok &= bool(np.array_equal(cand_id[order[:n_real]], want))
            # backward: a partial row per candidate, returned to slot (dst=rank, slot) of the owner, gathered in rank order
            part = np.where(cand_id >= 0, np.float32(0.1) * cand_id.astype(np.float32) + np.float32(rank + 1), 0).astype(np.float32)
            back = [torch.zeros(world * cap, dtype=torch.float32) for _ in range(world)]
            dist.all_gather(back, torch.from_numpy(part))                    # back[d][s*cap + slot]
            total = np.zeros(plan.count, dtype=np.float32)
            expect = np.zeros(plan.count, dtype=np.float32)
            for d in range(world):                                           # ascending rank: deterministic
                sel = np.nonzero((mask >> d) & 1)[0]
                total[sel] += back[d].numpy()[rank * cap + slots[d][sel]]
                expect[sel] += np.float32(0.1) * ids[sel].astype(np.float32) + np.float32(d + 1)
            ok &= bool(np.array_equal(total, expect)) and bool((total[mask == 0] == 0).all())
        out[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_sparse_exchange_protocol_keeps_global_order(world):
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_sparse_model_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert [out[r] for r in range(world)] == [True] * world


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
_CASE = {}


def _case():
    """Cloud, camera, dL and the single-GPU result, computed once for all world sizes."""
    if not _CASE:
        from gaussianeditor_b200 import synth
        from util import run_ours
        cloud, cams = synth.make_config("c3", P=60013)  # P not divisible by the world sizes: exercises the padded tail
        cam = cams[0]
        bg = (0.2, 0.5, 0.1)
        dL = np.random.default_rng(3).random((3, cam.image_height, cam.image_width), dtype=np.float32)
        _CASE.update(cloud=cloud, cam=cam, bg=bg, dL=dL, ref=run_ours(cloud, cam, bg=bg, dL=dL))
    return _CASE


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
def test_virtual_ranks_tile_the_single_gpu_result(world):
    """Drive the sharded C-ABI for `world` virtual ranks on one GPU (the all-gather is a shared buffer, the
    all-reduce / reduce-scatter are explicit sums) and compare with the single-GPU rasterizer."""
    from util import cloud_tensors, settings_from, rel_l2
    dev = torch.device("cuda")
    case = _case()
    cloud, cam, bg, dL, ref = case["cloud"], case["cam"], case["bg"], case["dL"], case["ref"]
    H, W = cam.image_height, cam.image_width
    rs = settings_from(cam, bg, cloud.sh_degree, dev)
    full = cloud_tensors(cloud, dev)
    P = cloud.means3D.shape[0]
    empty = torch.empty(0, device=dev)
    plans = [S.ShardPlan(P, world, r) for r in range(world)]
    # stage 1 on every rank into ONE set of global arrays == the state after the all-gather
    geom = radii = None
    bufs = []
    for p in plans:
        sl = lambda t: S.shard_slice(t, p)
        b = S.shard_preprocess(p, rs, sl(full["means3D"]), sl(full["shs"]), empty, sl(full["opacities"]),
                               sl(full["scales"]), sl(full["rotations"]), empty, geom=geom, radii=radii)
        geom, radii = b.geom, b.radii
        bufs.append(b)
    assert torch.equal(radii[:P], ref["radii"])
    for b in bufs:  # each rank continues on its own copy, as after a real all-gather (radii are rebuilt from the records)
        b.geom = geom.clone(); b.radii = torch.full_like(radii, -7)
    frames, accs, Rs = [], [], []
    gdL = torch.from_numpy(dL).to(dev)
    for b in bufs:
        Rs.append(S.shard_order(b))
        frame = torch.zeros(4, H, W, device=dev)
        S.shard_render(b, frame[:3], frame[3:])
        frames.append(frame)
        accs.append(S.shard_backward_render(b, gdL))
    assert sum(Rs) == ref["R"]
    assert all(torch.equal(b.radii[:P], ref["radii"]) and int(b.radii[P:].abs().sum()) == 0 for b in bufs)
    # every pixel is written by exactly one rank, rows interleaved by tile row
    total = torch.stack(frames).sum(0)
    assert torch.equal(total[:3], ref["color"]) and torch.equal(total[3:], ref["depth"])
    for r, f in enumerate(frames):
        rows = torch.zeros(H, dtype=torch.bool, device=dev)
        for ty in plans[r].owned_tile_rows(H):
            rows[16 * ty:16 * ty + 16] = True
        assert float(f[:, ~rows].abs().sum()) == 0.0
        assert torch.equal(f[:3][:, rows], ref["color"][:, rows])
    acc = torch.stack(accs).sum(0)
    names = ["dmean3D", "dmean2D", "dsh", None, "dopacity", "dscale", "drot", None]
    for b in bufs:
        p = b.plan
        grads = S.shard_backward_preprocess(b, acc[p.base:p.base + p.slice_len].contiguous())
        for name, g in zip(names, grads):
            if name is None:
                continue
            want = ref["grads"][name][p.base:p.base + p.count]
            assert g.shape == want.shape
            assert rel_l2(g.cpu().numpy(), want.cpu().numpy()) <= 2e-5, (name, p.rank)


@pytest.mark.gpu
@pytest.mark.parametrize("world,cap_mode", [(2, "full"), (3, "tight"), (8, "tight"), (8, "overflow")])
def test_sparse_exchange_virtual_ranks_match_single_gpu(world, cap_mode):
    """Sparse exchange (csrc/sparse_exchange.cu) with `world` virtual ranks on one GPU: records only travel to the ranks
    whose tile rows they touch, yet frames, depth, radii and the instance total must equal the single-GPU result bit for
    bit and the gathered gradients must match to summation order. `tight` uses the smallest legal segment capacity
    (exactly the largest segment), `overflow` starts too small and must be detected through the count matrix."""
    from gaussianeditor_b200 import sparse_sharded as SS
    from util import cloud_tensors, settings_from, rel_l2
    dev = torch.device("cuda")
    case = _case()
    cloud, cam, bg, dL, ref = case["cloud"], case["cam"], case["bg"], case["dL"], case["ref"]
    H, W = cam.image_height, cam.image_width
    rs = settings_from(cam, bg, cloud.sh_degree, dev)
    full = cloud_tensors(cloud, dev)
    P = cloud.means3D.shape[0]
    empty = torch.empty(0, device=dev)
    plans = [S.ShardPlan(P, world, r) for r in range(world)]
    ranks = [SS.SparseRank(p, dev, W, H) for p in plans]
    SS.link_virtual(ranks)

    def forward(cap):
        steps = []
        for rk in ranks:
            rk.matrix.zero_()    # the "all-reduce" below is a sum: rows of the other ranks must start at zero
        for rk in ranks:
            sl = lambda t: S.shard_slice(t, rk.plan)
            steps.append(SS.sparse_preprocess(rk, rs, sl(full["means3D"]), sl(full["shs"]), empty, sl(full["opacities"]),
                                              sl(full["scales"]), sl(full["rotations"]), empty, cap))
        matrix = torch.stack([rk.matrix for rk in ranks]).sum(0)            # the all-reduce
        for rk in ranks:
            rk.matrix.copy_(matrix)
        out = [SS.sparse_order(st) for st in steps]
        return steps, matrix, out

    cap0 = ranks[0].cap_alloc
    steps, matrix, out = forward(cap0)
    maxc = out[0][1]
    assert all(o[1] == maxc for o in out) and maxc == int(matrix.max()) and 0 < maxc <= cap0
    # the sparse exchange really is sparse: far fewer candidates than world * P
    assert int(matrix.sum()) < 0.75 * world * P
    if cap_mode == "tight":
        steps, matrix, out = forward(maxc)
    elif cap_mode == "overflow":
        steps, matrix, out = forward(max(1, maxc // 2))
        assert all(o[1] == maxc and o[1] > st.cap for o, st in zip(out, steps))      # detected on every rank alike
        steps, matrix, out = forward(SS.next_capacity(maxc, cap0))
    assert sum(o[0] for o in out) == ref["R"]
    for rk in ranks:
        assert torch.equal(rk.radii_local[:rk.plan.count], ref["radii"][rk.plan.base:rk.plan.base + rk.plan.count])
    # render the owned rows into the local frames, then broadcast them into everybody's frame
    for rk in ranks:
        rk.frame.fill_(float("nan"))
    for st in steps:
        SS.sparse_render(st, st.rk.frame[:3], st.rk.frame[3:])
    for rk in ranks:
        SS.frame_broadcast(rk)
    torch.cuda.synchronize()
    for rk in ranks:
        assert torch.equal(rk.frame[:3], ref["color"]) and torch.equal(rk.frame[3:], ref["depth"]), rk.plan.rank
    gdL = torch.from_numpy(dL).to(dev)
    accs = [SS.sparse_backward_render(st, gdL) for st in steps]
    for st, acc in zip(steps, accs):
        SS.sparse_return(st, acc)
    names = ["dmean3D", "dmean2D", "dsh", None, "dopacity", "dscale", "drot", None]
    for st in steps:
        p = st.rk.plan
        grads = SS.sparse_backward_preprocess(st)
        for name, g in zip(names, grads):
            if name is None:
                continue
            want = ref["grads"][name][p.base:p.base + p.count]
            assert g.shape == want.shape
            assert rel_l2(g.cpu().numpy(), want.cpu().numpy()) <= 2e-5, (name, p.rank)
        vis = ref["radii"][p.base:p.base + p.count] > 0
        assert float(grads[0][~vis].abs().sum()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["dense-nccl", "dense-p2p", "sparse"])
def test_two_process_nccl_matches_single_gpu(variant):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    extra = {"dense-nccl": [], "dense-p2p": ["--p2p"], "sparse": ["--mode", "sparse"]}[variant]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "sharded_check.py"), "--config", "c3",
           "--P", "30001"] + extra
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    if r.returncode != 0:   # the interesting part is the children's own traceback, not torchrun's summary
        lines = [l for l in (r.stdout + r.stderr).splitlines() if "Error" in l or "error" in l or "CHECK" in l or "assert" in l]
        print("\n".join(lines[-25:]))
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    assert "SHARDED_CHECK_OK" in r.stdout


def test_workspace_pool_hands_out_distinct_workspaces_in_a_fixed_order():
    """Host logic of the pooled step workspaces (CPU tensors): forwards that are alive at the same time never share
    a workspace, released workspaces are reused lowest index first (what keeps peer workspaces paired across ranks),
    and scratch buffers persist and only grow."""
    import gc
    import weakref
    pool = S.WorkspacePool(exchange=None, geometry_bytes=1024, p2p=False)
    dev = torch.device("cpu")

    class Holder:   # stands in for the ShardBuffers of one forward
        pass
    a, b = Holder(), Holder()
    wa, wb = pool.take(dev), pool.take(dev)
    weakref.finalize(a, pool.give, wa); weakref.finalize(b, pool.give, wb)
    assert wa is not wb and (wa.index, wb.index) == (0, 1) and len(pool.all) == 2
    t1 = wa.get("binning", 1000, torch.uint8, grow=1.25)
    assert t1.numel() == 1000 and wa.get("binning", 900, torch.uint8).data_ptr() == t1.data_ptr()   # reused, not re-allocated
    big = wa.get("binning", 5000, torch.uint8, grow=1.25)
    assert big.numel() == 5000 and wa.bufs["binning"].numel() >= 6250                                # grew with headroom
    del b; gc.collect()
    del a; gc.collect()
    assert [w.index for w in pool.free] == [0, 1]            # released in the other order, still sorted by index
    assert pool.take(dev) is wa and pool.take(dev) is wb and len(pool.all) == 2
    pool.close()
    assert pool.all == [] and pool.free == []


@pytest.mark.gpu
def test_peer_barrier_completes_and_reports_a_missing_rank():
    """gsr_peer_barrier over (virtually) peer-mapped control blocks: two ranks that both arrive pass and leave the error
    word clear; a rank whose peer never arrives gives up after its timeout and the host binding raises instead of using
    the step's data (SparseRank.queue_barrier_check / raise_if_barrier_failed)."""
    from gaussianeditor_b200 import sparse_sharded as SS
    dev = torch.device("cuda")
    plans = [S.ShardPlan(64, 2, r) for r in range(2)]
    ranks = [SS.SparseRank(p, dev, 64, 48) for p in plans]
    SS.link_virtual(ranks)
    ranks[0].matrix[0, :2] = torch.tensor([3, 4], dtype=torch.int32, device=dev)
    ranks[1].matrix[1, :2] = torch.tensor([5, 6], dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):            # the two barrier kernels must be able to run concurrently
        SS.peer_barrier(ranks[1], with_row=True)
    SS.peer_barrier(ranks[0], with_row=True)
    for rk in ranks:
        rk.queue_barrier_check()
    torch.cuda.synchronize()
    for rk in ranks:
        rk.raise_if_barrier_failed()
        assert rk.matrix[:2, :2].cpu().tolist() == [[3, 4], [5, 6]]     # both rows everywhere: the counts all-gather
    SS.peer_barrier(ranks[0])                # rank 1 never arrives at barrier 2
    ranks[0].queue_barrier_check()
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="peer barrier"):
        ranks[0].raise_if_barrier_failed()


def test_sparse_capacity_policy_is_deterministic_bounded_and_converges():
    """Host logic of the sparse exchange's adaptive segment capacity (CPU): every rank derives the next capacity from
    the same global count matrix, so the rule must be a pure function; it must cover the segment it was derived from
    (no redo loop on a static scene), stay within the allocation, and keep the headroom small (every spare slot is a
    hole the depth sort still carries)."""
    from gaussianeditor_b200 import sparse_sharded as SS
    alloc = 625_000
    for mc in (0, 1, 4095, 4096, 138_897, 486_775, 600_000, 625_000, 10_000_000):
        cap = SS.next_capacity(mc, alloc)
        assert cap == SS.next_capacity(mc, alloc) and 1 <= cap <= alloc
        assert cap % 4096 == 0 or cap == alloc
        if mc * 1.10 + 4096 <= alloc:
            assert cap >= mc and cap - mc <= 0.10 * mc + 2 * 4096
        else:
            assert cap >= min(mc, alloc)
    # a scene whose largest segment grows by <10 % per frame never overflows once adapted
    mc = 100_000
    cap = SS.next_capacity(mc, alloc)
    for _ in range(10):
        mc = int(mc * 1.09)
        assert mc <= cap
        cap = SS.next_capacity(mc, alloc)
