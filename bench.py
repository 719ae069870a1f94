#!/usr/bin/env python
"""bench.py - the hot path of BASELINE.json on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the unmodified reference extension (oracle/_ref)
    python bench.py ... --dump-outputs DIR      # also write the last timed step's outputs as DIR/<name>.npy

Metric (BASELINE.json): fwd+bwd Gaussians/s at 2M points, 1920x1280.
A "step" is one pass of the render hot path over one view: rasterizer forward
(preprocess, depth/tile sort, composite) + backward (composite, preprocess) for
P Gaussians through the drop-in GaussianRasterizer API, i.e. through the C ABI of
libs3g_b200.so.  At N > 1 every rank renders its own view of the same replicated
cloud (one camera per GPU, SURVEY.md 8e) and the per-Gaussian gradients are
all-reduced over NCCL inside the step; `value` = N * P / step time (weak scaling).

One JSON line on stdout (rank 0).  `value`: inputs resident in HBM, CUDA-event
timed, max over ranks.  `e2e`: the same step driven from HOST buffers - camera
matrices and the ground-truth image/depth come from pinned host memory every step,
loss = L1(rgb) + 0.5*L2(depth) is computed on the device and read back.
`roofline`: the dominant kernel (backward composite) timed with CUDA events on its
launching stream inside the library (s3g_profile_*), algorithmic bytes from
SURVEY.md 8d.  `cpu_baseline`: the CPU oracle on a bounded sample of the same
workload on the box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch
import torch.distributed as dist


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline metric and its e2e line; the training-iteration and config 1-4 "
                         "legs time their own fixed counts")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=2_000_000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1280)
    ap.add_argument("--mode", default="sh", choices=["sh", "rgb"])
    ap.add_argument("--workload", default="raster", choices=["raster", "fine"],
                    help="raster: rasterizer fwd+bwd (BASELINE metric, default). fine: full render() of the fine stage - "
                         "HexPlane + decoder + rgb/depth pass + feat pass, fwd+bwd (BASELINE config 3 shape)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-clocks", action="store_true")
    ap.add_argument("--nccl-allreduce", action="store_true",
                    help="N > 1: force ncclAllReduce for the gradient bucket")
    ap.add_argument("--peer-allreduce", action="store_true",
                    help="N > 1: force the peer-memory reduce-scatter/all-gather kernels (default at N <= 3)")
    ap.add_argument("--fused-exchange", action="store_true",
                    help="N > 1: fuse the first half of the gradient exchange into the backward kernel "
                         "(dp.FusedGradExchange).  Measured slower than the stand-alone all-reduce at N = 2 "
                         "(3.75 vs 3.36 ms/step, profiles/r02e_*), so it is opt-in")
    ap.add_argument("--no-train-iteration", action="store_true",
                    help="skip the whole-training-iteration leg (render + loss + stats + Adam, N == 1 only)")
    ap.add_argument("--cpu-sample", type=int, default=500_000)
    ap.add_argument("--no-extra-configs", action="store_true",
                    help="skip the BASELINE config 1-4 legs (bench_configs.py, N == 1 only)")
    ap.add_argument("--configs", default="config1,config2,config3,config4",
                    help="which of the extra config legs to run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (images, radii, gradients) "
                         "as DIR/<name>.npy, at most 64 MB in all, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def dump_outputs(out_dir, arrays, budget=64_000_000):
    """Write each (name, tensor) of `arrays` as out_dir/<name>.npy in float32 (float64 stays float64).  Every array
    gets an equal share of `budget` bytes; one that is larger is replaced by a fixed sample of its flattened elements
    (positions drawn from a generator seeded by the name), so that runs with the same arguments sample the same
    positions."""
    import zlib
    os.makedirs(out_dir, exist_ok=True)
    share = budget // max(len(arrays), 1) - 4096          # room for the .npy header
    for name, x in arrays:
        dt = torch.float64 if x.dtype == torch.float64 else torch.float32
        x = x.detach()
        k = share // (8 if dt == torch.float64 else 4)
        if x.numel() > k:
            idx = np.unique(np.random.default_rng(zlib.crc32(name.encode())).integers(0, x.numel(), k))
            x = x.reshape(-1)[torch.from_numpy(idx).to(x.device)]
        np.save(os.path.join(out_dir, name + ".npy"), x.to(dt).cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "500"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


ref_ext_mod = None


def count_launches(fn):
    """(kernels of libs3g_b200.so, all kernels) launched by one call of fn(), counted by CUPTI through
    torch.profiler in a separate untimed pass; (None, None) if the profiler is unavailable."""
    try:
        from torch.profiler import profile, ProfilerActivity
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        ours = total = 0
        for ev in prof.events():
            if str(getattr(ev, "device_type", "")).endswith("CUDA") and ev.name and not ev.name.startswith(("Memcpy", "Memset", "cuda")):
                total += 1
                if "s3g::" in ev.name:
                    ours += 1
        return ours, total
    except Exception:
        return None, None


def load_impl(name):
    if name == "ours":
        from s3gaussian_b200 import build
        build.build()
        from s3gaussian_b200 import diff_gaussian_rasterization as m
        return m
    import ref_ext
    global ref_ext_mod
    ref_ext_mod = ref_ext
    if not ref_ext.available():
        return None
    return ref_ext.load()


def main():
    a = parse()
    torch.manual_seed(0)            # host-side random inputs (ground-truth images) are the same from run to run
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")

    mod = load_impl(a.impl)
    if mod is None:
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (needs /root/reference at build time)"}))
        return
    from s3gaussian_b200 import synthetic as syn
    import util

    P, W, H = a.points, a.width, a.height
    if a.workload == "fine":
        return main_fine(a, rank, world, local, dev)
    cloud = syn.make_cloud(P, seed=0)
    ring = syn.waymo_ring(W, H, frames=50)
    cam = ring[1 + 3 * ((rank * 6) % 50)]          # front camera of frame 6*rank
    d = util.scene_inputs(cloud, cam, mode=a.mode, sh_degree=3, bg=(0.0, 0.0, 0.0))
    t = {k: (d[k].to(dev).requires_grad_(True) if d[k] is not None else None) for k in util.TENSOR_KEYS}
    m2d = torch.zeros_like(t["means3D"], requires_grad=True)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    gc = torch.randn(3, H, W, device=dev, generator=g)
    gd = torch.randn(1, H, W, device=dev, generator=g)
    leaves = [v for v in list(t.values()) + [m2d] if v is not None]
    settings = util.settings_for(mod, d, dev)
    rast = mod.GaussianRasterizer(settings)

    def zero_grads():
        for v in leaves:
            v.grad = None

    # gradient exchange of the view-parallel step.  Ours: reduce-scatter + all-gather kernels over NVLink peer
    # memory (csrc/peer.cuh, dp.PeerAllReduce); reference arm and fallback: ncclAllReduce of the same flat bucket.
    peer, peer_why = None, None
    # measured on the 8-GPU box (profiles/r01h_*): the peer kernels beat NCCL at 2 GPUs (0.75 vs 0.89 ms for
    # 472 MB), NCCL's in-switch (NVLS) reduction wins at 8 (1.18 vs 1.48 ms); default accordingly
    # opt-in: the exchange fused into the backward kernel (visible rows stored straight into the owner rank's
    # staging over NVLink, one reduce + multicast-gather kernel afterwards)
    fused = None
    if world > 1 and a.impl == "ours" and a.mode == "sh" and a.fused_exchange and not (a.nccl_allreduce or a.peer_allreduce):
        from s3gaussian_b200 import dp
        fused, fused_why = dp.make_fused_grad_exchange(
            {"means3D": (P, 3), "shs": (P, 16, 3), "opacities": (P, 1), "scales": (P, 3), "rotations": (P, 4)}, dev)
        agree = torch.tensor([1 if fused is not None else 0], device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        if int(agree[0]) == 0:
            fused = None
    use_peer = fused is None and (a.peer_allreduce or (world <= 3 and not a.nccl_allreduce))
    if world > 1 and a.impl == "ours" and use_peer:
        from s3gaussian_b200 import dp
        n_grad = sum(v.numel() for v in leaves if v is not m2d)
        peer, peer_why = dp.make_peer_all_reduce(n_grad, dev)
        agree = torch.tensor([1 if peer is not None else 0], device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)          # all ranks take the same path
        if int(agree[0]) == 0:
            peer = None

    # Gradient sink (ours, N > 1): the backward kernel writes the five per-Gaussian gradient tensors straight into
    # the communication bucket (symmetric memory for the peer kernels, a plain flat tensor for NCCL) - no gather copy
    # between the backward and the collective.  The reference arm keeps torch.cat + ncclAllReduce.
    bucket, comm_ev = None, None
    if fused is not None:
        fused.install()
        bucket = fused.bucket
        offs = {k: (o, c) for k, (o, c, _s) in fused.offsets.items()}
        comm_ev = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    elif world > 1 and a.impl == "ours":
        names = {"means3D": t["means3D"], "shs": t["shs"], "colors_precomp": t["colors_precomp"],
                 "opacities": t["opacities"], "scales": t["scales"], "rotations": t["rotations"]}
        offs, n_tot = {}, 0
        for k, v in names.items():
            if v is not None:
                offs[k] = (n_tot, v.numel())
                n_tot += v.numel()
        bucket = peer.flat(n_tot) if peer is not None else torch.zeros(n_tot, device=dev)

        def sink(name, shape, device):
            if name not in offs:
                return None
            o, n = offs[name]
            return bucket[o:o + n].view(shape)
        mod.set_grad_sink(sink)
        comm_ev = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]

    def allreduce_grads():
        if world > 1:
            if bucket is not None:
                comm_ev[0].record()
                if fused is not None:
                    fused.finish()
                elif peer is not None:
                    peer.all_reduce_()
                else:
                    dist.all_reduce(bucket)
                comm_ev[1].record()
                return bucket
            flat = torch.cat([v.grad.reshape(-1) for v in leaves if v is not m2d])
            dist.all_reduce(flat)
            return flat
        return None

    last = {}

    def step_resident():
        zero_grads()
        color, radii, depth = rast(means3D=t["means3D"], means2D=m2d, opacities=t["opacities"], shs=t["shs"],
                                   colors_precomp=t["colors_precomp"], scales=t["scales"],
                                   rotations=t["rotations"], cov3D_precomp=None)
        torch.autograd.backward([color, depth], [gc, gd])
        allreduce_grads()
        if a.dump_outputs:
            last.update(color=color, radii=radii, depth=depth)
        return radii

    # ---- host-driven end-to-end step -------------------------------------
    gt_img = torch.rand(3, H, W).pin_memory()
    gt_dep = (torch.rand(1, H, W) * 50).pin_memory()
    cam_host = torch.cat([d["viewmatrix"].reshape(-1), d["projmatrix"].reshape(-1), d["campos"].reshape(-1)]).pin_memory()
    h2d_bytes = gt_img.numel() * 4 + gt_dep.numel() * 4 + cam_host.numel() * 4
    loss_host = torch.zeros(1).pin_memory()

    copy_stream = torch.cuda.Stream(device=dev)
    copied = torch.cuda.Event()
    # The step's loss, same definition for both arms: Ll1 + 0.5 * compute_depth("l2") with lambda_dssim = 0
    # (train.py:395-419; SSIM is not evaluated when its weight is 0).  Each arm computes it with ITS OWN loss code:
    # ours through s3gaussian_b200.losses (fused kernels, no SSIM stencil), the reference arm through the reference's
    # utils/loss_utils.py functions (torch ops) - plain torch means only where oracle/_ref has no loss_utils.
    if a.impl == "ours":
        from s3gaussian_b200 import losses as _losses

        def e2e_loss(color, img_d, depth, dep_d):
            return _losses.training_loss(color, img_d, depth, dep_d, lambda_dssim=0.0, lambda_depth=0.5)
        e2e_loss_what = "s3gaussian_b200.losses.training_loss(lambda_dssim=0): fused L1 + depth-L2 kernels"
    else:
        _lu = ref_ext_mod.load_ref_loss_utils() if ref_ext_mod.loss_utils_available() else None

        def e2e_loss(color, img_d, depth, dep_d):
            if _lu is None:
                return (color - img_d).abs().mean() + 0.5 * ((depth - dep_d) ** 2).mean()
            return _lu.l1_loss(color, img_d) + 0.5 * _lu.compute_depth("l2", depth, dep_d)
        e2e_loss_what = "reference utils/loss_utils.py l1_loss + 0.5 * compute_depth('l2')" if _lu is not None else \
            "plain torch L1 + 0.5 * L2 (loss_utils.py not in oracle/_ref)"

    def step_e2e():
        zero_grads()
        main = torch.cuda.current_stream()
        cam_d = cam_host.to(dev, non_blocking=True)       # 140 bytes, needed by the first kernel
        # the ground-truth image / depth are first needed at the loss: their H2D copies run on a copy stream
        # underneath the forward pass (same step function for both arms)
        copy_stream.wait_stream(main)
        with torch.cuda.stream(copy_stream):
            img_d = gt_img.to(dev, non_blocking=True)
            dep_d = gt_dep.to(dev, non_blocking=True)
            copied.record(copy_stream)
        rs = settings._replace(viewmatrix=cam_d[:16].view(4, 4), projmatrix=cam_d[16:32].view(4, 4), campos=cam_d[32:35])
        r = mod.GaussianRasterizer(rs)
        color, radii, depth = r(means3D=t["means3D"], means2D=m2d, opacities=t["opacities"], shs=t["shs"],
                                colors_precomp=t["colors_precomp"], scales=t["scales"], rotations=t["rotations"],
                                cov3D_precomp=None)
        main.wait_event(copied)
        img_d.record_stream(main)
        dep_d.record_stream(main)
        loss = e2e_loss(color, img_d, depth, dep_d)
        loss.backward()
        allreduce_grads()
        loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(loss_host[0])

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()          # the reference launches on the legacy stream: device-wide sync
        ms = e0.elapsed_time(e1)
        local_ms["last"] = ms
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = float(tt[0])
        return ms
    local_ms = {}

    if a.impl == "ours":
        from s3gaussian_b200 import _lib
        _lib.profile_enable(False)      # the timed loops run the product build: no per-stage events
    sampler = ClockSampler(local) if (rank == 0 and not a.no_clocks) else None
    if sampler:
        sampler.start()
    ms_res = timed(step_resident, a.steps, max(a.warmup, 3))
    ms_res_local = local_ms["last"]
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        # the gradients of the last timed step are still on the leaves.  N > 1: ours writes them into the reduced
        # bucket, the reference arm reduces a concatenated copy, so there rank 0's own, unreduced gradients are written
        dump_outputs(a.dump_outputs, [(k, last[k]) for k in ("color", "depth", "radii")] +
                     [("grad_" + k, t[k].grad) for k in util.TENSOR_KEYS if t[k] is not None] +
                     [("grad_means2D", m2d.grad)])
    ms_e2e = timed(step_e2e, a.steps, 3)

    radii = step_resident()
    torch.cuda.synchronize()
    V = int((radii > 0).sum())
    launches_ours, launches_all = count_launches(step_resident)

    # ---- roofline of the dominant kernel ----------------------------------
    roofline, stages = None, None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    R = None
    if a.impl == "reference":
        E = torch.Tensor([])
        gg = lambda k: d[k].to(dev).contiguous() if d[k] is not None else E
        R = int(mod._C.rasterize_gaussians(d["bg"].to(dev), gg("means3D"), gg("colors_precomp"), gg("opacities"),
                                           gg("scales"), gg("rotations"), 1.0, gg("cov3D_precomp"),
                                           d["viewmatrix"].to(dev), d["projmatrix"].to(dev), d["tanfovx"], d["tanfovy"],
                                           H, W, gg("shs"), 3, d["campos"].to(dev), False, False)[0])
    if a.impl == "ours":
        from s3gaussian_b200 import _lib
        acc_f, acc_b, n = {}, {}, 5
        _lib.profile_enable(True)       # separate, untimed pass: per-stage CUDA events on the launching stream
        step_resident()
        for _ in range(n):
            step_resident()
            torch.cuda.synchronize()
            for k, v in _lib.profile_read(0).items():
                acc_f[k] = acc_f.get(k, 0.0) + v / n
            for k, v in _lib.profile_read(1).items():
                acc_b[k] = acc_b.get(k, 0.0) + v / n
        _lib.profile_enable(False)
        stages = {"forward_ms": {k: round(v, 4) for k, v in acc_f.items()},
                  "backward_ms": {k: round(v, 4) for k, v in acc_b.items()}}
        color, radii2, depth2, R, _views = util.ours_forward_state(d, dev)
        kern_ms = acc_b.get("render_backward", 0.0)
        # SURVEY.md 8d, backward composite: per instance id 4 + record 40, per pixel 24,
        # per visible Gaussian the 40-byte gradient record it produces
        alg = R * 44 + W * H * 24 + V * 40
        ach = alg / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else 0.0
        # dram__bytes_read+write of one launch of this kernel from the committed ncu --set full capture of the same
        # workload (profiles/ncu_traffic.json); only quoted when the workload is the one that was profiled
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            if (P, W, H, a.mode) == (2_000_000, 1920, 1280, "sh"):
                traffic = int(tj["kernels"]["render_backward_kernel"]["dram_bytes"])
        except Exception:
            pass
        roofline = {"kernel": "render_backward_kernel", "bound": "hbm", "achieved": round(ach, 2), "peak": hbm,
                    "unit": "GB/s", "frac": round(ach / hbm, 4), "traffic": traffic,
                    "algorithmic_bytes": int(alg), "kernel_ms": round(kern_ms, 4), "peak_source": peak_src,
                    "note": "issue-bound all-lanes composite; see DESIGN.md (roofline) for why the HBM fraction is low"}
        sh = a.mode == "sh"
        step_bytes = (P * (480 if sh else 120) + V * (356 if sh else 176) + R * 132 + W * H * 48)
        step_ms = ms_res / a.steps
        roofline["step"] = {"algorithmic_bytes": int(step_bytes), "achieved": round(step_bytes / (step_ms * 1e-3) / 1e9, 2),
                            "frac": round(step_bytes / (step_ms * 1e-3) / 1e9 / hbm, 4)}

    # ---- per-rank breakdown (N > 1): every rank renders a different camera; the step is the max over ranks ----
    per_rank = None
    if world > 1:
        comm_ms = None
        if comm_ev is not None:
            # ranks aligned at the start of the measured step: comm_ms = this rank's wait for the slowest view +
            # the collective itself (the event pair brackets the all-reduce on this rank's stream)
            vals = []
            for _ in range(5):
                torch.cuda.synchronize()
                dist.barrier()
                step_resident()
                torch.cuda.synchronize()
                vals.append(comm_ev[0].elapsed_time(comm_ev[1]))
            comm_ms = round(float(np.median(vals)), 4)
        mine = {"rank": rank, "step_ms": round(ms_res_local / a.steps, 4), "comm_ms": comm_ms, "visible": V,
                "num_rendered": R,
                "render_ms": (round(sum(stages["forward_ms"].values()) + sum(stages["backward_ms"].values()), 4)
                              if stages else None),
                "stages": stages}
        if bucket is not None:
            o, n = offs["means3D"]
            mine["sink_aliased"] = bool(t["means3D"].grad is not None and t["means3D"].grad.data_ptr() == bucket[o:o + n].data_ptr())
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = gathered

    # ---- CPU baseline (rank 0, N == 1) -------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline and a.impl == "ours":
        import dataclasses
        from oracle import splat_oracle
        splat_oracle.build()
        n = min(a.cpu_sample, P)
        sub = syn.GaussianCloud(*(getattr(cloud, f.name)[:n] for f in dataclasses.fields(cloud)))
        ds = util.scene_inputs(sub, cam, mode=a.mode, sh_degree=3, bg=(0.0, 0.0, 0.0))
        t0 = time.time()
        util.oracle_run(splat_oracle, ds, gc.cpu(), gd.cpu())
        dt = time.time() - t0
        cpu = {"value": round(n / dt, 1), "unit": "Gaussians/s", "cores": 1, "kind": "port",
               "sample": f"first {n} Gaussians of the workload cloud, same camera and resolution, fwd+bwd, "
                         f"oracle/splat_oracle.c single thread, {dt:.1f} s; host has {os.cpu_count()} cores"}

    # ---- whole training iteration (N == 1): render + image loss + backward + densify stats + Adam ----
    # SURVEY 8f rows f-1/f-2 either side of the rasterizer.  Ours: fused loss / stats / Adam kernels; reference
    # arm: the reference's own loss_utils + torch.optim.Adam(eps=1e-15) + the torch statements of train.py:489-491.
    # Runs last because Adam moves the parameters (learning rates are tiny: this is a timing leg).
    train_it = None
    if world == 1 and not a.no_train_iteration:
        params = [v for v in leaves if v is not m2d]
        groups = [{"params": [v], "lr": 1e-6, "name": str(i)} for i, v in enumerate(params)]
        acc = torch.zeros(P, 1, device=dev)
        den = torch.zeros(P, 1, device=dev)
        maxr = torch.zeros(P, device=dev)
        img_d, dep_d = gt_img.to(dev), gt_dep.to(dev)
        if a.impl == "ours":
            from s3gaussian_b200 import losses, optim
            opt = optim.FusedAdam(groups, lr=0.0, eps=1e-15)

            def loss_fn(color, depth):
                return losses.training_loss(color, img_d, depth, dep_d)

            def stats_fn(radii):
                optim.add_densification_stats(m2d.grad, radii, acc, den, maxr)
            what = "render fwd+bwd, fused L1+SSIM+depth loss, fused densify stats, FusedAdam step (5 launches + rasterizer)"
        else:
            opt = torch.optim.Adam(groups, lr=0.0, eps=1e-15)
            lu = None
            if ref_ext_mod.loss_utils_available():
                lu = ref_ext_mod.load_ref_loss_utils()

            def loss_fn(color, depth):
                if lu is None:
                    return (color - img_d).abs().mean() + 0.5 * ((depth - dep_d) ** 2).mean()
                return lu.l1_loss(color, img_d) + 0.5 * lu.compute_depth("l2", depth, dep_d) + \
                    0.2 * (1.0 - lu.ssim(color.unsqueeze(0), img_d.unsqueeze(0)))

            def stats_fn(radii):
                vis = radii > 0
                maxr[vis] = torch.max(maxr[vis], radii[vis])
                acc[vis] += torch.norm(m2d.grad[vis, :2], dim=-1, keepdim=True)
                den[vis] += 1
            what = ("reference extension fwd+bwd, reference utils/loss_utils.py (l1 + ssim + depth l2), torch statements of "
                    "train.py:489-491, torch.optim.Adam(eps=1e-15).step()") if lu is not None else \
                   "reference extension + plain L1/L2 loss (loss_utils.py not in oracle/_ref) + torch Adam"

        def step_train():
            zero_grads()
            color, radii, depth = rast(means3D=t["means3D"], means2D=m2d, opacities=t["opacities"], shs=t["shs"],
                                       colors_precomp=t["colors_precomp"], scales=t["scales"],
                                       rotations=t["rotations"], cov3D_precomp=None)
            loss_fn(color, depth).backward()
            with torch.no_grad():
                stats_fn(radii)
            opt.step()
        ms_train = timed(step_train, 10, 3)
        train_it = {"ms": round(ms_train / 10, 4), "iterations": 10, "what": what}

    # ---- BASELINE configs 1-4 as extra keys (N == 1): same legs for both arms, see bench_configs.py ----
    configs = None
    if world == 1 and not a.no_extra_configs:
        import bench_configs
        del t, leaves, gc, gd
        torch.cuda.empty_cache()
        want = set(a.configs.split(","))
        configs = bench_configs.run_all(a.impl, mod, dev, hbm,
                                        skip=[c for c in ("config1", "config2", "config3", "config4") if c not in want])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    step_ms = ms_res / a.steps
    value = world * P / (step_ms * 1e-3)
    e2e_ms = ms_e2e / a.steps
    out = {
        "metric": "fwd+bwd Gaussians/s (rasterizer forward+backward, one view per GPU)",
        "value": round(value, 1), "unit": "Gaussians/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": round(step_ms, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{P} Gaussians ({'SH deg 3 in-kernel' if a.mode == 'sh' else 'precomputed colours'}), "
                               f"{W}x{H}, 1 view/GPU of the 50-frame ring, rasterizer fwd+bwd"
                               + (", all-reduce of per-Gaussian grads" if world > 1 else ""),
                   "collective": (("fused: backward kernel stores visible rows into the owner rank's staging over NVLink, "
                                   "then one reduce + " + ("multimem.st" if fused.mc else "peer-store") + " gather kernel "
                                   "(dp.FusedGradExchange)") if fused is not None else
                                  ("NVLink peer-memory reduce-scatter/all-gather kernels (csrc/peer.cuh)" if peer is not None
                                   else "ncclAllReduce") if world > 1 else None),
                   "points": P, "width": W, "height": H, "visible": V, "num_rendered": R,
                   "parallelism": f"view-parallel dp{world}",
                   "l2": "inputs (>= 470 MB of Gaussian parameters + sort arenas) exceed the 126 MB L2; no flush needed"},
        "e2e": {"value": round(world * P / (e2e_ms * 1e-3), 1), "unit": "Gaussians/s", "ms_per_step": round(e2e_ms, 4),
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4,
                "what": "camera + GT image/depth H2D from pinned memory (images on a copy stream under the forward), render "
                        "through the GaussianRasterizer API, loss = Ll1 + 0.5 * depth-L2 (train.py:395-411, lambda_dssim = 0) "
                        "by " + e2e_loss_what + ", backward, loss D2H"},
        # kernels of libs3g_b200.so per step x steps, counted by CUPTI in an untimed pass (all kernels incl. torch
        # glue in gpu_launches_all)
        "gpu_launches": (launches_ours * a.steps if launches_ours is not None else None) if a.impl == "ours" else 0,
        "gpu_launches_all": launches_all * a.steps if launches_all is not None else None,
        "clocks": clocks,
    }
    if a.impl == "reference":
        out["impl"] = "reference"
        out["gpu_launches"] = 0
        out["cpu_baseline"] = {"value": out["value"], "unit": "Gaussians/s", "cores": 1, "kind": "reference",
                               "sample": "full workload; the reference's implementation of this path is its CUDA "
                                         "extension (oracle/_ref, unmodified, sm_100), timed on the same B200 as "
                                         "north_star asks - there is no CPU implementation of the rasterizer upstream"}
    else:
        out["roofline"] = roofline
        out["stages"] = stages
        if cpu:
            out["cpu_baseline"] = cpu
    if train_it:
        out["train_iteration"] = train_it
    if configs:
        out["configs"] = configs
    if per_rank:
        out["per_rank"] = per_rank
        nbytes = 4 * (bucket.numel() if bucket is not None else sum(v.numel() for v in leaves if v is not m2d))
        cm = [r["comm_ms"] for r in per_rank if r.get("comm_ms")]
        if nbytes and cm:
            out["comm"] = {"bytes": int(nbytes), "ms_max": max(cm),
                           "bus_gbs": round(2 * (world - 1) / world * nbytes / (max(cm) * 1e-3) / 1e9, 1)}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main_fine(a, rank, world, local, dev):
    """BASELINE config 3 shape at --points Gaussians: render(stage='fine', return_dx, render_feat) + the training
    loss terms that touch the path (train.py:395-425 without SSIM / plane regularisers) + backward."""
    from s3gaussian_b200 import synthetic as syn
    import util
    P, W, H = a.points, a.width, a.height
    cloud = syn.make_cloud(P, seed=0)
    ring = syn.waymo_ring(W, H, frames=50)
    cam = ring[1 + 3 * ((rank * 6) % 50)].to(dev)
    cam.time = 0.37 if rank == 0 else cam.time
    state = syn.make_deform_state(0, weight_scale=0.2)
    bg = torch.zeros(3, device=dev)
    gt_img = torch.rand(3, H, W).pin_memory()
    gt_dep = (torch.rand(1, H, W) * 50).pin_memory()
    gt_feat = torch.rand(3, H, W).pin_memory()
    h2d_bytes = (gt_img.numel() + gt_dep.numel() + gt_feat.numel()) * 4
    if a.impl == "ours":
        from s3gaussian_b200 import build, _lib
        build.build()
        from s3gaussian_b200.deformation import deform_network
        from s3gaussian_b200.gaussian_renderer import render, PipelineParams, GaussianModelLite
        import ref_ext
        net = deform_network(ref_ext.ref_deform_args(syn.DEFAULT_RESOLUTION, syn.DEFAULT_MULTIRES))
        net.deformation_net.set_aabb(*[list(x) for x in syn.WAYMO_AABB])
        net.load_state_dict(state, strict=False)
        pc = GaussianModelLite(cloud, net).to(dev)
        leaves = [p for p in pc.parameters()]
        pipe = PipelineParams()
        do_render = lambda: render(cam, pc, pipe, bg, stage="fine", return_dx=True, render_feat=True)
    else:
        import ref_ext
        if not (ref_ext.available() and ref_ext.deform_available()):
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built"}))
            return
        stack = util.RefFineStack(cloud, state, dev, syn.DEFAULT_RESOLUTION, syn.DEFAULT_MULTIRES)
        leaves = stack.leaves()
        do_render = lambda: stack.render(cam, bg, render_feat=True)
    img_d, dep_d, feat_d = gt_img.to(dev), gt_dep.to(dev), gt_feat.to(dev)

    def loss_of(out, im, de, fe):
        return ((out["render"] - im).abs().mean() + 0.5 * ((out["depth"] - de) ** 2).mean() +
                0.001 * ((out["feat"] - fe) ** 2).mean() + 0.001 * out["dx"].abs().mean() + 0.001 * out["dshs"].abs().mean())

    def sync_grads():
        if world > 1:
            flat = torch.cat([v.grad.reshape(-1) for v in leaves if v.grad is not None])
            dist.all_reduce(flat)

    last = {}

    def step_resident():
        for v in leaves:
            v.grad = None
        out = do_render()
        loss_of(out, img_d, dep_d, feat_d).backward()
        sync_grads()
        if a.dump_outputs:
            last.update(out)

    loss_host = torch.zeros(1).pin_memory()

    def step_e2e():
        for v in leaves:
            v.grad = None
        im, de, fe = gt_img.to(dev, non_blocking=True), gt_dep.to(dev, non_blocking=True), gt_feat.to(dev, non_blocking=True)
        loss = loss_of(do_render(), im, de, fe)
        loss.backward()
        sync_grads()
        loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt[0])
        return ms

    sampler = ClockSampler(local) if (rank == 0 and not a.no_clocks) else None
    if sampler:
        sampler.start()
    ms_res = timed(step_resident, a.steps, max(a.warmup, 3))
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, [(k, last[k]) for k in ("render", "depth", "feat", "radii", "dx", "dshs")] +
                     [("grad_viewspace_points", last["viewspace_points"].grad)] +
                     [(f"grad_leaf{i:02d}", v.grad) for i, v in enumerate(leaves) if v.grad is not None])
    ms_e2e = timed(step_e2e, a.steps, 3)
    # ---- whole fine-stage training iteration (N == 1): render + every loss term of train.py:395-425 incl. SSIM and
    # the plane regularisers + backward + densify stats + Adam over Gaussians, planes and decoder ------------------
    train_it = None
    if world == 1 and not a.no_train_iteration:
        acc, den, maxr = torch.zeros(P, 1, device=dev), torch.zeros(P, 1, device=dev), torch.zeros(P, device=dev)
        groups = [{"params": [v], "lr": 1e-7, "name": str(i)} for i, v in enumerate(leaves)]
        if a.impl == "ours":
            from s3gaussian_b200 import losses, optim
            opt = optim.FusedAdam(groups, lr=0.0, eps=1e-15)

            def full_loss(out):
                return (losses.training_loss(out["render"], img_d, out["depth"], dep_d) +
                        0.001 * ((out["feat"] - feat_d) ** 2).mean() + 0.001 * out["dx"].abs().mean() +
                        0.001 * out["dshs"].abs().mean() + pc.compute_regulation(0.01, 0.0001, 0.0001))

            def stats(out):
                optim.add_densification_stats(out["viewspace_points"].grad, out["radii"], acc, den, maxr)
            what = "render(fine) + fused L1/SSIM/depth loss + feat/dx/dshs terms + fused plane regularisers + backward + fused stats + FusedAdam"
        else:
            opt = torch.optim.Adam(groups, lr=0.0, eps=1e-15)
            lu = ref_ext.load_ref_loss_utils() if ref_ext.loss_utils_available() else None
            reg = ref_ext.load_ref_compute_regulation() if ref_ext.regulation_available() else None

            def full_loss(out):
                base = (out["render"] - img_d).abs().mean() + 0.5 * ((out["depth"] - dep_d) ** 2).mean() if lu is None else \
                    lu.l1_loss(out["render"], img_d) + 0.5 * lu.compute_depth("l2", out["depth"], dep_d) + \
                    0.2 * (1.0 - lu.ssim(out["render"].unsqueeze(0), img_d.unsqueeze(0)))
                loss = base + 0.001 * ((out["feat"] - feat_d) ** 2).mean() + 0.001 * out["dx"].abs().mean() + \
                    0.001 * out["dshs"].abs().mean()
                if reg is not None:
                    loss = loss + reg(stack.net, 0.01, 0.0001, 0.0001)
                return loss

            def stats(out):
                vis = out["radii"] > 0
                maxr[vis] = torch.max(maxr[vis], out["radii"][vis])
                acc[vis] += torch.norm(out["viewspace_points"].grad[vis, :2], dim=-1, keepdim=True)
                den[vis] += 1
            what = ("reference deform_network + reference extension (2 passes) + reference loss_utils (l1, ssim, depth l2)"
                    + (" + reference compute_regulation" if reg is not None else "") + " + backward + torch stats + torch.optim.Adam") \
                if lu is not None else "reference stack with plain L1/L2 (loss_utils.py not in oracle/_ref)"

        def step_train():
            for v in leaves:
                v.grad = None
            out = do_render()
            full_loss(out).backward()
            with torch.no_grad():
                stats(out)
            opt.step()
        ms_train = timed(step_train, 10, 3)
        train_it = {"ms": round(ms_train / 10, 4), "iterations": 10, "what": what}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline and a.impl == "ours":
        # north_star: the reference's PyTorch HexPlane/deformation path on the box's host cores
        import ref_ext
        n = 100_000
        if ref_ext.deform_available():
            dn, _ = ref_ext.load_ref_deform()
            cnet = dn(ref_ext.ref_deform_args(syn.DEFAULT_RESOLUTION, syn.DEFAULT_MULTIRES))
            cnet.deformation_net.set_aabb(*[list(x) for x in syn.WAYMO_AABB])
            cnet.load_state_dict(state, strict=False)
            torch.set_num_threads(os.cpu_count())
            x = cloud.xyz[:n].clone().requires_grad_(True)
            sh = cloud.get_features()[:n].clone().requires_grad_(True)
            t = torch.full((n, 1), 0.37)

            def cpu_step():
                for p_ in cnet.parameters():
                    p_.grad = None
                o = cnet(x, cloud.scaling[:n], cloud.rotation[:n], cloud.opacity[:n], sh, t)
                (o[0].sum() + o[5].abs().mean() + o[6].sum() + o[7].abs().mean()).backward()
            cpu_step()
            t0 = time.time()
            reps = 3
            for _ in range(reps):
                cpu_step()
            dt = (time.time() - t0) / reps
            cpu = {"value": round(n / dt, 1), "unit": "Gaussians/s", "cores": torch.get_num_threads(), "kind": "reference",
                   "sample": f"reference scene/deformation.py deform_network fwd+bwd on {n} of the workload's Gaussians, "
                             f"PyTorch CPU, {torch.get_num_threads()} threads of {os.cpu_count()} cores, {dt:.2f} s per pass "
                             "(HexPlane + decoder only: the rasterizer has no CPU implementation upstream)"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    step_ms, e2e_ms = ms_res / a.steps, ms_e2e / a.steps
    out = {"metric": "fwd+bwd Gaussians/s (full fine-stage render(): HexPlane + decoder + rgb/depth pass + feat pass)",
           "value": round(world * P / (step_ms * 1e-3), 1), "unit": "Gaussians/s", "n_gpus": world, "steps": a.steps,
           "warmup": max(a.warmup, 3), "ms_per_step": round(step_ms, 4), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"fine-stage render() of {P} Gaussians at {W}x{H}: default HexPlane (4 levels x 6 planes x 32 ch, "
                                  "35.8M params) + dx/dshs/feat heads, two rasterizer passes, L1+depth+feat+dx+dshs loss, backward",
                      "points": P, "width": W, "height": H, "parallelism": f"view-parallel dp{world}"},
           "e2e": {"value": round(world * P / (e2e_ms * 1e-3), 1), "unit": "Gaussians/s", "ms_per_step": round(e2e_ms, 4),
                   "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4},
           "gpu_launches": ((16 + 16 + 2 + 4) * a.steps) if a.impl == "ours" else 0, "clocks": clocks}
    if a.impl == "reference":
        out["impl"] = "reference"
    elif cpu:
        out["cpu_baseline"] = cpu
    if train_it:
        out["train_iteration"] = train_it
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
