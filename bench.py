#!/usr/bin/env python
"""bench.py — image-pairs/sec of the MicKey inference hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default workload (config.workload): BASELINE configs[2], the largest single-GPU configuration — a batch of 32
synthetic 720x540 pairs per step and per GPU, DINOv2 ViT-B/14, 1024 hypotheses (IT_MATCHES 16 x IT_RANSAC 64),
2048 sampled matches, seeded random-init weights.  With --gpus 8 this is BASELINE configs[3] (B = 256 sharded
32 pairs per GPU, ONE all-gather of the packed [B,13] poses per step; weak scaling).  `--workload c2` runs
configs[1] (one ViT-S pair per step, 512 hypotheses); at N = 1 the default run also reports it as `latency_c2`.

A step = one model(data) call = extraction of both images of every pair + dual-softmax matching + RANSAC pose.
The K timed steps are measured as a block between barrier + torch.cuda.synchronize() with CUDA events (max over
ranks); the block is repeated (`blocks`) and the MEDIAN block gives `value` / `ms_per_step`, min and max are
reported next to it.  `value`: inputs resident in HBM.  `e2e`: the same public API fed PINNED HOST images
(H2D of every image inside the timed region, D2H of the poses).  `roofline*`: CUDA-event timings of each kernel
class taken live in extra profiled steps of this run (mk_profile_*), divided into the algorithmic work stated in
DESIGN.md.  `cpu_baseline` / `--impl reference`: the reference's CPU path (oracle port) on the host cores;
`gpu_eager_baseline`: the same restatement run eagerly on this GPU with an fp16 backbone (the reference's own
`FLOAT16: True` CUDA path, mickey_extractor.py:31-35) — the same-box number to beat.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("MICKEY_SYNTHETIC_BACKBONE", "1")      # BASELINE.json: seeded random-init weights

from mickey_b200.config import mickey_cfg  # noqa: E402
from mickey_b200.weights import synthetic_checkpoint, synthetic_state_dict  # noqa: E402

H_IMG, W_IMG = 720, 540
WORKLOADS = {
    # name: (variant, it_matches, it_ransac, pairs per GPU per step, description)
    "c1": ("vitl", 20, 100, 1, "BASELINE configs[0] model on a synthetic pair: single 720x540 pair, ViT-L/14 (the reference's default backbone), 2000 hypotheses (20x100); "
                               "the reference-CPU number of configs[0] itself (its toy_example JPEGs) is in profiles/r02_c1_reference_cpu.json"),
    "c2": ("vits", 8, 64, 1, "BASELINE configs[1]: single 720x540 synthetic pair, ViT-S/14, 512 hypotheses (8x64), 2048 sampled matches"),
    "c3": ("vitb", 16, 64, 32, "BASELINE configs[2]: batch of 32 synthetic 720x540 pairs, ViT-B/14, dual-softmax matcher, 1024 hypotheses (16x64), 2048 sampled matches"),
}
VIT_DIMS = {"vits": (384, 12), "vitb": (768, 12), "vitl": (1024, 24)}
K_TOY = [[549.7, 0.0, 268.7], [0.0, 549.7, 351.8], [0.0, 0.0, 1.0]]
N_KP = (H_IMG // 14) * (W_IMG // 14)
COLLECT_INST_PER_CELL = 113.4     # thread instructions per cell and group of 8 streams in sampler_collect (ncu: 13.32 M warp inst / 3.76 M cells)


def synthetic_pair(batch, seed):
    g = torch.Generator().manual_seed(seed)
    im0 = torch.rand(batch, 3, H_IMG, W_IMG, generator=g)
    im1 = torch.rand(batch, 3, H_IMG, W_IMG, generator=g)
    K = torch.tensor(K_TOY)[None].repeat(batch, 1, 1)
    return im0, im1, K


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tflops": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "tflops_burst": p["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json; sustained bf16 GEMM, copy bandwidth)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "source": "fallback (B200_PROFILING.md)"}


# ---------------------------------------------------------------------------------------------------------------
# algorithmic work per step (DESIGN.md §Rooflines; SURVEY.md §8d)
# ---------------------------------------------------------------------------------------------------------------
def work_model(D=384, depth=12, n_pairs=1, it_matches=8):
    N, T = N_KP, N_KP + 1
    imgs = 2 * n_pairs
    M = imgs * T
    flops = {
        "vit.patch_embed": 2 * imgs * N * 588 * D,
        "vit.qkv": depth * 2 * M * D * 3 * D, "vit.proj": depth * 2 * M * D * D,
        "vit.fc1": depth * 2 * M * D * 4 * D, "vit.fc2": depth * 2 * M * D * 4 * D,
        "vit.attention": depth * imgs * 4 * T * T * D,
    }
    px = imgs * N
    dims = [D, 512, 256, 128]
    c3 = c1 = 0
    for r in range(3):
        cin, cout = dims[r], dims[r + 1]
        c3 += 4 * 2 * px * 9 * (cin * cout + cout * cout)
        c1 += 4 * 2 * px * cin * cout
    c3 += 3 * 2 * px * 9 * (128 * 64 + 64 * 64) + 2 * px * 9 * (128 * 128 + 128 * 128)
    c1 += 3 * 2 * px * 128 * 64
    flops["head.conv3x3"], flops["head.conv1x1"] = c3, c1
    flops["head.att.qkv"] = 3 * 4 * 2 * px * 128 * 384
    flops["head.att.merge_ln"] = 3 * 4 * 2 * px * 128 * 128
    flops["head.att.mlp0"] = 3 * 4 * 2 * px * 256 * 256
    flops["head.att.mlp2_ln"] = 3 * 4 * 2 * px * 256 * 128
    nbytes = {
        # dual-softmax pass 2 alone: read both descriptor sets + scores, write scores, kp_scores, final_scores
        "match.dual_softmax": n_pairs * (2 * 128 * N * 4 + 2 * N * 4 + 3 * N * N * 4),
        # the matcher as a whole (every match.* launch): the same contract-preserving 47.07 MB per pair
        "match.*": n_pairs * (2 * 128 * N * 4 + 2 * N * 4 + 3 * N * N * 4),
        # solver: final_scores read once (SURVEY.md §8d "RANSAC bytes")
        "solve.sample_outer": n_pairs * (N * N * 4),
        "solve.*": n_pairs * (N * N * 4 + 6 * N * 4 * 2 + 52),
    }
    # the outer sampler is instruction-bound, not HBM-bound: Philox rounds per cell and group of 8 streams
    warp_inst = {"solve.sample_outer": n_pairs * N * N * -(-it_matches // 8) * COLLECT_INST_PER_CELL / 32.0}
    return flops, nbytes, warp_inst


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled through NVML DURING the timed region (the same counters
    `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints; B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.power, self.reasons, self.stop_flag, self.max_sm, self.err = index, [], [], set(), False, None, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            while not self.stop_flag:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1e3)
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception as e:          # noqa: BLE001
            self.err = repr(e)

    def finish(self):
        self.stop_flag = True
        self.join(timeout=2)
        sm = sorted(self.sm)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
               "samples": len(sm), "power_w_max": max(self.power) if self.power else None}
        if self.err:
            out["error"] = self.err
        return out


def usable_cpus():
    """Host threads this process may really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:      # noqa: BLE001
        pass
    return n


def cpu_threads():
    # torch CPU kernels at these sizes stop scaling (and then regress badly) past a few dozen threads
    return min(usable_cpus(), 32)


# ---------------------------------------------------------------------------------------------------------------
# baselines: the reference's path restated by oracle/mickey_oracle.py (pinned to the reference by tests/golden)
# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_run(wl, n_timed, n_warm, threads, budget_s=25.0):
    """fp32 CPU path ('port': the Python reference cannot travel to the GPU box), ONE pair of the workload's model
    configuration per sample.  Returns per-pair seconds."""
    from oracle import mickey_oracle as mo
    variant, im, ir = wl[0], wl[1], wl[2]
    torch.set_num_threads(threads)
    cfg = mickey_cfg(variant, im, ir, float16=False)
    sd = synthetic_state_dict(cfg, seed=0)
    im0, im1, K = synthetic_pair(1, seed=0)
    durs, spent = [], 0.0
    with torch.no_grad():
        for i in range(n_warm + n_timed):
            data = {"image0": im0, "image1": im1, "K_color0": K, "K_color1": K}
            torch.manual_seed(i)
            t0 = time.perf_counter()
            mo.model_forward(sd, data, cfg)
            dt = time.perf_counter() - t0
            spent += dt
            if i >= n_warm:
                durs.append(dt)
            if spent > budget_s and durs:
                break
    return durs


def gpu_eager_run(wl, dev, budget_s=40.0):
    """The reference's eager-CUDA path on THIS GPU: the oracle restatement (same torch ops the reference issues: cuDNN
    convs, cuBLAS GEMMs, materialised T x T attention, torch.multinomial / torch.svd RANSAC) with the backbone in fp16
    (`FLOAT16: True`, mickey_extractor.py:31-35) and fp32 heads / matcher / solver.  The batch is the workload's, halved
    until one step fits the time budget."""
    from oracle import mickey_oracle as mo
    variant, im, ir, B = wl[0], wl[1], wl[2], wl[3]
    cfg = mickey_cfg(variant, im, ir, float16=True)
    sd = {k: v.to(dev) for k, v in synthetic_state_dict(cfg, seed=0).items()}
    sd = {k: (v.half() if (k.startswith(mo.BACKBONE) and v.is_floating_point()) else v) for k, v in sd.items()}
    out = {"kind": "oracle restatement of the reference run eagerly on cuda (fp16 backbone, fp32 heads/matcher/solver)"}

    def step(b):
        im0, im1, K = (t.to(dev) for t in synthetic_pair(b, seed=0))
        data = {"image0": im0, "image1": im1, "K_color0": K, "K_color1": K}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        with torch.no_grad():
            R, t = mo.model_forward(sd, data, cfg)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3, bool(R.abs().sum() > 0)

    b = B
    try:
        while True:
            try:
                step(b)                              # warm-up (cuDNN autotune, allocator)
                dt, ok = step(b)
                if dt > budget_s / 3 and b > 1:
                    b = max(1, b // 2)
                    continue
                break
            except torch.cuda.OutOfMemoryError:
                torch.cuda.empty_cache()
                if b == 1:
                    raise
                b = max(1, b // 2)
        durs = [dt]
        while sum(durs) < min(budget_s / 2, 6.0) and len(durs) < 5:
            d2, ok2 = step(b)
            durs.append(d2)
            ok = ok and ok2
        durs.sort()
        med = durs[len(durs) // 2]
        out.update(value=b / med, unit="pairs/s", pairs_per_step=b, ms_per_step=1e3 * med, steps=len(durs), solver_returned_pose=ok)
    except Exception as e:      # noqa: BLE001
        out.update(value=None, error=repr(e)[:300])
    del sd
    torch.cuda.empty_cache()
    return out


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = cpu_threads()
    # a "step" is one pair of the workload's configuration through the CPU path
    steps, warm = args.steps, max(0, min(args.warmup, 1))
    durs = cpu_reference_run(wl, steps, warm, threads, budget_s=float("inf"))
    val = len(durs) / sum(durs)
    line = {"impl": "reference", "metric": "image-pairs/sec @720x540", "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": 1e3 * sum(durs) / len(durs), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl[4], "note": "reference CPU path (oracle port of the PyTorch reference), rank 0 only; "
                                                  "each step = ONE pair of the workload's model / hypothesis configuration"},
            "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": threads, "kind": "port",
                             "sample": f"{steps} pair(s) of the workload's configuration ({warm} warm-up), "
                                       f"torch threads = {threads} of {usable_cpus()} usable"},
            "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
class Runner:
    """One workload on this rank's GPU: model, inputs, the two step functions and the block timer."""

    def __init__(self, wl, dev, rank, world):
        from mickey_b200.model import build_model
        from mickey_b200 import dist as mkdist
        self.mkdist, self.dev, self.rank, self.world = mkdist, dev, rank, world
        self.variant, self.im, self.ir, self.B, self.desc = wl
        self.cfg = mickey_cfg(self.variant, self.im, self.ir)
        self.model = build_model(self.cfg, synthetic_checkpoint(self.cfg, seed=0, with_backbone=True))
        self.model.static_outputs = True     # hand out the engine's static output buffers (no per-call clones)
        B = self.B
        im0, im1, K = synthetic_pair(B, seed=rank)
        self.dev_data = {"image0": im0.to(dev), "image1": im1.to(dev), "K_color0": K.to(dev), "K_color1": K.to(dev)}
        self.pin = {"image0": im0.pin_memory(), "image1": im1.pin_memory()}
        self.pose_host = torch.empty(B, 13).pin_memory()

    def step_device(self):
        B = self.B
        data = dict(self.dev_data)
        R, t = self.model(data)
        packed = torch.cat([R.reshape(B, 9), t.reshape(B, 3), data["inliers"].reshape(B, 1)], dim=1)
        poses = self.mkdist.gather_poses(packed)
        self.last = (data, poses)
        return poses

    def step_e2e(self):
        # pinned HOST images go straight into model(): the engine's H2D copies land in its static input buffer
        B = self.B
        data = {"image0": self.pin["image0"], "image1": self.pin["image1"], "K_color0": self.dev_data["K_color0"],
                "K_color1": self.dev_data["K_color1"]}
        R, t = self.model(data)
        packed = torch.cat([R.reshape(B, 9), t.reshape(B, 3), data["inliers"].reshape(B, 1)], dim=1)
        allp = self.mkdist.gather_poses(packed)
        self.pose_host.copy_(allp[self.rank * B:(self.rank + 1) * B], non_blocking=True)
        return allp

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed_block(self, fn, steps, flush=None):
        """K steps between two synchronisation points.  flush given: one event pair per step with a 256 MiB write in
        between (steps strictly one after the other).  Otherwise one event pair around all K steps (steps may overlap
        on the engine's streams; the per-step working set exceeds the L2, see config).  Returns (max over ranks, own)."""
        self.barrier()
        if flush is not None:
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for e0, e1 in evs:
                flush.fill_(1)
                e0.record()
                fn()
                e1.record()
            self.barrier()
            ms = sum(e0.elapsed_time(e1) for e0, e1 in evs)
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            self.barrier()
            ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)       # max over ranks
        return float(t.item()), ms

    def blocks(self, fn, steps, n_blocks, flush=None):
        res = [self.timed_block(fn, steps, flush) for _ in range(n_blocks)]
        mx = sorted(r[0] for r in res)
        own = sorted(r[1] for r in res)
        return {"median_ms": mx[len(mx) // 2], "min_ms": mx[0], "max_ms": mx[-1], "own_median_ms": own[len(own) // 2], "n": n_blocks}


def snapshot_outputs(data, poses, n_cols=256, n_cells=1 << 18):
    """What the caller of a step receives, as float32 host arrays: the gathered [B,13] poses, R, t, inliers and the
    per-keypoint outputs in full; the descriptors and the three N x N score tensors (480 MB each at B = 32) as a fixed
    seeded sample of keypoint columns / cells, the same for every run of a workload."""
    dev = data["dsc0"].device
    B, _, N = data["dsc0"].shape
    g = torch.Generator().manual_seed(0)
    cols = torch.randperm(N, generator=g)[:n_cols].sort().values.to(dev)
    b, i, j = (torch.randint(n, (n_cells,), generator=g).to(dev) for n in (B, N, N))
    out = {"poses": poses}
    for k in ("R", "t", "inliers", "kps0", "kps1", "depth_kp0", "depth_kp1", "scr0", "scr1"):
        out[k] = data[k]
    for k in ("dsc0", "dsc1"):
        out[k + "_sample"] = data[k][:, :, cols]
    for k in ("scores", "kp_scores", "final_scores"):
        out[k + "_sample"] = data[k][b, i, j]
    return {k: v.float().cpu().numpy() for k, v in out.items()}


def stats(blk, steps, pairs_per_step_all_ranks):
    return {"value": pairs_per_step_all_ranks * steps / (blk["median_ms"] / 1e3), "ms_per_step": blk["median_ms"] / steps,
            "ms_per_step_min": blk["min_ms"] / steps, "ms_per_step_max": blk["max_ms"] / steps, "blocks": blk["n"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="steps in each timed block")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS),
                    help="c3 (default: B=32, ViT-B, 1024 hypotheses; the largest single-GPU configuration) or c2 (one ViT-S pair)")
    ap.add_argument("--blocks", type=int, default=0, help="repetitions of the K-step block (default: 5 for c3, 9 for c2)")
    ap.add_argument("--depth", type=int, default=int(os.environ.get("MICKEY_PIPELINE_DEPTH", "0")),
                    help="steps kept in flight on alternating engines/streams (default: 1 for c3, 3 for c2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-c2", action="store_true", help="skip the latency_c2 object of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, float32, ~14 MB for c3; "
                         "the inputs are seeded, so two builds run with the same arguments can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, wl)
        return
    args.warmup = max(args.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(1234 + rank)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def measure(wl_, depth, n_blocks, with_profile=True, dump=False):
        """Full measurement of one workload: single-step latency, pipelined throughput, e2e, per-kernel profile.
        dump: also return the outputs of the last timed throughput step (snapshot_outputs)."""
        r = Runner(wl_, dev, rank, world)
        model, B = r.model, r.B
        # (1) latency: one step at a time (pipeline depth 1), L2 flushed between steps
        model.pipeline_depth = 1
        for _ in range(args.warmup):
            r.step_device()
        ncu_range = os.environ.get("MICKEY_NCU_RANGE") == "1"     # `ncu --profile-from-start off`: capture the latency steps only
        if ncu_range:
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
        lat = r.blocks(r.step_device, args.steps, 3, flush)
        if ncu_range:
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        eng = model._engine()
        # (2) throughput: `depth` steps in flight on alternating engines/streams (inputs are constant device tensors)
        model.pipeline_depth = max(1, depth)
        model.assume_inputs_ready = True
        for _ in range(max(args.warmup, 4 * max(1, depth))):        # each engine x 2 buffer sets: one eager call + one capture
            r.step_device()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        engines = model._engine_pool()
        l0 = sum(e.total_kernel_launches for e in engines)
        dev_blk = r.blocks(r.step_device, args.steps, n_blocks)
        launches = (sum(e.total_kernel_launches for e in engines) - l0) // n_blocks
        clock_info = clocks.finish() if rank == 0 else None
        outputs = snapshot_outputs(*r.last) if dump else None      # before the e2e steps overwrite the static outputs
        ws_bytes = sum(int(e.ws.numel()) for e in engines)
        for _ in range(4 * max(1, depth)):
            r.step_e2e()
        e2e_blk = r.blocks(r.step_e2e, args.steps, n_blocks)
        model.pipeline_depth = 1
        model.assume_inputs_ready = False
        # per-rank spread of the median block (host-side contention shows up here at 8 GPUs)
        spread = None
        if world > 1:
            import torch.distributed as dist
            mine = torch.tensor([dev_blk["own_median_ms"] / args.steps, e2e_blk["own_median_ms"] / args.steps], device=dev, dtype=torch.float64)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            spread = {"device_ms_per_step": [round(float(x[0]), 4) for x in allr], "e2e_ms_per_step": [round(float(x[1]), 4) for x in allr]}
        # ---- per-kernel-class device times (CUDA events on the launch stream), extra profiled steps
        prof = {}
        if rank == 0 and with_profile:
            n_prof = 3
            eng.profile(True)
            model.use_graph = False                 # per-kernel events need eager launches
            for _ in range(n_prof):
                flush.fill_(1)
                model(dict(r.dev_data))             # no collective here: the other ranks are already done
            model.use_graph = True
            raw = eng.profile_read()
            eng.profile(False)
            prof = {k: {"scopes_per_step": v[0] / n_prof, "ms_per_step": v[1] / n_prof} for k, v in raw.items()}
        out = dict(B=B, lat=lat, dev=dev_blk, e2e=e2e_blk, launches=int(launches), clocks=clock_info, ws_bytes=ws_bytes,
                   prof=prof, spread=spread, depth=max(1, depth), outputs=outputs)
        del r, model, eng, engines
        torch.cuda.empty_cache()
        return out

    depth = args.depth or (1 if args.workload == "c3" else 3)
    n_blocks = args.blocks or (5 if args.workload == "c3" else 9)
    m = measure(wl, depth, n_blocks, dump=bool(args.dump_outputs) and rank == 0)
    if m["outputs"] is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in m["outputs"].items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
    c2 = None
    if args.workload == "c3" and world == 1 and not args.no_c2:
        c2 = measure(WORKLOADS["c2"], 3, 9, with_profile=True)

    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    B, prof = m["B"], m["prof"]
    variant = wl[0]
    dev_s, e2e_s = stats(m["dev"], args.steps, world * B), stats(m["e2e"], args.steps, world * B)
    flops, nbytes, warp_inst = work_model(D=VIT_DIMS[variant][0], depth=VIT_DIMS[variant][1], n_pairs=B, it_matches=wl[1])
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)
    except Exception:      # noqa: BLE001
        traffic = {}
    sm_mhz = (m["clocks"] or {}).get("sm_mhz") or 1965.0
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count

    def group_ms(prefix):
        ks = [k for k in prof if k == prefix or (prefix.endswith("*") and k.startswith(prefix[:-1]))]
        return sum(prof[k]["ms_per_step"] for k in ks), sum(prof[k]["scopes_per_step"] for k in ks)

    def roof(cls):
        ms, n = group_ms(cls)
        if ms <= 0:
            return None
        base = {"kernel": cls, "launches_per_step": n, "avg_launch_ms": ms / max(n, 1), "peak_source": peaks["source"],
                "traffic": traffic.get(cls)}       # DRAM bytes per launch from the committed ncu --set full capture (or null)
        if cls in flops:
            ach = flops[cls] / (ms / 1e3) / 1e12
            return {**base, "bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"]}
        if cls in nbytes:
            ach = nbytes[cls] / (ms / 1e3) / 1e9
            return {**base, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"]}
        return None

    def attention_roof():
        """The tensor roofline object plus the bound that head_dim 64 really imposes: one MUFU.EX2 per logit at 16 per
        clock per SM (measured, tools/ubench/pipe_rates.cu) costs twice the tile's MMA time."""
        r = roof("vit.attention")
        if r is None:
            return None
        D_, depth_ = VIT_DIMS[variant]
        T_ = N_KP + 1
        exps = depth_ * 2 * B * (D_ // 64) * T_ * (-(-T_ // 128) * 128)           # padded key tiles are exponentiated too
        rate = exps / (prof["vit.attention"]["ms_per_step"] / 1e3) / (sm_mhz * 1e6) / n_sm
        r["mufu"] = {"achieved": rate, "peak": 16.0, "unit": "exp2/clk/SM", "frac": rate / 16.0,
                     "note": "head_dim 64: 1024 MUFU clk vs 512 tensor clk per 128x128 tile, so 16 exp2/clk/SM caps a kernel that sends "
                             "every exp2 to the MUFU at half of the tensor peak; this one evaluates a quarter of them on the FMA pipe"}
        return r

    def sampler_roof():
        """The outer sampler against the roof that binds it: instruction issue (one Philox4x32-7 call per cell and group
        of 8 streams), not HBM (final_scores is read once, mostly out of L2)."""
        ms, n = group_ms("solve.sample_outer")
        if ms <= 0:
            return None
        peak = n_sm * 4 * sm_mhz * 1e6 / 1e12                                       # warp instructions per second (4 schedulers per SM)
        ach = warp_inst["solve.sample_outer"] / (ms / 1e3) / 1e12
        hb = nbytes["solve.sample_outer"] / (ms / 1e3) / 1e9
        return {"kernel": "solve.sample_outer", "bound": "alu (instruction issue)", "achieved": ach, "peak": peak, "unit": "T warp-inst/s",
                "frac": ach / peak, "launches_per_step": n, "avg_launch_ms": ms / max(n, 1),
                "hbm_view": {"achieved": hb, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hb / peaks["hbm_gbs"]},
                "note": f"{COLLECT_INST_PER_CELL} thread instructions per cell and 8 streams in sampler_collect (ncu smsp__inst_executed); "
                        "histogram / threshold / select kernels are counted in the time but not in the instruction model"}

    known = [k for k in prof if k in flops or k in nbytes]
    dominant = max(known, key=lambda k: prof[k]["ms_per_step"]) if known else None
    vit_keys = ("vit.qkv", "vit.proj", "vit.fc1", "vit.fc2")
    vit_gemm_ms = sum(prof[k]["ms_per_step"] for k in vit_keys if k in prof)
    vit_gemm_fl = sum(flops[k] for k in vit_keys)
    tensor_ms = sum(prof[k]["ms_per_step"] for k in prof if k in flops)
    tensor_fl = sum(flops[k] for k in prof if k in flops)
    line = {
        "metric": "image-pairs/sec @720x540", "value": dev_s["value"], "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_s["ms_per_step"], "ms_per_step_min": dev_s["ms_per_step_min"],
        "ms_per_step_max": dev_s["ms_per_step_max"], "blocks": dev_s["blocks"],
        "latency_ms_single_step": m["lat"]["median_ms"] / args.steps,
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16 operands / f32 accumulate (tensor core), f32 matcher+solver", "data": "synthetic",
        "config": {"workload": wl[4] + (f"; {world} GPUs = BASELINE configs[3] (B={world * B} sharded {B} pairs per GPU, NCCL gather of poses)"
                                        if world > 1 and args.workload == "c3" else ""),
                   "pairs_per_gpu_per_step": B, "parallelism": f"dp{world} (pairs sharded, one all-gather of [B,13] poses)",
                   "timing": f"{dev_s['blocks']} blocks of {args.steps} steps, each between barrier+synchronize, CUDA events, max over ranks; "
                             "value / ms_per_step = median block",
                   "pipelining": f"{m['depth']} step(s) in flight (engines on alternating CUDA streams); latency_ms_single_step is the "
                                 "un-pipelined time of one step with the L2 flushed in between",
                   "l2": f"no flush between the steps of a block: each step streams its {m['ws_bytes'] // m['depth'] / 1e6:.0f} MB workspace + "
                         f"{B * 3 * N_KP * N_KP * 4 / 1e6:.0f} MB of N x N outputs + the weights, larger than the 126 MB L2; the latency run "
                         "flushes a 256 MiB buffer",
                   "weights": "seeded random init", "launch": "one mk_forward C call per step, replayed from a CUDA graph"},
        "e2e": {"value": e2e_s["value"], "unit": "pairs/s", "ms_per_step": e2e_s["ms_per_step"], "ms_per_step_min": e2e_s["ms_per_step_min"],
                "ms_per_step_max": e2e_s["ms_per_step_max"], "h2d_bytes_per_step": int(2 * B * 3 * H_IMG * W_IMG * 4) * world,
                "d2h_bytes_per_step": int(B * 13 * 4) * world, "api": "model(data) with pinned-host image0/image1; poses read back to the host"},
        "gpu_launches": int(m["launches"]),
        "clocks": m["clocks"],
        "roofline": (attention_roof() if dominant == "vit.attention" else roof(dominant)) if dominant else None,
        "roofline_step_tensor": ({"kernel": "every tensor-core kernel of the step", "bound": "tensor", "achieved": tensor_fl / (tensor_ms / 1e3) / 1e12,
                                  "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": tensor_fl / (tensor_ms / 1e3) / 1e12 / peaks["tflops"],
                                  "whole_step_frac": tensor_fl * dev_s["value"] / (world * B) / 1e12 / peaks["tflops"]} if tensor_ms > 0 else None),
        "roofline_vit_gemm": ({"kernel": "vit.qkv+proj+fc1+fc2", "bound": "tensor", "achieved": vit_gemm_fl / (vit_gemm_ms / 1e3) / 1e12,
                               "peak": peaks["tflops"], "unit": "TFLOP/s",
                               "frac": vit_gemm_fl / (vit_gemm_ms / 1e3) / 1e12 / peaks["tflops"], "traffic": None}
                              if vit_gemm_ms > 0 else None),
        "roofline_attention": attention_roof(), "roofline_head_conv": roof("head.conv3x3"),
        "roofline_matcher": roof("match.*"), "roofline_matcher_pass2": roof("match.dual_softmax"),
        "roofline_sampler": sampler_roof(), "roofline_solver": roof("solve.*"),
        "stage_ms": {k: round(v["ms_per_step"], 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms_per_step"])},
    }
    if m["spread"]:
        line["per_rank"] = m["spread"]
    if c2 is not None:
        d2, e2 = stats(c2["dev"], args.steps, c2["B"]), stats(c2["e2e"], args.steps, c2["B"])
        line["latency_c2"] = {"workload": WORKLOADS["c2"][4], "value": d2["value"], "unit": "pairs/s", "ms_per_step": d2["ms_per_step"],
                              "ms_per_step_min": d2["ms_per_step_min"], "ms_per_step_max": d2["ms_per_step_max"], "blocks": d2["blocks"],
                              "latency_ms_single_step": c2["lat"]["median_ms"] / args.steps, "steps_in_flight": c2["depth"],
                              "e2e": {"value": e2["value"], "ms_per_step": e2["ms_per_step"], "h2d_bytes_per_step": int(2 * 3 * H_IMG * W_IMG * 4),
                                      "d2h_bytes_per_step": 52}, "gpu_launches": c2["launches"],
                              "stage_ms": {k: round(v["ms_per_step"], 4) for k, v in sorted(c2["prof"].items(), key=lambda kv: -kv[1]["ms_per_step"])}}
    if world == 1 and not args.no_eager_baseline:
        line["gpu_eager_baseline"] = gpu_eager_run(wl, dev)
    if world == 1 and not args.no_cpu_baseline:
        cores = cpu_threads()
        durs = cpu_reference_run(wl, n_timed=3, n_warm=1, threads=cores, budget_s=25.0)
        line["cpu_baseline"] = {"value": len(durs) / sum(durs), "unit": "pairs/s", "cores": cores, "kind": "port",
                                "sample": f"{len(durs)} pair(s) (B=1) of the workload's model configuration ({variant}, {wl[1]}x{wl[2]} hypotheses) "
                                          f"after 1 warm-up ({sum(durs) / len(durs):.2f} s/pair), fp32 oracle, torch threads = {cores} of {usable_cpus()} usable"}
    print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
