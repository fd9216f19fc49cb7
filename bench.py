#!/usr/bin/env python
"""bench.py -- end-to-end frames/s of the depth -> stereo hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 1080p|4k] [--impl ours|reference]
                    [--no-4k] [--no-cpu-baseline] [--dof S] [--exact] [--dump-outputs DIR]

A step = one batch of `frames_per_step` synthetic frames through the hot path (DPT processor + Depth-Anything-V2
forward + u8 depth handoff in HBM + the DIBR frame loop of render_sbs_3d + pack).  With the defaults (20 steps of
15 frames) the timed region is the 300-frame clip of BASELINE.json configs[1].
`value`   : frames/s, inputs resident in HBM, CUDA events on the engine's stream, max over ranks.
`e2e`     : the same through the public host-buffer API (vd3d_render_clip_depth on pinned host frames, H2D and D2H
            inside the timed region).
`roofline`: the dominant kernel of the step -- the persistent tcgen05 GEMM (its fc1 launches timed live with CUDA
            events) against the measured bf16 peak; `roofline_depth_stage`, `roofline_dibr_stage` (whole DIBR frame,
            SURVEY 8(d) algorithmic bytes) and `roofline_dibr_render` (the fused warp/feather/compose/pack kernel)
            against the measured HBM peak explain the rest.  `dibr_only` is the DIBR stage run back to back on
            device-resident depth (its throughput form: bytes_per_frame x stage_fps).
`arm_4k`  : the same measurement on configs[2]'s per-GPU share (4K, DA-V2-Large, Full-SBS), emitted in the same run.
`cpu_baseline`: the oracle port of the reference path timed on a bounded sample on the host cores (rank 0, N=1).
`--impl reference`: that CPU port as the timed arm, same JSON line and the same `config`.
Multi-GPU: one process per GPU (torchrun), contiguous chunks of frames per rank, one NCCL broadcast of the weights,
no per-frame collective; max-over-ranks device time.  `--sharding exact` hands the temporal state from rank to
rank (bit-identical to one GPU); the default `replicas` keeps independent state per chunk.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# depth forward FLOPs per frame at 518x924 (SURVEY 8(d): linears + convs + 4*N^2*d*L attention)
DEPTH_GFLOP = {"vits": 253.8, "vitb": 775.3, "vitl": 2583.1}

WORKLOADS = {
    # BASELINE.json configs[1]: 300-frame clip = 20 steps x 15 frames
    "1080p": dict(name="1080p 300-frame synthetic clip, Depth-Anything-V2-Base, Half-SBS", w=1920, h=1080,
                  fmt="Half-SBS", preserve=False, model="vitb", pool=30, frames_per_step=15,
                  # SURVEY 8(d): 3*Ws*Hs + 1*Ws*Hs + 8*Wt*Ht + 3*Wout*Hout
                  dibr_bytes=3 * 1920 * 1080 + 1920 * 1080 + 8 * 960 * 540 + 3 * 1920 * 1080),
    # BASELINE.json configs[2] (per-GPU share of the 1000-frame clip)
    "4k": dict(name="4K synthetic clip, Depth-Anything-V2-Large, Full-SBS (per-GPU share of the 1000-frame clip)",
               w=3840, h=2160, fmt="Full-SBS", preserve=True, model="vitl", pool=12, frames_per_step=12,
               dibr_bytes=18 * 3840 * 2160),
}
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the fused render kernel from `ncu --set full`
# (profiles/r02_ncu_dibr.md); None until captured for that configuration
NCU_RENDER_TRAFFIC = {"4k": 115_862_272, "1080p": 49_949_440}
# smsp__issue_active.avg.pct_of_peak_sustained_active of the same launches: the DIBR kernels are issue bound, not HBM
# bound (DESIGN.md section 3.1), so this is the roofline fraction that describes them
NCU_RENDER_ISSUE_ACTIVE = {"4k": 70.6, "1080p": 62.9}
# same for one fc1 launch of k_umma_gemm<128,3> of a 4-frame forward (DA-V2-Base: M=10123, N=3072, K=768): 20.4 MB read +
# 11.7 MB written, cold L2 (profiles/r02_ncu_depth_final.md; algorithmic: 15.5 MB A + 4.7 MB W + 62.2 MB out, the output
# mostly stays in the 126 MB L2 for fc2)
NCU_GEMM_FC1_TRAFFIC = {"vitb": 32_100_000, "vitl": None, "vits": None}
COMMON = dict(fg=4.5, mg=-1.5, bg=-6.0, sharp=0.2, feather=10.0, ksize=9, tracking=True, floating=True,
              zps=0.01, dof=0.0)
# --dump-outputs: elements kept per workload arm, shared between ranks (16 MB of float32; the default run has two arms)
DUMP_ELEMS = 1 << 22


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1400.0, "fallback"


def peaks_burst():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("bf16_tflops", 1590.0)
    return 1590.0


def common_config(wl, world, sharding="replicas"):
    """The workload description: identical in the `ours` and the `reference` arm."""
    return {
        "workload": wl["name"], "resolution": [wl["w"], wl["h"]], "output_format": wl["fmt"],
        "depth_model": f"Depth-Anything-V2 {wl['model']} @518x924, random-init seed 0 (no checkpoints offline)",
        "frames_per_step": wl["frames_per_step"], "frame_pool": wl["pool"],
        "l2_policy": "inputs+outputs larger than L2 (pool of distinct frames cycled)",
        "params": dict(COMMON),
        "sharding": ("contiguous chunks per rank, temporal state handed from rank to rank (exact)" if sharding == "exact"
                     else "contiguous chunks per rank, independent temporal state per chunk (replicas)"),
    }


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, pw, reasons = [], None, [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


def make_pool(wl, n, seed0=0):
    """n (frame, depth) pairs of the noise (throughput) set, depth as 3-channel BGR like a decoded depth video."""
    from visiondepth3d_b200.synth import synth_frame
    return [synth_frame(seed0 + i, wl["w"], wl["h"], "noise") for i in range(n)]


def render_params(R, wl):
    return R.make_render_params(
        wl["w"], wl["h"], COMMON["fg"], COMMON["mg"], COMMON["bg"], COMMON["sharp"], wl["fmt"], 16 / 9,
        COMMON["dof"], COMMON["feather"], COMMON["ksize"], COMMON["tracking"], COMMON["floating"],
        preserve_original_aspect=wl["preserve"], zero_parallax_strength=COMMON["zps"])


def oracle_params(wl):
    from oracle import dibr as O
    return O.RenderParams(output_width=wl["w"], output_height=wl["h"], fg_shift=COMMON["fg"], mg_shift=COMMON["mg"],
                          bg_shift=COMMON["bg"], sharpness_factor=COMMON["sharp"], output_format=wl["fmt"],
                          dof_strength=COMMON["dof"], feather_strength=COMMON["feather"], blur_ksize=COMMON["ksize"],
                          use_subject_tracking=COMMON["tracking"], use_floating_window=COMMON["floating"],
                          preserve_original_aspect=wl["preserve"], zero_parallax_strength=COMMON["zps"])


# ======================================================================================================
# CPU arm: the port of the reference path (oracle/) on the host cores.  Depth forward = torch fp32 on all threads;
# the DIBR loop (numpy, one thread per clip) runs one independent chunk per worker process so that every core works.
# ======================================================================================================
_CPU_MODEL = {}


def _cpu_threads():
    return min(32, os.cpu_count() or 1)


def _dibr_workers():
    return max(1, min(8, (os.cpu_count() or 1) // 2))


def _dibr_chunk(job):
    """Worker: render one chunk with its own temporal state; returns (seconds for the timed frames, frames)."""
    wl, frames_idx, depths, common = job
    COMMON.update(common)   # spawned workers re-import this module: carry the parent's parameters over
    from oracle import dibr as O
    from visiondepth3d_b200.synth import synth_frame
    gs, cs, rp = O.GlobalState(), O.ClipState(), oracle_params(wl)
    t = 0.0
    for k, (i, d8) in enumerate(zip(frames_idx, depths)):
        fr, _ = synth_frame(i, wl["w"], wl["h"], "noise")
        t0 = time.perf_counter()
        O.render_frame(gs, cs, fr, np.repeat(d8[..., None], 3, axis=2), rp)
        if k > 0:  # the first frame of a chunk initialises the trackers (untimed warm-up)
            t += time.perf_counter() - t0
    return t, max(len(frames_idx) - 1, 0)


class CpuPort:
    def __init__(self, wl):
        import torch
        from visiondepth3d_b200.depth_weights import CONFIGS, hf_config
        self.wl, self.torch = wl, torch
        torch.set_num_threads(_cpu_threads())
        if wl["model"] not in _CPU_MODEL:
            from transformers import DepthAnythingForDepthEstimation
            torch.manual_seed(0)
            _CPU_MODEL[wl["model"]] = DepthAnythingForDepthEstimation(hf_config(wl["model"])).eval().state_dict()
        self.sd, self.cfg = _CPU_MODEL[wl["model"]], CONFIGS[wl["model"]]
        self.mean = torch.tensor([0.485, 0.456, 0.406]).view(3, 1, 1)
        self.std = torch.tensor([0.229, 0.224, 0.225]).view(3, 1, 1)
        self.i = 0
        self.pool = None

    def depth_u8(self, i):
        import torch.nn.functional as F
        from oracle import depth as OD
        from visiondepth3d_b200.synth import synth_frame
        torch, wl = self.torch, self.wl
        fr, _ = synth_frame(i, wl["w"], wl["h"], "noise")
        with torch.no_grad():
            t = torch.from_numpy(fr[..., ::-1].copy()).permute(2, 0, 1)[None].float()
            t = F.interpolate(t, size=(518, 924), mode="bicubic", align_corners=False, antialias=True).round().clamp(0, 255)
            pv = (t[0] / 255.0 - self.mean) / self.std
            d = OD.forward(self.sd, self.cfg, pv)
            d = F.interpolate(d[None, None], size=(wl["h"], wl["w"]), mode="bicubic", align_corners=False)[0, 0].numpy()
        return ((d - d.min()) / (d.max() - d.min() + np.float32(1e-6)) * 255).astype(np.uint8)

    def sample(self, frames_per_worker=1):
        """One bounded sample: W chunks of (1 warm-up + frames_per_worker) frames.  Returns (frames/s, frames)."""
        import multiprocessing as mp
        W = _dibr_workers()
        per = frames_per_worker + 1
        idx = [[self.i + c * per + k for k in range(per)] for c in range(W)]
        self.i += W * per
        t0 = time.perf_counter()
        depths = [[self.depth_u8(i) for i in ch] for ch in idx]
        t_depth = time.perf_counter() - t0
        n_depth = W * per
        if self.pool is None:
            # spawn, not fork: the parent may hold a CUDA context, OpenMP pools and helper threads (fork-unsafe)
            self.pool = mp.get_context("spawn").Pool(W)
        res = self.pool.map_async(_dibr_chunk, [(self.wl, ch, dp, dict(COMMON)) for ch, dp in zip(idx, depths)]).get(timeout=600)
        t_dibr = max(r[0] for r in res)          # chunks run concurrently: the slowest one is the stage time
        n = sum(r[1] for r in res)
        # per-frame cost = depth (all threads, one frame at a time) + DIBR (W chunks in parallel)
        sec_per_frame = t_depth / n_depth + t_dibr / max(n, 1)
        return 1.0 / sec_per_frame, n, {"depth_s_per_frame": t_depth / n_depth, "dibr_s_per_frame_effective": t_dibr / max(n, 1),
                                        "dibr_workers": W}

    def close(self):
        if self.pool is not None:
            self.pool.terminate()
            self.pool = None


def cpu_baseline_obj(wl):
    port = CpuPort(wl)
    try:
        fps, n, parts = port.sample(1)
    finally:
        port.close()
    return {"value": fps, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"{n} timed frames of the workload ({parts['dibr_workers']} independent chunks of 1 warm-up + 1 timed frame): "
                      f"depth forward oracle/depth.py torch fp32 on {_cpu_threads()} threads ({parts['depth_s_per_frame']:.2f} s/frame) + "
                      f"DIBR oracle/dibr.py numpy, one process per chunk ({parts['dibr_s_per_frame_effective']:.2f} s/frame effective); "
                      "the reference is Python and cannot travel to the GPU box"}


def run_reference(args, wl, rank, world):
    """--impl reference: the reference's CPU path (port: oracle/; /root/reference does not exist on the GPU box and
    its Python cannot travel).  Rank 0 only.  A step is a bounded sample of the workload."""
    if rank != 0:
        return
    t_all = time.perf_counter()
    port = CpuPort(wl)
    per_step, total, parts = [], 0, {}
    try:
        for s in range(args.warmup + args.steps):
            if time.perf_counter() - t_all > 200.0 and per_step:
                break
            if s >= args.warmup or s == 0:   # one warm-up sample is enough for a CPU path (lazy imports, page-in)
                fps, n, parts = port.sample(1)
                if s >= args.warmup:
                    per_step.append(fps)
                    total += n
    finally:
        port.close()
    value = float(np.mean(per_step))
    line = {
        "impl": "reference", "metric": "end-to-end frames/sec (depth+stereo)", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * wl["frames_per_step"] / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(wl, world, args.sharding),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
                         "sample": f"{len(per_step)} samples x {parts.get('dibr_workers', 0)} timed frames (each step a bounded sample of the "
                                   f"{wl['frames_per_step']}-frame step): depth forward torch fp32 on {_cpu_threads()} threads + DIBR numpy port, "
                                   f"{parts.get('dibr_workers', 0)} chunks in parallel processes"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "stage_seconds": parts, "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line), flush=True)


# ======================================================================================================
# GPU arm
# ======================================================================================================
class GpuArm:
    def __init__(self, args, key, rank, local_rank, world, dist):
        import torch
        wl = WORKLOADS[key]
        self.key = key
        from visiondepth3d_b200 import _lib
        from visiondepth3d_b200 import render_3d as R
        from visiondepth3d_b200.depth_engine import DepthEngine
        from visiondepth3d_b200.depth_weights import hf_config
        from visiondepth3d_b200.sharding import broadcast_state_dict
        from transformers import DepthAnythingForDepthEstimation
        self.args, self.wl, self.rank, self.world, self.dist, self.torch, self._lib = args, wl, rank, world, dist, torch, _lib
        self.dev = torch.device("cuda", local_rank)
        self.ctx = _lib.Context(local_rank)
        self.lib = self.ctx.lib
        if args.exact:
            self.ctx.set_exact(True)
        # depth model: the architecture BASELINE names, random-init (seed 0) -- no checkpoints offline.
        # One NCCL broadcast of the weights at init (rank 0 builds them), no per-frame collective.
        sd = None
        if rank == 0:
            torch.manual_seed(0)
            with torch.device("cpu"):
                sd = DepthAnythingForDepthEstimation(hf_config(wl["model"])).eval().state_dict()
        else:
            with torch.device("meta"):
                sd = DepthAnythingForDepthEstimation(hf_config(wl["model"])).state_dict()
        sd = broadcast_state_dict(sd, src=0, device=self.dev)
        from visiondepth3d_b200.depth_engine import processed_size
        ih, iw = processed_size(wl["w"], wl["h"])     # what the DPT processor picks for this frame shape (518 x 924)
        self.deng = DepthEngine(wl["model"], ih, iw, ctx=self.ctx)
        self.deng.load_state_dict(sd)
        del sd
        self.rp = render_params(R, wl)
        self.pl = R.plan_sizes(wl["w"], wl["h"], self.rp)
        self.oshape = R.output_shape(self.rp, self.pl)
        self.B, self.P = wl["frames_per_step"], wl["pool"]
        pool = make_pool(wl, self.P, seed0=rank * 1000)
        self.f_dev = [torch.from_numpy(f).to(self.dev) for f, _ in pool]
        self.d_dev = [torch.from_numpy(d).to(self.dev) for _, d in pool]      # synthetic depth (DIBR-only arm)
        self.o_dev = [torch.empty(self.oshape, dtype=torch.uint8, device=self.dev) for _ in range(self.P)]
        self.f_host = [torch.from_numpy(f).pin_memory() for f, _ in pool]
        self.o_host = [torch.empty(self.oshape, dtype=torch.uint8).pin_memory() for _ in range(self.P)]
        self.in_bytes = sum(t.numel() for t in self.f_dev) + sum(t.numel() for t in self.o_dev)
        torch.cuda.synchronize()
        self.stream = torch.cuda.ExternalStream(self.lib.vd3d_stream(self.ctx.h), device=self.dev)
        self.step_idx = 0

    def ptr_array(self, ts, idx):
        return (C.c_void_p * len(idx))(*[ts[i].data_ptr() for i in idx])

    def _idx(self):
        i0 = (self.step_idx * self.B) % self.P
        self.step_idx += 1
        return [(i0 + k) % self.P for k in range(self.B)]

    def step(self, mem):
        idx, wl, _lib = self._idx(), self.wl, self._lib
        self.last_idx = idx
        if mem == _lib.MEM_DEVICE:
            a, c = self.ptr_array(self.f_dev, idx), self.ptr_array(self.o_dev, idx)
        else:
            a, c = self.ptr_array(self.f_host, idx), self.ptr_array(self.o_host, idx)
        self.ctx.check(self.lib.vd3d_render_clip_depth(self.ctx.h, self.deng.h, self.B, a, wl["h"], wl["w"],
                                                       C.byref(self.rp), c, mem))

    def step_dibr(self):
        idx, wl, _lib = self._idx(), self.wl, self._lib
        a, d, c = self.ptr_array(self.f_dev, idx), self.ptr_array(self.d_dev, idx), self.ptr_array(self.o_dev, idx)
        self.ctx.check(self.lib.vd3d_render_clip(self.ctx.h, self.B, a, d, 3, wl["h"], wl["w"], C.byref(self.rp), c,
                                                 _lib.MEM_DEVICE, None))

    def step_dibr_host(self):
        idx, wl, _lib = self._idx(), self.wl, self._lib
        if not hasattr(self, "d_host"):
            self.d_host = [t.cpu().pin_memory() for t in self.d_dev]
        a, d, c = self.ptr_array(self.f_host, idx), self.ptr_array(self.d_host, idx), self.ptr_array(self.o_host, idx)
        self.ctx.check(self.lib.vd3d_render_clip(self.ctx.h, self.B, a, d, 3, wl["h"], wl["w"], C.byref(self.rp), c,
                                                 _lib.MEM_HOST, None))

    def python_surface(self, n_frames):
        """render_sbs_3d -- the call a user of the reference makes -- on an in-memory source and a counting sink
        (cv2.VideoCapture / the writer patched out, as tools/gen_golden.py does), so that the number is the drop-in's
        reader thread + pinned ring + batched vd3d_render_clip pipeline and not a codec's."""
        import cv2
        from visiondepth3d_b200 import render_3d as R
        wl = self.wl
        pool_f = [t.numpy() for t in self.f_host]
        pool_d = [t.cpu().numpy() for t in self.d_dev]
        P = len(pool_f)

        class Cap:
            def __init__(self, which):
                self.src, self.pos = (pool_f if which == "rgb" else pool_d), 0

            def isOpened(self):
                return True

            def get(self, prop):
                if prop == cv2.CAP_PROP_FRAME_COUNT:
                    return float(n_frames + 1)
                if prop == cv2.CAP_PROP_FPS:
                    return 24.0
                if prop == cv2.CAP_PROP_POS_FRAMES:
                    return float(self.pos)
                return 0.0

            def set(self, prop, v):
                if prop == cv2.CAP_PROP_POS_FRAMES:
                    self.pos = int(v)
                return True

            def read(self):
                if self.pos > n_frames:
                    return False, None
                self.pos += 1
                return True, self.src[self.pos % P]

            def release(self):
                pass

        class Sink:
            count = 0

            def __init__(self, *a, **k):
                pass

            def ok(self):
                return True

            def write(self, frame):
                Sink.count += 1

            def close(self):
                pass

        class Var:
            def get(self):
                return "Default (16:9)"

        real_cap, real_sink = cv2.VideoCapture, R._FrameSink
        cv2.VideoCapture, R._FrameSink = Cap, Sink
        R._lib._default_ctx[self.dev.index] = self.ctx
        try:
            def go():
                Sink.count = 0
                t0 = time.perf_counter()
                R.render_sbs_3d("rgb", "depth", "out.mp4", "mp4v", 24.0, wl["w"], wl["h"], COMMON["fg"], COMMON["mg"],
                                COMMON["bg"], COMMON["sharp"], wl["fmt"], Var(), R.aspect_ratios, COMMON["dof"],
                                feather_strength=COMMON["feather"], blur_ksize=COMMON["ksize"],
                                use_subject_tracking=COMMON["tracking"], use_floating_window=COMMON["floating"],
                                preserve_original_aspect=wl["preserve"], zero_parallax_strength=COMMON["zps"],
                                suspend_flag=threading.Event(), cancel_flag=threading.Event())
                return Sink.count / (time.perf_counter() - t0), Sink.count
            go()                       # warm-up (workspaces, graphs)
            fps, n = go()
        finally:
            cv2.VideoCapture, R._FrameSink = real_cap, real_sink
        return fps, n

    def dump_outputs(self, out_dir):
        """The packed output frames of the last step timed, as float32 `<workload>_frames.npy`: the flattened
        (frames_per_step, H, W, C) stack when it fits this rank's share n of DUMP_ELEMS, else the elements at the
        sorted unique draws of numpy default_rng(0).integers(0, size, n)."""
        out = self.torch.stack([self.o_dev[i] for i in self.last_idx]).flatten()
        n = DUMP_ELEMS // self.world
        if out.numel() > n:
            pick = np.unique(np.random.default_rng(0).integers(0, out.numel(), n))
            out = out[self.torch.from_numpy(pick).to(self.dev)]
        name = f"{self.key}_frames" + (f"_rank{self.rank}" if self.world > 1 else "")
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, name + ".npy"), out.float().cpu().numpy())

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce_max(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup):
        torch = self.torch
        self.ctx.reset()
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        self.barrier()
        wall = self.reduce_max(time.perf_counter() - t0)
        return self.reduce_max(e0.elapsed_time(e1)), wall

    def measure(self, local_rank, full=True):
        args, wl, _lib, lib, ctx, deng = self.args, self.wl, self._lib, self.lib, self.ctx, self.deng
        B, world = self.B, self.world
        frames = args.steps * B
        # ---------------- device-resident arm (value) ----------------
        clocks = ClockSampler(local_rank)
        clocks.start()
        l0 = ctx.launches + deng.launches
        ms, _ = self.timed(lambda: self.step(_lib.MEM_DEVICE), args.steps, args.warmup)
        launches = ctx.launches + deng.launches - l0 - 0
        value = world * frames / (ms / 1000.0)
        if args.dump_outputs:  # before the arms below reuse the output buffers
            self.dump_outputs(args.dump_outputs)
        # ---------------- end-to-end arm (pinned host buffers through the public API) ----------------
        _, e2e_s = self.timed(lambda: self.step(_lib.MEM_HOST), args.steps, args.warmup)
        clk = clocks.stop()
        e2e_value = world * frames / e2e_s
        h2d = B * (wl["w"] * wl["h"] * 3)
        d2h = B * int(np.prod(self.oshape))
        # ---------------- DIBR stage alone, back to back on device-resident u8 depth (graph replay) ----------------
        dsteps = max(4, min(args.steps, 10))
        dms, _ = self.timed(self.step_dibr, dsteps, 3)
        dibr_fps = dsteps * B / (dms / 1000.0)          # per GPU
        # ---------------- DIBR stage through host buffers, and through the Python drop-in surface (rank 0, N = 1) -----
        py_fps = py_n = dibr_host_fps = None
        if world == 1:
            _, hs = self.timed(self.step_dibr_host, dsteps, 3)
            dibr_host_fps = dsteps * B / hs
            try:
                py_fps, py_n = self.python_surface(max(300, dsteps * B))   # long enough to amortise the pinned-ring set-up
            except Exception as e:  # informational arm: never take the bench line down
                py_fps, py_n = None, str(e)
        # ---------------- per-stage device timing (CUDA events around the stages; serial eager launches) ----------
        lib.vd3d_profile(ctx.h, 1)
        lib.vd3d_depth_profile(deng.h, 1)
        tot = [C.c_double() for _ in range(3)]
        cnt = [C.c_int() for _ in range(3)]
        g_ms, g_n, g_gf = C.c_double(), C.c_int(), C.c_double()
        self.step(_lib.MEM_DEVICE)  # un-timed: first eager pass through the serial path allocates its workspaces
        for st in (0, 1, 2):
            lib.vd3d_profile_collect(ctx.h, st, C.byref(tot[st]), C.byref(cnt[st]))
        lib.vd3d_depth_profile_collect(deng.h, C.byref(g_ms), C.byref(g_n), C.byref(g_gf))
        for _ in range(2):
            self.step(_lib.MEM_DEVICE)
        for st in (0, 1, 2):
            lib.vd3d_profile_collect(ctx.h, st, C.byref(tot[st]), C.byref(cnt[st]))
        lib.vd3d_depth_profile_collect(deng.h, C.byref(g_ms), C.byref(g_n), C.byref(g_gf))
        lib.vd3d_depth_profile(deng.h, 0)
        lib.vd3d_profile(ctx.h, 0)
        if self.rank != 0:
            return None
        hbm_peak, tf_peak, which = peaks()
        pl = self.pl
        # fused render kernel: source RGB in (u8 at the source size on the identity path, f32 RGBx otherwise is an
        # intermediate -- algorithmic = the u8 frame) + packed output out
        src_px = wl["w"] * wl["h"]
        out_px = int(np.prod(self.oshape[:2]))
        rend_bytes = 3 * src_px + 3 * out_px
        rend_ms = tot[1].value / max(cnt[1].value, 1)
        stage_ms = tot[0].value / max(cnt[0].value, 1)
        rend_gbs = rend_bytes / (rend_ms * 1e-3) / 1e9 if rend_ms > 0 else 0.0
        stage_gbs = wl["dibr_bytes"] / (stage_ms * 1e-3) / 1e9 if stage_ms > 0 else 0.0
        tput_gbs = wl["dibr_bytes"] * dibr_fps / 1e9
        depth_ms = tot[2].value / max(cnt[2].value, 1)
        depth_tf = DEPTH_GFLOP[wl["model"]] / max(depth_ms, 1e-9)
        gemm_ms = g_ms.value / max(g_n.value, 1)
        gemm_tf = g_gf.value / max(gemm_ms, 1e-9)
        tf_burst = peaks_burst()
        cfg = common_config(wl, world, args.sharding)
        line = {
            "metric": "end-to-end frames/sec (depth+stereo)", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 GEMM operands, fp32 accumulate; DIBR fp32", "data": "synthetic",
            "config": cfg,
            "run": {
                "timed_frames": frames, "timed_region_s": ms / 1000.0,
                "pool_mb": self.in_bytes / 1e6,
                "stage": "DPT processor + depth forward + min-max u8 handoff in HBM + DIBR frame loop + pack",
                "launch_mode": "CUDA graph replay; one batched depth forward per group of depth_batch frames on two "
                               "alternating engine instances / streams, DIBR frame by frame behind it "
                               "(stage timings in roofline* are taken in a separate serial, eager pass)",
                "dibr_mode": "exact" if args.exact else "fast",
                "graphs_active": int(lib.vd3d_graphs_active(ctx.h)),
                "depth_batch": int(lib.vd3d_get_depth_batch(ctx.h)),
            },
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "k_umma_gemm<128,3> (fc1 launches)",
                         "achieved": gemm_tf, "peak": tf_burst, "unit": "TFLOP/s", "frac": gemm_tf / tf_burst,
                         "traffic": NCU_GEMM_FC1_TRAFFIC.get(wl["model"]),
                         "peak_source": which + " (cuBLAS bf16 burst: kernel timed alone)",
                         "algorithmic_gflop_per_launch": g_gf.value, "avg_launch_ms": gemm_ms, "launches_timed": g_n.value},
            "roofline_depth_stage": {"bound": "tensor", "achieved": depth_tf, "peak": tf_peak, "unit": "TFLOP/s",
                                     "frac": depth_tf / tf_peak, "peak_source": which + " (cuBLAS bf16 sustained)",
                                     "algorithmic_gflop_per_frame": DEPTH_GFLOP[wl["model"]], "avg_frame_ms": depth_ms,
                                     "share_of_step": depth_ms / max(depth_ms + stage_ms, 1e-9),
                                     "achieved_in_timed_region": DEPTH_GFLOP[wl["model"]] * (value / world) / 1000.0},
            "roofline_dibr_render": {"bound": "hbm", "kernel": "k_render (warp edges + box feather + compose + sharpen + fit + pack)",
                                     "achieved": rend_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": rend_gbs / hbm_peak,
                                     "traffic": NCU_RENDER_TRAFFIC.get(self.key),
                                     "issue_active_pct": NCU_RENDER_ISSUE_ACTIVE.get(self.key),
                                     "note": "instruction-issue bound (~1000 thread-instructions per eye pixel against a machine "
                                             "balance of 5.5 instructions per byte): frac vs HBM is not the binding roofline",
                                     "peak_source": which, "algorithmic_bytes_per_launch": rend_bytes, "avg_launch_ms": rend_ms},
            "roofline_dibr_stage": {"bound": "hbm", "what": "whole DIBR frame (ingest..pack), serial eager launches",
                                    "achieved": stage_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": stage_gbs / hbm_peak,
                                    "algorithmic_bytes_per_frame": wl["dibr_bytes"], "avg_frame_ms": stage_ms},
            "dibr_only": {"what": "DIBR stage back to back on device-resident u8 depth (vd3d_render_clip, graph replay)",
                          "frames_per_s_per_gpu": dibr_fps, "achieved": tput_gbs, "peak": hbm_peak, "unit": "GB/s",
                          "frac": tput_gbs / hbm_peak, "ms_per_frame": 1000.0 / dibr_fps},
            "python_surface": {"what": "render_sbs_3d (drop-in call surface: reader thread -> pinned ring -> batched "
                                       "vd3d_render_clip -> writer thread) on an in-memory source / counting sink, given depth "
                                       "frames (no depth engine on this path), against the same stage through the C ABI on "
                                       "pinned host buffers", "frames_per_s": py_fps, "frames": py_n,
                               "c_abi_host_buffers_frames_per_s": dibr_host_fps,
                               "ratio": (py_fps / dibr_host_fps) if (py_fps and dibr_host_fps) else None},
        }
        return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="1080p", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-4k", action="store_true", help="skip the 4K / DA-V2-Large / Full-SBS arm of the default run")
    ap.add_argument("--exact", action="store_true", help="DIBR in the bit-exact one-kernel-per-op mode")
    ap.add_argument("--sharding", default="replicas", choices=["replicas", "exact"])
    ap.add_argument("--dof", type=float, default=None,
                    help="dof_strength (default 0 = the warp/fill/compose variant; 2.0 = the reference GUI default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the output frames of the last one (a fixed sample when large) "
                         "to DIR/<workload>_frames.npy as float32, for comparing two builds on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.sharding == "exact"):
        ap.error("--dump-outputs covers the default GPU arm (--impl ours --sharding replicas)")
    if args.dof is not None:
        COMMON["dof"] = args.dof
    args.warmup = max(args.warmup, 3)
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libvd3d has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.sharding == "exact":
        from visiondepth3d_b200 import sharding_bench
        sharding_bench.run(args, wl, rank, local_rank, world, dist, common_config)
        if world > 1:
            dist.destroy_process_group()
        return
    arm = GpuArm(args, args.workload, rank, local_rank, world, dist)
    line = arm.measure(local_rank)
    del arm
    torch.cuda.empty_cache()
    if args.workload == "1080p" and not args.no_4k:
        a4 = GpuArm(args, "4k", rank, local_rank, world, dist)
        l4 = a4.measure(local_rank)
        del a4
        if rank == 0:
            keep = ("value", "unit", "ms_per_step", "config", "run", "clocks", "e2e", "gpu_launches", "roofline",
                    "roofline_depth_stage", "roofline_dibr_render", "roofline_dibr_stage", "dibr_only", "python_surface")
            line["arm_4k"] = {k: l4[k] for k in keep}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_obj(wl)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
