"""bench.py -- headline benchmark of the MOFA-Video hot path on B200; prints one JSON result line.

    python bench.py --gpus N --steps K --warmup W            # engine arm (this repo's sm_100a path)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle restatement of the reference
    python bench.py ... --dump-outputs DIR                    # also save what the last timed clip computed

--dump-outputs writes DIR/frames.npy: a fixed, seeded sample (float32) of the uint8 frames of the last timed clip, whose
inputs and initial noise are seeded, so two builds run with the same arguments can be compared output for output.  Compare
with a tolerance: two runs of one build on a B200 differed by 1 (of 255) in 5 % of the sampled values.

Metric (BASELINE.json): frames/sec @ 576x1024x25f, 25 Euler steps.  One "step" of this benchmark is ONE CLIP
through FlowControlNetPipeline.__call__ (CLIP embed + VAE encode + adapter cond branch + 25 x (adapter + UNet +
CFG + Euler) + VAE decode) = configs[1] of BASELINE.json.  Synthetic image / flow, random-init weights in the
reference checkpoint layout (no network here).
  value : device-resident inputs (image, flow, initial noise already in HBM), frames left on the device.
  e2e   : the reference-facing call with HOST inputs (PIL image, host flow tensor) and uint8 frames copied back
          to the host; for N>1 the frames of all ranks are gathered to rank 0 with NCCL inside the timed region.
  roofline : dominant kernel family (tcgen05 GEMM / implicit-GEMM conv), CUDA-event timed per launch on the
          launching stream during the last timed clip; algorithmic FLOPs = 2*M*N*K of each launch.
  cpu_baseline : the fp32 oracle on the host cores, bounded sample (see _cpu_sample).
Multi-GPU: independent clips per rank (weak scaling), no collective on the data path except the final gather.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, T, STEPS = 576, 1024, 25, 25
METRIC = "frames/sec @ 576x1024x25f, 25 steps"


def _peaks():
    fn = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(fn):
        with open(fn) as f:
            p = json.load(f)
        return {"tflops_burst": p["bf16_tflops"], "tflops_sustained": p["bf16_tflops_sustained"],
                "hbm_gbs": p["hbm_gbs"], "src": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = max([int(float(r[2])) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle): bounded sample of the same workload, ALWAYS at 576x1024
# ------------------------------------------------------------------------------------------------
WORKLOAD = "configs[1]: Traj adapter 576x1024, 25 frames, 25 steps, fp16 on 1xB200 (CFG 1->3)"


def shared_config(world):
    """The `config` object of BOTH arms (the driver compares them): what is measured, not how."""
    return {"workload": WORKLOAD, "step": "one clip through FlowControlNetPipeline.__call__",
            "height": H, "width": W, "num_frames": T, "num_inference_steps": STEPS, "clips_per_gpu_per_step": 1,
            "parallelism": f"clip-parallel x{world}",
            "l2": "working set >> L2 (each level-0 activation is 295 MB; weights 4.4 GB)"}


class CpuSampler:
    """The reference's PyTorch-CPU path for this workload = the fp32 oracle (the reference itself cannot execute here:
    SURVEY.md 8c).  One SAMPLE = one denoise step (adapter cond branch + trunk + UNet, fp32) at the FULL 576x1024
    spatial size on 2 of the 50 CFG-batched frames of a step (one CFG half, 2 frames: batch items and frames are
    processed independently except for the T-wide temporal layers); clip time = sample x25 (frames) x25 (steps),
    VAE / CLIP excluded (3 % of a clip).  The spatial shape is never reduced, so every run measures the same thing."""

    FRAMES = 2

    def __init__(self):
        from oracle.models import FlowControlNet, UNetSpatioTemporalConditionControlNetModel
        self.host_cores = os.cpu_count() or 1
        # 32 threads: on the 128-core GPU box the fp32 oracle got slower with 128 (contended host, round-1 measurement);
        # tune() may raise this to 64 when that is measurably faster
        self.threads = min(self.host_cores, 32)
        torch.set_num_threads(self.threads)
        cfg = dict(num_frames=self.FRAMES)
        with torch.device("meta"):
            unet = UNetSpatioTemporalConditionControlNetModel(**cfg)
            adapter = FlowControlNet(**cfg)
        for m in (unet, adapter):
            m.to_empty(device="cpu")
            with torch.no_grad():
                for n_, p in m.named_parameters():
                    if p.ndim > 1:
                        p.normal_(0.0, 0.02)
                    elif n_.endswith("weight"):
                        p.fill_(1.0)
                    else:
                        p.zero_()
            m.eval()
        g = torch.Generator().manual_seed(0)
        Tm = self.FRAMES
        self.unet, self.adapter = unet, adapter
        self.emb = torch.randn(1, 1, 1024, generator=g)
        self.ids = torch.tensor([[6.0, 128.0, 0.02]])
        self.t = torch.tensor(1.6377)
        self.sample = torch.randn(1, Tm, 8, H // 8, W // 8, generator=g)
        self.cond = torch.rand(1, 3, H, W, generator=g) * 2 - 1
        self.flow = torch.randn(1, Tm - 1, 2, H, W, generator=g)

    def one(self):
        t0 = time.perf_counter()
        with torch.no_grad():
            dres, mid, _, _ = self.adapter(self.sample, self.t, self.emb, self.ids, controlnet_cond=self.cond,
                                           controlnet_flow=self.flow)
            out = self.unet(self.sample, self.t, self.emb, dres, mid, added_time_ids=self.ids)[0]
        assert out.shape == (1, self.FRAMES, 4, H // 8, W // 8)
        return time.perf_counter() - t0

    def tune(self, first_s):
        """Second warm-up sample with 64 threads when the host has them; keep whichever was faster."""
        if self.host_cores < 64:
            return self.one()
        torch.set_num_threads(64)
        dt = self.one()
        if dt < 0.9 * first_s:
            self.threads = 64
        else:
            torch.set_num_threads(self.threads)
        return dt

    def fps(self, sample_s):
        return T / (sample_s * (2 * T / self.FRAMES) * STEPS)

    def describe(self):
        return (f"1 denoise step (oracle adapter + UNet, fp32, {self.threads} threads of {self.host_cores} host cores) at "
                f"{H}x{W} on {self.FRAMES} of {2 * T} frames; clip time = sample x{2 * T // self.FRAMES} (frames) "
                f"x{STEPS} (steps); VAE/CLIP excluded")


def _cpu_sample(steps, warmup):
    """-> (frames/s, seconds per sample, threads, host cores, description): `warmup` untimed + `steps` timed samples."""
    cs = CpuSampler()
    first = cs.one() if warmup >= 1 else None
    if warmup >= 2:
        cs.tune(first)
    for _ in range(max(warmup - 2, 0)):
        cs.one()
    dts = [cs.one() for _ in range(steps)]
    dt = sum(dts) / len(dts)
    return cs.fps(dt), dt, cs.threads, cs.host_cores, cs.describe()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K = max(args.steps, 1)
    W_ = min(max(args.warmup, 1), 2)   # each warm-up is a 10 s CPU sample: 2 (the second picks the thread count)
    fps, dt, threads, host, desc = _cpu_sample(K, W_)
    out = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
           "steps": K, "warmup": args.warmup, "warmup_samples_run": W_, "ms_per_step": dt * 1e3,
           "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
           "config": shared_config(max(args.gpus, 1)),
           "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "host_cores": host, "kind": "port",
                            "sample": desc},
           "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
# engine arm
# ------------------------------------------------------------------------------------------------
def _pin_to_gpu_numa_node(gpu_index):
    """Keep this rank's host threads on the CPUs of its GPU's NUMA node (NVML's ideal affinity): with 8 ranks on one host
    the enqueue threads otherwise migrate across sockets (round-1 SCALE: per-clip time grew 2.5 % from N=1 to N=8)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, wd in enumerate(mask) for b in range(64) if (wd >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:  # noqa: BLE001  (no NVML / restricted container: run unpinned)
        return None



DUMP_SAMPLES = 1 << 23   # 32 MiB of float32; one 576x1024x25 clip is 44 M values (177 MB in float32)


def _frames_sample(frames):
    """A fixed, seeded sample of a clip's uint8 frames [T, H, W, 3] as float32: the same flat indices on every run."""
    flat = frames.reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLES].sort().values
    return flat[idx.to(flat.device)].float().cpu().numpy()


def _write_dump(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_engine(args):
    import torch.distributed as dist
    from mofa_video_b200 import lib, parallel
    from mofa_video_b200.factory import build_synthetic_pipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()
    affinity = _pin_to_gpu_numa_node(local)
    torch.set_num_threads(min(8, os.cpu_count() or 1))  # host work of this arm is tiny; 128 OpenMP threads on a busy
                                                        # host made it 10x slower (round-1 observation)

    # per-rank clip (independent clips, seeds 1234+rank / 1235+rank -- SURVEY.md §8d config 5)
    import numpy as np
    import PIL.Image
    g = torch.Generator().manual_seed(1234 + rank)
    img = torch.nn.functional.avg_pool2d(torch.rand(1, 3, H + 8, W + 8, generator=g), 9, stride=1)[0]
    img = (img - img.min()) / (img.max() - img.min())
    img_u8 = (img * 255).round().to(torch.uint8).permute(1, 2, 0).contiguous().numpy()
    pil = PIL.Image.fromarray(img_u8)
    g2 = torch.Generator().manual_seed(1235 + rank)
    ys = torch.arange(H, dtype=torch.float32)[:, None] / H
    xs = torch.arange(W, dtype=torch.float32)[None, :] / W
    base = torch.stack([(torch.sin(6.2832 * ys) * torch.cos(6.2832 * xs)).expand(H, W),
                        (torch.cos(6.2832 * ys) * torch.sin(6.2832 * xs)).expand(H, W)], 0) * (0.06 * H)
    flow_host = torch.stack([(i + 1) / (T - 1) * base + torch.randn(2, H, W, generator=g2) for i in range(T - 1)])[None]
    flow_host = flow_host.half().pin_memory()

    pipe = build_synthetic_pipeline(device=dev, seed=0)
    img_dev = (torch.from_numpy(img_u8).permute(2, 0, 1).float() / 255.0).to(dev)  # [3,H,W] in [0,1]
    flow_dev = flow_host.to(dev)
    lat_gen = torch.Generator(device=dev).manual_seed(42 + rank)

    def clip_device():
        return pipe(img_dev, img_dev, flow_dev, height=H, width=W, num_frames=T, num_inference_steps=STEPS,
                    decode_chunk_size=8, generator=lat_gen, output_type="uint8_pt")

    host_out = torch.empty(world if rank == 0 else 1, T, H, W, 3, dtype=torch.uint8).pin_memory()
    # N > 1: the decoder's uint8 epilogue stores straight into rank 0's gather buffer over NVLink (parallel.PeerFrameGather,
    # SURVEY 8f-3); if peer mapping is unavailable on this box the portable NCCL gather is used and the line says so
    gather, gather_kind = None, "none (1 GPU)"
    if world > 1:
        try:
            gather = parallel.PeerFrameGather((T, H, W, 3))
            gather_kind = "decoder epilogue -> NVLink peer stores into rank 0 (no NCCL on the data path)"
        except Exception as exc:  # noqa: BLE001
            gather_kind = f"nccl gather (peer mapping unavailable: {type(exc).__name__}: {exc})"[:200]
        flags = [gather is not None]
        allf = [None] * world
        dist.all_gather_object(allf, flags[0])
        if not all(allf):
            gather = None

    host_gen = torch.Generator().manual_seed(42 + rank)   # PIL inputs: the noise is drawn on the CPU (pipeline.py:339-341)

    def clip_e2e():
        out = pipe(pil, pil, flow_host, height=H, width=W, num_frames=T, num_inference_steps=STEPS,
                   decode_chunk_size=8, generator=host_gen, output_type="uint8_pt")
        u8 = out.frames[0]  # uint8 [T, H, W, 3] (post-processing fused in the decoder tail); with the peer gather this
                            # IS slot `rank` of rank 0's buffer, already written over NVLink by the tail kernel
        if gather is not None:
            gather.publish()
            if rank == 0:
                host_out.copy_(gather.collect(), non_blocking=True)
                gather.release()
        else:
            bufs = parallel.gather_frames(u8, dst=0)  # portable form: one NCCL gather; identity at N=1
            if rank == 0:
                for r, b in enumerate(bufs):
                    host_out[r].copy_(b, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        sync_all()
        return float(ms.item())

    for _ in range(max(args.warmup, 0)):
        clip_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.launch_count_reset()
    K = args.steps
    if K > 1:
        ms_dev = timed(clip_device, K - 1)
    else:
        ms_dev = 0.0
    # last timed clip: per-launch CUDA events for the roofline line.  Its initial noise is re-seeded so that the frames
    # --dump-outputs writes depend only on the seeds, not on how many clips --warmup / --steps ran before it.
    lib.profile_start()
    lat_gen.manual_seed(42 + rank)
    last = []
    ms_last = timed(lambda: last.append(clip_device()), 1)
    prof = lib.profile_stop()
    tim = pipe.last_timings_ms()
    ms_dev += ms_last
    launches = lib.launch_count()
    # sampled now: later clips may reuse the pipeline's output buffer
    dump = {"frames": _frames_sample(last[0].frames[0])} if args.dump_outputs and rank == 0 else None
    del last
    if world > 1 and gather is None:  # NCCL communicator / buffers are created at the first collective: not timed
        parallel.gather_frames(torch.zeros(T, H, W, 3, dtype=torch.uint8, device=dev), dst=0)
        torch.cuda.synchronize()
    pipe.frame_sink = gather
    clip_e2e()                      # one untimed e2e clip (first use of the host-input path and of the gather)
    ms_e2e = timed(clip_e2e, K)
    pipe.frame_sink = None
    if gather is not None:
        gather.check()
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        peaks = _peaks()
        fps = world * K * T / (ms_dev / 1e3)
        fps_e2e = world * K * T / (ms_e2e / 1e3)
        gem = {k: v for k, v in prof.items() if k.startswith("gemm_")}
        g_ms = sum(v["ms"] for v in gem.values())
        g_fl = sum(v["work"] for v in gem.values())
        g_n = sum(v["launches"] for v in gem.values())
        ach = g_fl / (g_ms * 1e-3) / 1e12 if g_ms else 0.0
        traffic = None
        for name in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):   # ncu capture of this kernel family (newest first)
            tf = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tf):
                with open(tf) as f:
                    traffic = json.load(f).get("dram_bytes_per_launch")
                break
        att = prof.get("attn_spatial", {"ms": 0.0, "work": 0.0, "launches": 0})
        roof = {"bound": "tensor", "kernel": "gemm_tc_kernel (linear / conv3x3 / temporal3 implicit GEMM)",
                "achieved": round(ach, 1), "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                "frac": round(ach / peaks["tflops_sustained"], 4), "traffic": traffic,
                "peak_source": peaks["src"] + " bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_timed": g_n, "avg_launch_ms": round(g_ms / max(g_n, 1), 4),
                "flops_per_launch_avg": g_fl / max(g_n, 1),
                "share_of_clip": round(g_ms / ms_last, 4),
                "by_kind": {k: {"ms": round(v["ms"], 2), "tflops": round(v["work"] / (v["ms"] * 1e-3) / 1e12, 1),
                                "launches": v["launches"]} for k, v in prof.items()},
                "attention": {"achieved": round(att["work"] / max(att["ms"], 1e-9) / 1e9, 1), "unit": "TFLOP/s",
                              "share_of_clip": round(att["ms"] / ms_last, 4)}}
        other = None
        if world == 1 and not args.no_other_configs:
            del pipe
            other = _other_configs(dev, peaks)
        cpu = None
        if not args.no_cpu_baseline:
            cfps, cdt, threads, host, desc = _cpu_sample(1, 1)
            cpu = {"value": cfps, "unit": "frames/s", "cores": threads, "host_cores": host, "kind": "port",
                   "sample": desc, "seconds_per_sample": round(cdt, 2)}
        h2d = img_u8.nbytes * 2 + flow_host.numel() * 2
        d2h = world * T * H * W * 3
        out = {"metric": METRIC, "value": round(fps, 4), "unit": "frames/s", "n_gpus": world, "steps": K,
               "warmup": args.warmup, "ms_per_step": round(ms_dev / K, 2), "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
               "config": shared_config(world),
               "engine": {"vae_clip": "VAE encode / decode and the CLIP ViT-H image encoder all run on the sm_100a kernels "
                                      "(pipelines re-host the caller's modules: vae_engine / clip_engine); VAE encode "
                                      "keeps fp16 storage where the reference upcasts to fp32 (max 2.6e-3 of max|ref| at "
                                      "576x1024, tests/test_fullsize_parity_gpu.py)",
                          "phase_ms_last_clip": {k: round(v, 1) for k, v in tim.items()}},
               "roofline": roof, "cpu_baseline": cpu, "other_configs": other,
               "e2e": {"value": round(fps_e2e, 4), "unit": "frames/s", "h2d_bytes_per_step": int(h2d),
                       "d2h_bytes_per_step": int(d2h), "ms_per_step": round(ms_e2e / K, 2)},
               "gather": gather_kind, "host": {"cpus_pinned_to_gpu_numa_node": affinity, "cuda_graph_step": True},
               "gpu_launches": int(launches), "clocks": clocks}
        if dump is not None:
            _write_dump(args.dump_outputs, dump)
        print(json.dumps(out), flush=True)
    if world > 1:
        if gather is not None:
            try:
                gather.close()
            except Exception:  # noqa: BLE001  (shutdown only: the line is already printed)
                pass
        dist.destroy_process_group()


def _other_configs(dev, peaks):
    """BASELINE.json configs[2] (Keypoint 512x512x25f) and configs[3] (Hybrid 576x1024x25f), 25 steps, one B200: one timed
    clip each through their reference-facing pipelines (device-resident inputs, uint8 frames left on the device), after a
    2-step warm-up clip.  Algorithmic FLOPs per clip from BASELINE.md section 2 (de-duplicated Keypoint views; hoisted
    occlusion nets): the rate is whole-clip FLOPs / clip time, against the measured sustained tensor peak."""
    from mofa_video_b200.factory import build_synthetic_pipeline
    out = {}
    specs = (("configs[2]: Keypoint adapter 512x512, 25 frames, 25 steps", "keypoint", 512, 512, 2.07e15 + 0.076e15),
             ("configs[3]: Hybrid dual-adapter 576x1024, 25 frames, 25 steps", "hybrid", 576, 1024,
              25 * 266.3e12 + 6.4e12 + 0.174e15))
    for name, variant, hh, ww, flops in specs:
        torch.cuda.empty_cache()
        pipe = build_synthetic_pipeline(device=dev, seed=0, variant=variant)
        g = torch.Generator().manual_seed(7)
        image = torch.rand(3, hh, ww, generator=g).to(dev)
        flow = (torch.randn(1, T - 1, 2, hh, ww, generator=g) * 8).half().to(dev)
        ldmk = torch.rand(1, T, 3, hh, ww, generator=g).half().to(dev)
        gen = torch.Generator(device=dev).manual_seed(3)
        kw = dict(height=hh, width=ww, num_frames=T, decode_chunk_size=8, generator=gen, output_type="uint8_pt")
        if variant == "keypoint":
            call = lambda steps: pipe(image, image, flow, ldmk, num_inference_steps=steps, **kw)  # noqa: E731
        else:
            mask = torch.zeros(1, 1, hh, ww)
            yy, xx = torch.meshgrid(torch.arange(hh), torch.arange(ww), indexing="ij")
            mask[0, 0] = (((yy - hh / 2) ** 2 + (xx - ww / 2) ** 2) < (0.25 * min(hh, ww)) ** 2).float()
            call = lambda steps: pipe(image, image, flow, ldmk, flow * 0.5, mask.to(dev),  # noqa: E731
                                      num_inference_steps=steps, **kw)
        call(2)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        frames = call(STEPS).frames[0]
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        tf = flops / (ms * 1e-3) / 1e12
        out[name] = {"frames_per_s": round(T / (ms * 1e-3), 4), "ms_per_clip": round(ms, 1),
                     "algorithmic_pflop_per_clip": round(flops / 1e15, 3), "achieved_tflops": round(tf, 1),
                     "frac_of_sustained_tensor_peak": round(tf / peaks["tflops_sustained"], 4),
                     "frames_shape": list(frames.shape), "inputs": "device-resident", "clips_timed": 1}
        del pipe, call
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of the last timed clip's frames to DIR/frames.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs applies to the engine arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
