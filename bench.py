#!/usr/bin/env python
"""bench.py -- 4-agent OPV2V-H-shape GenComm frames/s, raw points -> NMS-filtered boxes (BASELINE.json configs[2]:
PointPillars front end -> BaseBEVBackbone -> shrink -> MessageExtractorv2 -> GenComm 3-step diffusion sampler ->
Enhancer -> warp + AttFusion -> heads -> decode + rotated NMS), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape opv2v_h|v2xreal] [--dump-outputs DIR]

A "step" is one pass of the whole frame path over F synthetic frames per GPU (F x 4 agents x 100 k points; --shape v2xreal:
configs[3], 5 agents, C = 256).  Frames are independent, so ranks shard them (weak scaling); the path's one exchange step
-- the all-gather of the padded per-frame detections (SURVEY.md 8e) -- runs over NCCL inside the timed region when N > 1.
Secondary sections of the same line: the configs[1] HBM step (voxelize + PFN + scatter -> 256x256x64 canvas -> warp +
AttFusion) with its per-kernel roofline figures, the configs[3]-shaped frame, component microbenches.
Rank 0 prints ONE JSON line (contract: see the task statement / DESIGN.md section 7).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

POINTS = 100_000
FUSION = "att"
SHAPES = {
    "opv2v_h": {"agents": 4, "metric": "4-agent OPV2V-H-shape GenComm frames/s (raw points -> NMS-filtered boxes)",
                "workload": "configs[2]: GenComm stage-1 detector (m1_att.yaml model args), 4 LiDAR agents x 100k pts, "
                            "OPV2V-H grid 512x256, C=128 at 64x128, T=3 diffusion sampler, AttFusion, decode + rotated NMS"},
    "v2xreal": {"agents": 5, "metric": "5-agent V2X-Real-shape GenComm frames/s (raw points -> NMS-filtered boxes)",
                "workload": "configs[3]: GenComm detector at the V2X-Real shape (5 LiDAR agents x 100k pts, z +-15 m, "
                            "C=256 at 64x128, T=3 sampler, AttFusion, decode + rotated NMS), frames sharded over the GPUs, "
                            "NCCL all-gather of detections"},
}
HBM_WORKLOAD = "configs[1]: PointPillars + AttFusion, 4 agents x 100k pts, 256x256x64 BEV (voxelize+PFN+scatter -> warp+AttFusion)"


def env_int(name, default):
    return int(os.environ.get(name, default))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock, power and clock-event reasons of one GPU while the timed region runs: NVML in a background
    thread (every 20 ms: a 2 ms poll measurably slows the step, profiles/r02z_clock_sampler.txt), `nvidia-smi -lms` as the fallback when NVML is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        import threading
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.power = []
        self._stop = threading.Event()
        self.thread = self.p = self.f = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may remap indices: resolve through the PCI bus id of the current device
            bus = torch.cuda.get_device_properties(gpu_index).pci_bus_id if hasattr(
                torch.cuda.get_device_properties(gpu_index), "pci_bus_id") else None
            h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hi).bus == bus:
                        h = hi
                        break
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            names = {pynvml.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                     pynvml.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     pynvml.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     pynvml.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}

            def run():
                while not self._stop.is_set():
                    try:
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
                        mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        for bit, n in names.items():
                            if mask & bit:
                                self.reasons.add(n)
                    except Exception:
                        pass
                    time.sleep(float(os.environ.get("GC_BENCH_CLOCK_MS", "20")) * 1e-3)

            self.thread = threading.Thread(target=run, daemon=True)
            self.thread.start()
            self.how = "nvml"
        except Exception:
            self.how = "nvidia-smi"
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            try:
                self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                           "-lms", "20", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
            except OSError:
                self.p = None

    def mark(self):
        """Start of the timed region: drop what was sampled during warm-up."""
        self._mark = len(self.samples)

    def stop(self):
        if self.thread is not None:
            self._stop.set()
            self.thread.join(timeout=2)
            sm = self.samples[getattr(self, "_mark", 0):] or self.samples
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                    "power_w_max": max(self.power) if self.power else None, "samples": len(sm),
                    "reasons": sorted(self.reasons), "how": self.how}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = [r.strip().split(",") for r in self.f.read().splitlines() if r.count(",") >= 6]
        self.f.close()
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "how": self.how}


def load_tensor_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        if "bf16_tflops_sustained" in d:
            return float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
    return 2250.0, "fallback (nominal dense bf16, B200_PROFILING.md)"


def kernel_traffic(kernel):
    """ncu DRAM bytes per launch of `kernel` from the committed capture (profiles/traffic.json), or None when the capture
    is stale: every entry records the sha1 of the source file the kernel lived in when it was profiled."""
    import hashlib
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        entry = json.load(f).get(kernel)
    if not isinstance(entry, dict):
        return None
    src = os.path.join(ROOT, entry.get("source", ""))
    if not os.path.exists(src):
        return None
    with open(src, "rb") as f:
        if hashlib.sha1(f.read()).hexdigest() != entry.get("source_sha1"):
            return None
    return entry.get("dram_bytes_per_launch")


def bind_to_gpu_numa(local_rank):
    """Pin this process (and the pinned host buffers it allocates afterwards, first touch) to the CPUs of the NUMA node its
    GPU hangs off.  Without it every rank runs on node 0 and the host side of the copies serialises (round 1: e2e scaled
    1.6x on 8 GPUs).  Returns a description for the JSON line."""
    try:
        prop = torch.cuda.get_device_properties(local_rank)
        bus = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        cpus = set()
        if node >= 0:
            with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
                for part in f.read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
        else:   # sysfs has no node for the device (virtualised PCI): ask NVML for the ideal CPU set (nvidia-smi topo -m)
            import pynvml
            pynvml.nvmlInit()
            h = None
            for i in range(pynvml.nvmlDeviceGetCount()):
                hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                if pynvml.nvmlDeviceGetPciInfo(hi).bus == prop.pci_bus_id:
                    h = hi
            words = (os.cpu_count() + 63) // 64
            mask = pynvml.nvmlDeviceGetCpuAffinity(h, words) if h is not None else []
            for wi, word in enumerate(mask):
                cpus.update(wi * 64 + b for b in range(64) if (int(word) >> b) & 1)
            if not cpus:
                return {"numa_node": None, "note": "no NUMA / CPU affinity reported for the GPU"}
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node if node >= 0 else None, "cpus": len(allowed) if allowed else 0, "pci": bus,
                "source": "sysfs numa_node" if node >= 0 else "nvmlDeviceGetCpuAffinity"}
    except Exception as exc:   # best effort
        return {"numa_node": None, "note": repr(exc)}


# ------------------------------------------------------------------------------------------------
# CPU path (the oracle = restatement of the reference's algorithm; test/bench infrastructure only)
# ------------------------------------------------------------------------------------------------
_CPU_STAGES = ("voxelize", "pillar_vfe", "scatter", "bev_backbone", "downsample_conv", "message_extractor_v2",
               "gencomm_sample", "enhancer", "att_fusion", "det_heads", "post_process")


class CpuFrame:
    """One GenComm frame through the reference's CPU algorithm (oracle/ref_ops.py restates every stage with file:line
    citations; pinned to the unmodified reference classes by tests/golden): voxelize -> PillarVFE -> scatter -> backbone ->
    shrink -> MessageExtractorv2 -> GenComm (T=3) -> Enhancer -> warp + AttFusion -> heads -> decode + rotated NMS.
    Per-stage wall-clock through timing wrappers around the oracle's own stage functions."""

    def __init__(self, shape, device="cpu"):
        import gencomm_b200 as G
        from gencomm_b200 import synth
        from oracle import ref_ops as R
        self.R, self.synth, self.shape, self.device = R, synth, shape, torch.device(device)
        self.n_agents = SHAPES[shape]["agents"]
        self.args = synth.gencomm_v2xreal_args(FUSION) if shape == "v2xreal" else synth.gencomm_stage1_args(FUSION)
        m = G.HeterModelBaselineWGenComm(self.args)        # parameter container only: key names + shapes (no kernels run)
        self.sd = {k: v.to(self.device) for k, v in synth.fill_state_dict(m.state_dict(), 11).items()}
        self.rng = list(self.args["lidar_range"])
        self.vs = self.args["m1"]["encoder_args"]["voxel_size"]
        self.pp = synth.postprocess_params(score_threshold=0.6)
        self.pp["gt_range"] = list(self.rng)
        self.pp["anchor_args"]["cav_lidar_range"] = list(self.rng)
        self.anchors = torch.from_numpy(R.generate_anchor_box(self.pp["anchor_args"], self.pp["order"])).float()
        self._cur = {}
        self._wrapped = {}
        for name in _CPU_STAGES:
            if hasattr(R, name):
                self._wrap(name)

    def _wrap(self, name):
        fn = getattr(self.R, name)
        self._wrapped[name] = fn

        def timed(*a, **k):
            if self.device.type == "cuda":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn(*a, **k)
            if self.device.type == "cuda":
                torch.cuda.synchronize()
            self._cur[name] = self._cur.get(name, 0.0) + time.perf_counter() - t0
            return out
        setattr(self.R, name, timed)

    def close(self):
        for name, fn in self._wrapped.items():
            setattr(self.R, name, fn)

    def run(self, frame):
        R, synth, N, dev = self.R, self.synth, self.n_agents, self.device
        clouds = [synth.lidar_points(frame, a, POINTS, lidar_range=self.rng) for a in range(N)]
        pw = torch.from_numpy(synth.pairwise_t_matrix(frame, N, 5, spread=(40.0, 15.0))[None])
        C = int(self.args["in_head"])
        n0, steps = synth.sampler_noise(frame, N, C, 64, 128, T=3)
        self._cur = {}
        if dev.type == "cuda":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        vox = R.collate_voxels([R.voxelize(c, self.rng, self.vs, 32, 70000) for c in clouds])   # CPU (spconv is a CPU op)
        vox = {k: v.to(dev) for k, v in vox.items()}
        out = R.heter_gencomm_forward(self.sd, self.args, vox, pw.to(dev), torch.tensor([N]), n0.to(dev),
                                      [s.to(dev) for s in steps])
        boxes, scores = R.post_process(out["cls_preds"].cpu(), out["reg_preds"].cpu(), out["dir_preds"].cpu(), self.anchors,
                                       np.eye(4, dtype=np.float32), self.pp)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        self._cur["frame"] = dt
        return dt, (0 if boxes is None else int(boxes.shape[0]))

    def timed_frames(self, warmup, frames, seed0, budget_s):
        """warmup untimed frames, then up to `frames` timed ones (stops early once budget_s of timed work is spent, unless
        budget_s is None).  Returns (per-frame seconds, {stage: {median_ms, p90_ms}})."""
        for w in range(warmup):
            self.run(10_000 + seed0 + w)
        tot, ts, per = 0.0, [], []
        for k in range(frames):
            dt, _ = self.run(20_000 + seed0 + k)
            ts.append(dt)
            per.append(dict(self._cur))
            tot += dt
            if budget_s is not None and tot > budget_s:
                break
        stages = {}
        for name in list(_CPU_STAGES):
            v = [p[name] for p in per if name in p]
            if v:
                stages[name] = {"median_ms": round(1e3 * float(np.median(v)), 3), "p90_ms": round(1e3 * float(np.percentile(v, 90)), 3)}
        return ts, stages


def cpu_info():
    model = "unknown"
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    return model, os.cpu_count() or 1


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    shape = args.shape
    model, cores = cpu_info()
    torch.set_num_threads(cores)
    cpu = CpuFrame(shape)
    ts, stages = cpu.timed_frames(max(args.warmup, 1), args.steps, 0, budget_s=None)
    done, total = len(ts), float(np.sum(ts))
    fps = done / total
    k1 = None
    if args.cpu_protocol:   # BASELINE.md section 3: also k = 1 thread (bounded: a frame takes ~10x longer)
        torch.set_num_threads(1)
        t1, s1 = cpu.timed_frames(1, 3, 500, budget_s=120.0)
        torch.set_num_threads(cores)
        k1 = {"threads": 1, "frames": len(t1), "median_ms": 1e3 * float(np.median(t1)), "p90_ms": 1e3 * float(np.percentile(t1, 90)),
              "frames_per_s": len(t1) / float(np.sum(t1)), "stages": s1}
    cpu.close()
    gpu_eager = None
    if torch.cuda.is_available() and not args.no_gpu_eager:
        # the like-for-like GPU bar (BASELINE.md section 3): the SAME reference op sequence, torch eager on the B200
        # (cuDNN / ATen kernels, PyTorch defaults incl. TF32 convolutions); voxelization stays on the CPU as in the reference
        try:
            torch.cuda.set_device(env_int("LOCAL_RANK", 0))
            g = CpuFrame(shape, device="cuda")
            tg, sg = g.timed_frames(3, 20, 900, budget_s=60.0)
            g.close()
            gpu_eager = {"frames": len(tg), "median_ms": 1e3 * float(np.median(tg)), "p90_ms": 1e3 * float(np.percentile(tg, 90)),
                         "frames_per_s": len(tg) / float(np.sum(tg)), "stages": sg,
                         "note": "oracle op sequence (= the reference's torch ops) run eagerly on cuda:0, 1 frame per call, "
                                 "CPU voxelizer + H2D of the voxels + host NMS included as in the reference's loop"}
        except Exception as exc:
            gpu_eager = {"error": repr(exc)}
    sample = (f"{done} frames timed after {max(args.warmup, 1)} warm-up, 1 frame per "
              f"step ({SHAPES[shape]['agents']} agents x 100k pts), torch CPU threads={cores}, {model}")
    print(json.dumps({
        "impl": "reference", "metric": SHAPES[shape]["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": done, "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * total / done,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": SHAPES[shape]["workload"], "frames_per_step": 1, "agents": SHAPES[shape]["agents"],
                   "points_per_agent": POINTS, "fusion": FUSION},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample,
                         "cpu_model": model, "median_ms": 1e3 * float(np.median(ts)), "p90_ms": 1e3 * float(np.percentile(ts, 90)),
                         "stages": stages, "k1": k1},
        "gpu_eager_baseline": gpu_eager,
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------
# secondary measurements
# ------------------------------------------------------------------------------------------------
def _time_calls(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def gencomm_sampler_extra(dev, frames=8, agents=4, C=128, H=64, W=128, iters=20):
    """GenComm eval sampler (cond_diff.py:331-383) on F frames x N agents, device resident, pre-drawn noise, CUDA events."""
    import gencomm_b200 as G
    from gencomm_b200 import synth
    torch.manual_seed(0)
    m = G.GenComm({"model": {"embed_dim": C + 2, "in_channels": C, "out_ch": C, "ch": 8, "ch_mult": [1, 1],
                             "num_res_blocks": 2, "attn_resolutions": [16], "dropout": 0.0, "resamp_with_conv": True},
                   "diffusion": {"beta_schedule": "linear", "beta_start": 0.0005, "beta_end": 0.02,
                                 "num_diffusion_timesteps": 3}}).to(dev).eval()
    A = frames * agents
    feat = synth.bev_features(40, A, C, H, W).to(dev)
    cond = synth.bev_features(40, A, 2, H, W, salt=4).to(dev)
    n0, steps = synth.sampler_noise(40, A, C, H, W, T=3)
    noise = (n0.to(dev), torch.stack(steps).to(dev))
    rl = torch.full((frames,), agents, dtype=torch.int64, device=dev)   # on the device: no H2D copy inside the CUDA graph
    flop = 486.8e6 if C == 128 else 788.8e6
    hbm = A * 3 * (4 * (C + 2) * H * W + 8 * C * H * W)
    out = {"workload": f"GenComm sampler, {frames} frames x {agents} agents, C={C}, {H}x{W}, T=3", "mandatory_hbm_bytes": hbm}
    for name in ("cluster", "tc", "fp32"):
        m.precision = name
        ms = _time_calls(lambda: m(feat, cond, rl, noise=noise), iters)
        try:   # device time of the same call replayed from a CUDA graph (the eager figure includes the host launch path)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                m(feat, cond, rl, noise=noise)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                m(feat, cond, rl, noise=noise)
            eager_ms, ms = ms, _time_calls(graph.replay, iters)
        except Exception as exc:
            eager_ms = ms
            out.setdefault("graph_errors", {})[name] = repr(exc)
        out[name] = {"ms_per_call": ms, "eager_ms_per_call": eager_ms, "frames_per_s": frames / (ms * 1e-3),
                     "tflops": A * 3 * flop / (ms * 1e-3) / 1e12,
                     "hbm_frac_of_mandatory": hbm / (ms * 1e-3) / 1e9 / load_peaks()[0]}
    out["launches_per_call"] = {"cluster": 1 + 3 * 3, "tc": 1 + 3 * 28}
    out["precision_note"] = ("cluster (default): bf16 tcgen05 conv_in / conv_out + ONE cluster-resident launch for the 26 width-8 "
                             "layers (tf32 tcgen05, activations in distributed shared memory); tc: the same arithmetic as one "
                             "kernel per layer; fp32: all CUDA-core fp32")
    return out


def component_extras(dev, frames=8, agents=4, C=128, H=64, W=128, iters=10):
    import gencomm_b200 as G
    torch.manual_seed(0)
    A = frames * agents
    xs = [torch.randn(A, C, H, W, device=dev) for _ in range(3)]
    out = {}
    me = G.MessageExtractorv2(C, 2).to(dev).eval()
    k = [0]

    def call(m):
        k[0] += 1
        return m(xs[k[0] % 3])
    ms = _time_calls(lambda: call(me), iters)
    out["message_extractor"] = {"ms_per_call": ms, "tflops": 2.0 * A * H * W * (9 * C * (18 + 64) + 64 * 64 + 2 * 64) / (ms * 1e-3) / 1e12}
    en = G.Enhancer(C, [8, 8], 4).to(dev).eval()
    ms = _time_calls(lambda: call(en), iters)
    out["enhancer"] = {"ms_per_call": ms,
                       "tflops": 2.0 * A * H * W * (9 * (C // 4) ** 2 + 4 * C * C + 2 * C * C + 2 * C * 9) / (ms * 1e-3) / 1e12}
    out["workload"] = f"{frames} frames x {agents} agents, C={C}, {H}x{W}"
    return out


def hbm_step_section(dev, rank, F, K, Wm, peak):
    """BASELINE configs[1]: voxelize + PFN + scatter -> 256x256x64 canvas -> warp + AttFusion, device resident; the two
    north-star HBM kernels with the WHOLE front-end unit timed (voxelizer kernels included)."""
    from gencomm_b200 import pipeline, synth
    rng, pfn = synth.SQUARE_RANGE, synth.pfn_weights(0)
    pipe = pipeline.FramePipeline(F, 4, POINTS, rng, synth.VOXEL_SIZE, 70000, FUSION, 5, dev, pfn)
    n_sets = 3
    sets = []
    for s in range(n_sets):
        p, pw = pipeline.synthetic_step_inputs(1 + rank * n_sets + s, F, 4, POINTS, rng)
        sets.append((torch.from_numpy(p).to(dev), torch.from_numpy(pw).to(dev)))
    for w in range(Wm):
        pipe.step(*sets[w % n_sets])
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(K)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for k in range(K):
        ev[k][0].record()
        pipe.step(*sets[k % n_sets], ev_canvas=ev[k][1:3], ev_fuse=ev[k][3:5])
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / K
    front = float(np.mean([e[0].elapsed_time(e[2]) for e in ev]))      # voxelizer kernels + canvas writer
    canvas = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
    fuse = float(np.mean([e[3].elapsed_time(e[4]) for e in ev]))
    kern = {
        "front end: k_cell_assign2+k_pillar_build+k_canvas_persist (voxelize+PFN+scatter)":
            {"ms": front, "bytes": pipe.scatter_bytes()},
        "k_canvas_persist alone (PFN+scatter writer)": {"ms": canvas, "bytes": pipe.scatter_bytes()},
        "k_fuse_persist<ATT> (warp+regroup+AttFusion, 4x64x256x256)": {"ms": fuse, "bytes": pipe.fuse_bytes()},
    }
    for v in kern.values():
        v["gbs"] = v["bytes"] / (v["ms"] * 1e-3) / 1e9
        v["frac"] = v["gbs"] / peak
    return {"workload": HBM_WORKLOAD, "frames_per_step": F, "ms_per_step": ms, "frames_per_s": F / (ms * 1e-3),
            "l2": f"{n_sets} input sets cycled; {pipe.scatter_bytes() / 1e6:.0f} MB canvas traffic per step >> 126 MB L2",
            "kernels": kern, "checksum": float(pipe.fused.double().sum().item())}


# ------------------------------------------------------------------------------------------------
# GPU path
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    import gencomm_b200  # noqa: F401  (raises if the CUDA library is missing)
    from gencomm_b200 import pipeline, shard

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # the sampler noise is drawn on the device from the default CUDA generator, whose seed torch otherwise picks anew in
    # every process: seeded, so that every run with the same arguments draws the same noise and finds the same boxes
    torch.manual_seed(0)
    affinity = bind_to_gpu_numa(local)      # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    shape = args.shape
    N = SHAPES[shape]["agents"]
    F, K, Wm = args.frames_per_step, args.steps, max(args.warmup, 3)
    peak, peak_src = load_peaks()
    tpeak, tpeak_src = load_tensor_peak()

    # CPU baseline first (rank 0, N=1 only), bounded sample of the same workload
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        model, cores = cpu_info()
        torch.set_num_threads(cores)
        cpu = CpuFrame(shape)
        ts, stages = cpu.timed_frames(1, 6, 0, budget_s=20.0)
        cpu.close()
        cpu_baseline = {"value": len(ts) / float(np.sum(ts)), "unit": "frames/s", "cores": cores, "kind": "port",
                        "cpu_model": model, "median_ms": 1e3 * float(np.median(ts)), "stages": stages,
                        "sample": f"{len(ts)} frames ({N} agents x 100k pts each) of the same workload after 1 warm-up "
                                  f"(20 s cap), oracle restatement of the reference CPU path, torch threads={cores}"}

    pipe = pipeline.DetectorPipeline(F, N, POINTS, shape=shape, fusion=FUSION, device=dev)
    # steps in flight: consecutive steps alternate between independent pipeline instances (own weights, workspaces, planes)
    # on their own CUDA streams, so that the thin tails of one step -- NMS (15 - 128 CTAs), the sampler's 120-CTA cluster
    # launches, the last wave of every persistent kernel -- are filled by the other step's kernels
    n_fly = max(1, args.steps_in_flight)
    pipes = [pipe] + [pipeline.DetectorPipeline(F, N, POINTS, shape=shape, fusion=FUSION, device=dev) for _ in range(n_fly - 1)]
    n_sets = 3   # distinct input sets cycled; every stage streams >> 126 MB per step (canvas alone is 1.1 GB)
    host_pts, host_pw = [], []
    for s in range(n_sets):
        p, pw = pipeline.synthetic_detector_inputs(1 + rank * n_sets + s, F, N, POINTS, pipe.lidar_range)
        host_pts.append(torch.from_numpy(p).pin_memory())
        host_pw.append(torch.from_numpy(pw).pin_memory())
    dev_pts = [t.to(dev) for t in host_pts]
    dev_pw = [t.to(dev) for t in host_pw]
    gathered_det = [torch.empty((world * F, shard.DET_WIDTH), dtype=torch.float32, device=dev) if world > 1 else None
                    for _ in range(n_fly)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def full_step(pts, pw, i=0):
        boxes, scores, counts = pipes[i].step(pts, pw)
        if world > 1:      # the path's one exchange step: every rank ends the step with every frame's detections
            return shard.gather_detections_device(boxes, scores, counts, out=gathered_det[i])
        return boxes, scores, counts

    # ---------------- device-resident timing ----------------
    sampler = ClockSampler(local) if rank == 0 else None   # covers both timed regions (device-resident and e2e)
    pipe.enable_stage_timing()
    for w in range(Wm):
        full_step(dev_pts[w % n_sets], dev_pw[w % n_sets])
    torch.cuda.synchronize()
    pipe._marks.clear()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.mark()
    t_start.record()
    for k in range(K):
        res = full_step(dev_pts[k % n_sets], dev_pw[k % n_sets])
    t_end.record()
    barrier()
    elapsed_ms = serial_ms = t_start.elapsed_time(t_end)
    stage_ms = pipe.stage_ms(K)
    pipe._marks = None     # the regions below run on side streams: no hook events there
    if n_fly > 1:
        # the headline region: the same K steps, n_fly in flight.  (The region above, one step in flight with the per-stage
        # events, is what stage_ms / kernels / roofline are computed from and is reported as `one_in_flight`.)
        fly = [torch.cuda.Stream() for _ in range(n_fly)]
        cur = torch.cuda.current_stream()

        def fly_steps(n):
            out = None
            for st in fly:
                st.wait_stream(cur)
            for k in range(n):
                with torch.cuda.stream(fly[k % n_fly]):
                    out = full_step(dev_pts[k % n_sets], dev_pw[k % n_sets], k % n_fly)
            for st in fly:
                cur.wait_stream(st)
            return out

        fly_steps(max(Wm, 2 * n_fly))
        barrier()
        t_start.record()
        res = fly_steps(K)
        t_end.record()
        barrier()
        elapsed_ms = t_start.elapsed_time(t_end)
    det_counts = (res[:, 0] if world > 1 else res[2].float()).tolist()
    payload = res if world > 1 else shard.pack_detections(*res)
    checksum = float(payload.double().sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, payload)

    # ---------------- end-to-end timing: pinned host points -> device -> detections back in pinned host memory ----------------
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    slots = 2 * n_fly    # every step in flight is double buffered: the inputs of its successor on the same stream are
                         # copied in while it computes
    s_comps = [torch.cuda.Stream() for _ in range(n_fly)]   # slot s computes on pipeline / stream s % n_fly
    d_pts = [torch.empty_like(dev_pts[0]) for _ in range(slots)]
    d_pw = [torch.empty_like(dev_pw[0]) for _ in range(slots)]
    d_out = [torch.empty((F, shard.DET_WIDTH), dtype=torch.float32, device=dev) for _ in range(slots)]
    h_out = [torch.empty((F, shard.DET_WIDTH), dtype=torch.float32).pin_memory() for _ in range(slots)]
    ev_in = [torch.cuda.Event() for _ in range(slots)]
    ev_comp = [torch.cuda.Event() for _ in range(slots)]
    ev_out = [torch.cuda.Event() for _ in range(slots)]

    def e2e_step(k):
        s = k % slots
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_comp[s])          # compute of step k - slots has consumed this slot's inputs
            d_pts[s].copy_(host_pts[k % n_sets], non_blocking=True)
            d_pw[s].copy_(host_pw[k % n_sets], non_blocking=True)
            ev_in[s].record()
        s_comp = s_comps[s % len(s_comps)]
        with torch.cuda.stream(s_comp):
            s_comp.wait_event(ev_in[s])
            s_comp.wait_event(ev_out[s])         # D2H of step k - slots has drained this slot's result
            d_out[s].copy_(shard.pack_detections(*pipes[s % len(s_comps)].step(d_pts[s], d_pw[s])))
            ev_comp[s].record()
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_comp[s])
            h_out[s].copy_(d_out[s], non_blocking=True)
            ev_out[s].record()

    for w in range(max(Wm, slots)):
        e2e_step(w)
    barrier()
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_start.record(s_in)
    for k in range(K):
        e2e_step(k)
    for s_comp in s_comps:
        s_out.wait_stream(s_comp)
    s_out.wait_stream(s_in)
    e_end.record(s_out)
    barrier()
    e2e_ms = e_start.elapsed_time(e_end)
    clocks = sampler.stop() if sampler else None
    h2d = host_pts[0].numel() * 4 + host_pw[0].numel() * 8
    d2h = h_out[0].numel() * 4
    e2e_check = float(h_out[(K - 1) % slots].double().sum().item())

    # ---------------- secondary sections (rank 0, N = 1) ----------------
    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        del d_pts, d_pw, d_out
        for name, fn in (("hbm_step", lambda: hbm_step_section(dev, rank, 8, max(K, 50), 3, peak)),
                         ("gencomm_sampler", lambda: gencomm_sampler_extra(dev)),
                         ("components", lambda: component_extras(dev)),
                         ("other_shape", lambda: other_shape_section(dev, "v2xreal" if shape == "opv2v_h" else "opv2v_h", F)),
                         ("single_frame", lambda: single_frame_section(dev, shape))):
            try:
                extras[name] = fn()
            except Exception as exc:   # a secondary measurement must never take the headline down
                extras[name] = {"error": repr(exc)}
            torch.cuda.empty_cache()

    # ---------------- max over ranks, gather of checksums + timings ----------------
    times = torch.tensor([elapsed_ms, e2e_ms, serial_ms], dtype=torch.float64, device=dev)
    gathered = None
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        mine = torch.tensor([checksum, e2e_check, elapsed_ms, e2e_ms] + [stage_ms.get(k, 0.0) for k in STAGE_ORDER],
                            dtype=torch.float64, device=dev)
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
    elapsed_ms, e2e_ms, serial_ms = float(times[0]), float(times[1]), float(times[2])

    if rank == 0:
        frames = world * F * K
        work = pipe.work()
        kernels = {}
        for st, w in work.items():
            ms = stage_ms.get(st)
            if not ms:
                continue
            e = {"ms": ms, "bound": w["bound"]}
            if "bytes" in w:
                e.update({"bytes": w["bytes"], "gbs": w["bytes"] / (ms * 1e-3) / 1e9})
                e["hbm_frac"] = e["gbs"] / peak
            if "flops" in w:
                e.update({"flops": w["flops"], "tflops": w["flops"] / (ms * 1e-3) / 1e12})
                e["tensor_frac"] = e["tflops"] / tpeak
            if st == "pillars" and getattr(pipe.model.encoder_m1, "sparse_planes", False):
                e["note"] = ("bytes = SURVEY 8(d)'s dense figure (16 B per point + every canvas byte once), kept so that rounds "
                             "compare; the planes are maintained sparsely since r02bj -- a frame stores its occupied cells only "
                             "(k_pillar_planes_sparse) and zeroes them again after the backbone's first convolution "
                             "(k_planes_clear, ~0.08 ms per step, inside the backbone stage's time) -- so the DRAM traffic of the "
                             "stage is ~1.1 GB per step (+ 0.28 GB for the clear), not 2.1 GB: ncu per kernel in "
                             "profiles/r02bp_front_end_ncu.txt; hbm_frac is NOT a fraction of moved bytes for this stage")
            kernels[STAGE_KERNELS.get(st, st)] = e
        dom_stage = max(stage_ms, key=stage_ms.get)
        dom = kernels.get(STAGE_KERNELS.get(dom_stage, dom_stage))
        roofline = None
        if dom is not None:
            if dom["bound"] == "tensor":
                roofline = {"bound": "tensor", "kernel": STAGE_KERNELS[dom_stage], "achieved": dom["tflops"], "peak": tpeak,
                            "unit": "TFLOP/s", "frac": dom["tensor_frac"], "traffic": kernel_traffic("k_conv_tma"),
                            "issued_tflops": 3.0 * dom["tflops"], "issued_frac": 3.0 * dom["tensor_frac"],
                            "peak_source": tpeak_src, "algorithmic_flops_per_step": dom["flops"], "ms_per_step": dom["ms"],
                            "note": "achieved / frac count the dense fp32-grade convolution FLOPs of the 22 launches of the stage; the "
                                    "kernel issues 3 bf16 MMAs per product (bf16x3), so the tensor pipe executes issued_tflops = 3x "
                                    "that figure (issued_frac of the measured bf16 peak); traffic = ncu DRAM bytes of one 256-channel "
                                    "3x3 launch (profiles/traffic.json)"}
            else:
                roofline = {"bound": "hbm", "kernel": STAGE_KERNELS[dom_stage], "achieved": dom["gbs"], "peak": peak,
                            "unit": "GB/s", "frac": dom["hbm_frac"], "traffic": None, "peak_source": peak_src,
                            "algorithmic_bytes_per_step": dom["bytes"], "ms_per_step": dom["ms"]}
        line = {
            "metric": SHAPES[shape]["metric"], "value": frames / (elapsed_ms * 1e-3), "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (tensor-core operands bf16x3 / tf32 / bf16, fp32 accumulation)", "data": "synthetic",
            "config": {"workload": SHAPES[shape]["workload"], "frames_per_step_per_gpu": F, "agents": N,
                       "points_per_agent": POINTS, "grid": [pipe.nx, pipe.ny], "fusion": FUSION,
                       "sampler_precision": pipe.model.gencomm.precision, "weights": "seeded synthetic (synth.fill_state_dict)",
                       "noise": "drawn on the device with torch.randn inside the step, like the reference (GenComm.predraw: on a "
                                "side stream under the backbone)",
                       "steps_in_flight": n_fly,
                       "l2": f"{n_sets} distinct input sets cycled; every stage streams more than the 126 MB L2 per step "
                             f"(canvas {F * N * 64 * pipe.nx * pipe.ny * 4 / 1e6:.0f} MB)"},
            "clocks": clocks,
            "e2e": {"value": frames / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / K,
                    "note": "pinned host points + poses -> device -> padded detections (count | scores | boxes per frame) "
                            "copied back to pinned host memory; copy-in, copy-out and one compute stream per step in flight, "
                            "double buffered; ranks bound to their GPU's NUMA node"},
            "cpu_affinity": affinity,
            "collective": ({"op": "all_gather_into_tensor (NCCL)", "bytes_per_rank_per_step": F * shard.DET_WIDTH * 4,
                            "in_timed_region": True, "payload": "padded gc_postprocess output of the rank's frames"}
                           if world > 1 else None),
            "gpu_launches": K * pipeline_launches(pipe, stage_ms),
            "one_in_flight": {"ms_per_step": serial_ms / K, "frames_per_s": frames / (serial_ms * 1e-3),
                              "note": "the same K steps, one after the other on one stream, with the per-stage CUDA events: "
                                      "stage_ms, kernels and roofline are measured in this region"},
            "roofline": roofline,
            "kernels": kernels,
            "stage_ms": {k: round(v, 4) for k, v in stage_ms.items()},
            "detections_per_frame": det_counts[:F],
            "cpu_baseline": cpu_baseline,
            "checksum": checksum,
        }
        line.update(extras)
        if gathered is not None:
            line["per_rank"] = {"columns": ["checksum", "e2e_checksum", "elapsed_ms", "e2e_ms"] + list(STAGE_ORDER),
                                "rows": [[float(x) for x in g.tolist()] for g in gathered]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


STAGE_ORDER = ("pillars", "backbone", "shrink", "message_extractor", "sampler", "enhancer", "warp_fuse", "postprocess")
STAGE_KERNELS = {
    "pillars": "front end: k_cell_assign2+k_pillar_build+k_pillar_planes_sparse (voxelize+PFN+scatter into the "
               "backbone's bf16 operand planes, 512x256 grid)",
    "backbone": "k_conv_tma (BaseBEVBackbone, 19 3x3 + 3 phase-fused deblock TMA-fed tcgen05 implicit GEMMs, bf16x3)",
    "warp_fuse": "k_fuse_persist<ATT> (warp+regroup+AttFusion at the native shape)",
    "sampler": "GenComm sampler (k_q_sample, 3 x [k_conv_in_tc, k_unet_middle_cluster, k_conv_out_tc]; the torch.randn noise "
               "is drawn ahead on a side stream, under the backbone)",
}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, payload):
    """--dump-outputs: the detections of the last timed step, i.e. what the callers of DetectorPipeline.step receive
    (every rank's frames when N > 1), as out_dir/{frames,counts,scores,boxes}.npy: frame indices (float64), then float32
    counts [n], scores [n,1000] and boxes [n,1000,8,3] with the rows beyond each frame's count zeroed (gc_postprocess
    leaves them unspecified).  The inputs, and the sampler noise drawn from the seeded CUDA generator in a fixed order,
    are the same from run to run for the same arguments, so two builds can be compared output for output.  Above 64 MB
    a fixed, seeded sample of the frames is written."""
    p = payload.cpu().numpy()
    n, top = p.shape[0], (p.shape[1] - 1) // 25      # a row: count | scores [top] | boxes [top, 8, 3]
    frames = np.arange(n)
    keep = DUMP_LIMIT_BYTES // (p.shape[1] * 4 + 8)
    if n > keep:
        frames = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        p = p[frames]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"frames": frames.astype(np.float64), "counts": p[:, 0], "scores": p[:, 1:1 + top],
              "boxes": p[:, 1 + top:].reshape(len(frames), top, 8, 3)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def pipeline_launches(pipe, stage_ms):
    """Kernels of this repo launched per detector step (counted from the launch sequence of each stage; the torch.randn /
    elementwise launches of the wrappers are not counted)."""
    n = 3                      # front end: k_cell_assign2, k_pillar_build, k_pillar_planes_sparse (no to_planes)
    n += 22 + 1                # backbone: 19 convs + 3 deblocks (all phases of a ConvTranspose2d in one launch; shrink header's
                               # planes) + k_planes_clear after the first conv
    n += 2                     # shrink header: 2 convs
    n += 5                     # message extractor
    cluster = pipe.model.gencomm.precision == "cluster"
    n += 2 + 1 + 3 * (3 if cluster else 28)   # weight pack x2, q_sample, steps
    n += 11 + pipe.C // 64 + pipe.C // 128    # enhancer
    n += 2                     # normalize_pairwise_tfm + warp_fuse
    n += 2                     # heads: to_planes + GEMM
    n += 4                     # decode, select, iou, greedy
    return n


def other_shape_section(dev, shape, F):
    """The other frame shape (configs[3] when the headline is configs[2]) at N = 1, device resident."""
    from gencomm_b200 import pipeline
    N = SHAPES[shape]["agents"]
    pipe = pipeline.DetectorPipeline(F, N, POINTS, shape=shape, fusion=FUSION, device=dev)
    sets = []
    for s in range(2):
        p, pw = pipeline.synthetic_detector_inputs(50 + s, F, N, POINTS, pipe.lidar_range)
        sets.append((torch.from_numpy(p).to(dev), torch.from_numpy(pw).to(dev)))
    pipe.enable_stage_timing()
    k = [0]

    def call():
        k[0] += 1
        return pipe.step(*sets[k[0] % 2])
    for _ in range(2):
        det = call()
    torch.cuda.synchronize()
    pipe._marks.clear()
    iters = 6
    ms = _time_calls(call, iters, warm=0)
    stages = pipe.stage_ms(iters)
    return {"workload": SHAPES[shape]["workload"], "frames_per_step": F, "ms_per_step": ms, "frames_per_s": F / (ms * 1e-3),
            "stage_ms": {k2: round(v, 4) for k2, v in stages.items()}, "detections_per_frame": det[2].tolist()}


def single_frame_section(dev, shape):
    """The reference's actual operating point (tools/inference.py:114-120 runs batch 1): one frame per call, eager launches
    and the same sequence replayed from a CUDA graph."""
    from gencomm_b200 import pipeline
    N = SHAPES[shape]["agents"]
    pipe = pipeline.DetectorPipeline(1, N, POINTS, shape=shape, fusion=FUSION, device=dev)
    p, pw = pipeline.synthetic_detector_inputs(77, 1, N, POINTS, pipe.lidar_range)
    pts, pwd = torch.from_numpy(p).to(dev), torch.from_numpy(pw).to(dev)
    eager = _time_calls(lambda: pipe.step(pts, pwd), 20)
    out = {"workload": f"1 frame x {N} agents per call (batch-1 inference loop)", "eager_ms": eager}
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                pipe.step(pts, pwd)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            det = pipe.step(pts, pwd)
        ms = _time_calls(graph.replay, 50)
        out.update({"cuda_graph_ms": ms, "frames_per_s_graph": 1e3 / ms, "detections": int(det[2][0].item())})
    except Exception as exc:
        out["cuda_graph_error"] = repr(exc)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="opv2v_h", choices=sorted(SHAPES))
    ap.add_argument("--frames-per-step", type=int, default=15,
                    help="collaborative frames per step and GPU.  15 frames x 4 agents = 60 agents = four full rounds of the 15 "
                         "co-resident sampler clusters (8 frames: 32 agents = 2.13 rounds); measured 8 -> 876, 12 -> 882, 15 -> 925, "
                         "16 -> 921, 24 -> 925 frames/s (profiles/r02ax_frames_per_step.txt)")
    ap.add_argument("--steps-in-flight", type=int, default=2, choices=[1, 2, 3],
                    help="independent pipeline instances / CUDA streams the consecutive steps alternate between")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary sections (configs[1] HBM step, sampler, ...)")
    ap.add_argument("--cpu-protocol", action="store_true", help="--impl reference: also time k = 1 thread (BASELINE.md section 3)")
    ap.add_argument("--no-gpu-eager", action="store_true", help="--impl reference: skip the torch-eager-on-GPU bar")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the detections of the last timed step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    # The contract is ONE JSON line on stdout.  Libraries write to fd 1 behind Python's back (NCCL prints its version
    # banner there at communicator creation), so fd 1 is pointed at stderr for the whole run and the JSON line goes to a
    # private duplicate of the original stdout.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        real_stdout.flush()


if __name__ == "__main__":
    main()
