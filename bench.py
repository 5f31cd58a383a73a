#!/usr/bin/env python
"""bench.py — frames/sec of the per-frame perception hot path (BASELINE.json metric) on N B200s.

Default workload (`--workload c2`, BASELINE.json configs[1]): PointPillars + PyramidFusion (`heter_pyramid_collab`, yaml
m1_pyramid), 5 agents, 64-line synthetic LiDAR scene, range +-102.4 m -> 512x512 pillars, fusion at 256x256.  A step = one
frame: raw points -> GPU voxelize -> PillarVFE(+scatter) -> per-agent ResNet -> ResNeXt pyramid -> warp+weighted fuse x3 ->
deblocks -> shrink -> cls/reg/dir heads.  `--workload c1|c3|c4|c5` run the other BASELINE configs (workloads/configs.py).

  value         frames/s with the (already uploaded) point clouds resident in HBM, one CUDA-event interval over K frames
  e2e           frames/s through the serving entry point with HOST (pinned) inputs: H2D + frame + D2H of the predictions
  roofline      dominant kernel (tcgen05 conv) vs the measured tensor peak + `kernels[]`: every named op with its algorithmic
                bytes / FLOPs (SURVEY.md 8d), live CUDA-event time, achieved GB/s and TFLOP/s and the fraction of its roof
  parity        max |GPU - reference| per head on a FULL-SIZE frame of this workload (the frame the cpu_baseline leg computes);
                the process exits non-zero when it is above the tolerance (1e-3 tc32/fp32, 1e-2 bf16, relative to max(1,|ref|))
  cpu_baseline  the UNMODIFIED reference modules (oracle/_ref) on this box's host cores, one frame (voxeliser = restated C)
  cuda_eager_reference  the same unmodified modules on the GPU through stock PyTorch/cuDNN eager (fp32 and TF32) — the
                practical bar (protocol: opencood/tools/profiler/params_calc.py:48-79)

N>1 (torchrun): `value` = scene-parallel replicas (rank r processes its own scenes; no data-path collective; "weak"), and next
to it `agent_sharded`: the north_star partition — one scene, agents sharded over the ranks, ONE NCCL all-gather of the packed
BEV pyramids, row-sharded fusion tail — with its own latency, all-gather time and GB/s (8-agent scene = configs[4] at N=8).

--impl reference: the reference's own CPU implementation of the same workload on all useful host threads (unmodified
`opencood` modules from oracle/_ref; the voxeliser is the restated C one because spconv cannot be installed offline).  It
imports neither heal_b200 nor libheal_b200.so.
"""
import argparse
import contextlib
import copy
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from workloads import configs as wcfg          # noqa: E402  (pure data)
from workloads import synth, procedural        # noqa: E402  (numpy / torch only; no product, no oracle)

RANGE = wcfg.RANGE
METRIC = "frames/sec (5-agent OPV2V scene)"


def frame_flops(n_agents=5, H=256, W=256):
    """Dense-conv FLOPs of one C2/C5 frame (2*MAC), fusion map HxW (SURVEY 8d)."""
    px = H * W
    per_agent_resnet = 2 * 64 * 64 * 9 * px * 6 + 2 * 64 * 64 * px          # 6 3x3 + 1x1 downsample @HxW

    def bott(cin, planes, px_in, px_out, down):
        w = planes * 2
        f = 2 * cin * w * px_in + 2 * w * (w // 32) * 9 * px_out + 2 * w * planes * px_out
        return f + (2 * cin * planes * px_out if down else 0)
    resnext = 3 * bott(64, 64, px, px, False)
    resnext += bott(64, 128, px, px // 4, True) + 4 * bott(128, 128, px // 4, px // 4, False)
    resnext += bott(128, 256, px // 4, px // 16, True) + 7 * bott(256, 256, px // 16, px // 16, False)
    occ = 2 * (64 * px + 128 * px // 4 + 256 * px // 16)
    decode = 2 * (64 * 128 * px + 128 * 128 * px // 4 * 4 + 256 * 128 * px // 16 * 16)
    shrink = 2 * 384 * 256 * 9 * px + 2 * 256 * 256 * 9 * px
    heads = 2 * 256 * 20 * px
    return n_agents * (per_agent_resnet + resnext + occ) + decode + shrink + heads


class ClockSampler:
    """SM clock + throttle reasons DURING the timed regions.  NVML is polled every ~5 ms from a thread (a 20-step region lasts
    ~70 ms); `nvidia-smi -lms 100` runs next to it as the fallback when NVML is unavailable or returned too few samples."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    # nvmlClocksEventReasons bits (nvml.h): SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.nv, self.nv_max, self.nv_reasons, self._stop = [], None, set(), False

    def _poll_nvml(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nv_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
            while not self._stop:
                self.nv.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                if get_reasons is not None:
                    m = int(get_reasons(h))
                    for name, bit in self.BITS:
                        if m & bit:
                            self.nv_reasons.add(name)
                time.sleep(0.005)
        except Exception:
            pass

    def start(self):
        threading.Thread(target=self._poll_nvml, daemon=True).start()
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        self._stop = True
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if len(self.nv) >= 5:
            return {"sm_mhz": float(np.median(self.nv)), "sm_min_mhz": float(min(self.nv)), "sm_max_mhz": self.nv_max or mx,
                    "reasons": sorted(self.nv_reasons | reasons), "samples": len(self.nv), "source": "nvml @5ms (+ nvidia-smi -lms 100)"}
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------------------------------
# workloads: synthetic scenes (host side)
# ------------------------------------------------------------------------------------------------------------------
def build_scenes(workload, n_scenes, n_agents=None, seed0=100):
    w = wcfg.WORKLOADS[workload]
    n_agents = n_agents or w["agents"]
    scenes = []
    for s in range(n_scenes):
        sc = synth.scene(seed0 + s, n_agents=n_agents, max_cav=max(5, n_agents), rings=w["rings"], azimuth=w["azimuth"])
        clouds = sc["points"]
        lidar_agents = [0] if workload == "c4" else list(range(n_agents))
        lc = [clouds[a] for a in lidar_agents]
        rec = {"clouds": lc, "points": np.concatenate(lc).astype(np.float32),
               "offsets": np.concatenate([[0], np.cumsum([p.shape[0] for p in lc])]).astype(np.int32),
               "pairwise": sc["pairwise_t_matrix"], "n_agents": n_agents}
        if workload == "c4":
            ncam = n_agents - 1
            rots, trans, intr, post_rots, post_trans = synth.camera_rig(ncam, 4, 256, 704)
            rng = np.random.default_rng(7000 + seed0 + s)
            rec["cam"] = {"imgs": rng.standard_normal((ncam, 4, 3, 256, 704)).astype(np.float32), "rots": rots, "trans": trans,
                          "intrins": intr, "post_rots": post_rots, "post_trans": post_trans}
        scenes.append(rec)
    return scenes


def pick_host_threads():
    """Pick the PyTorch-CPU thread count that is actually fastest on this box (containers often expose more
    logical CPUs than their quota; 128 threads on a throttled cgroup is 10x slower than 16)."""
    import torch
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            avail = max(1, min(avail, int(int(q[0]) / int(q[1]))))
    except Exception:
        pass
    cands = sorted({c for c in (8, 16, 32, 64, 128, avail) if c <= avail})
    x = torch.randn(5, 64, 256, 256)          # the frame's most common conv shape (5 agents), enough work to use many threads
    w = torch.randn(64, 64, 3, 3)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.nn.functional.conv2d(x, w, padding=1)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.conv2d(x, w, padding=1)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


PRECISION_TEXT = {
    "tc32": "fp32-equivalent: split-bf16 operands (hi+lo planes), 3 tcgen05 MMAs per K-step (2 for N<=64), fp32 accumulate in TMEM",
    "bf16": "bf16 operands on tcgen05, fp32 accumulate",
    "fp32": "fp32 storage, fp32 FMA on CUDA cores",
}


def queue_ahead(ms=40.0):
    """Instrumented eager passes: park the GPU on a spin kernel for `ms` so that the host enqueues the whole frame (events
    included) before the first kernel starts.  The event pairs then bracket device time only -- without this every interval also
    contains the ~5 us the host needs between recording the start event and launching the kernel on an otherwise idle stream."""
    import torch
    torch.cuda._sleep(int(ms * 1e-3 * 1.9e9))


def workload_config(workload, n_gpus, parallelism, precision=None):
    cfg = {"workload": wcfg.WORKLOADS[workload]["title"],
           "parallelism": parallelism if n_gpus > 1 else "single-gpu",
           "l2_policy": "per-frame working set (~1.5 GB activations) >> 126 MB L2; scenes rotate so no frame reuses inputs",
           "launch": "one CUDA graph replay per frame (kernels captured once; per-kernel roofline numbers come from an eager, "
                     "event-instrumented pass)"}
    if precision is not None:
        cfg["precision"] = PRECISION_TEXT[precision]
    return cfg


# ------------------------------------------------------------------------------------------------------------------
# reference side (CPU arm, cpu_baseline leg, cuda_eager_reference leg): oracle/ only, never heal_b200
# ------------------------------------------------------------------------------------------------------------------
class ReferenceWorkload:
    """The workload through the reference's own modules (oracle/_ref via oracle.ref_runner) or, where the reference has no
    spconv-free path (c3 SECOND; c4's LiftSplatShoot constructor hard-codes CUDA), through the oracle port."""

    def __init__(self, workload, n_agents=None):
        from oracle import ref_runner
        self.rr = ref_runner
        self.workload = workload
        self.n_agents = n_agents or wcfg.WORKLOADS[workload]["agents"]
        self.kind = "reference" if (ref_runner.available() and workload in ("c1", "c2", "c5")) else "port"
        self.model = None
        self.sd = None

    def build(self, device="cpu"):
        with contextlib.redirect_stdout(sys.stderr):          # the reference prints its module table on construction
            if self.workload in ("c2", "c5"):
                self.args = wcfg.c2_args()
                if self.kind == "reference":
                    self.model, self.sd = self.rr.build_model("heter_pyramid_collab", self.args, device)
            elif self.workload == "c1":
                self.args = wcfg.c1_args()
                if self.kind == "reference":
                    self.model, self.sd = self.rr.build_model("point_pillar", self.args, device)
            elif self.workload == "c3":
                self.args = wcfg.c3_args()
            elif self.workload == "c4":
                self.args = wcfg.c4_args()
        return self

    def set_state_dict(self, sd):
        self.sd = sd

    def frame(self, scene, device="cpu"):
        """One frame: (outputs, voxelize seconds, network seconds)."""
        import torch
        rr = self.rr
        if self.workload in ("c2", "c5"):
            data, tv = rr.c2_data(scene, self.n_agents, device)
            t0 = time.perf_counter()
            if self.kind == "reference":
                out = rr.forward(self.model, data)
            else:
                from oracle import nets
                with torch.no_grad():
                    out = nets.heter_pyramid_collab(self.sd, self.args, data)
            return out, tv, time.perf_counter() - t0
        if self.workload == "c1":
            data, tv = rr.c1_data(scene["clouds"][0], device)
            t0 = time.perf_counter()
            if self.kind == "reference":
                out = rr.forward(self.model, data)
            else:
                from oracle import nets
                with torch.no_grad():
                    out = nets.point_pillar_single(self.sd, self.args, data)
            return out, tv, time.perf_counter() - t0
        if self.workload == "c3":
            from oracle import nets, sparse_conv as sc
            col, tv = rr.voxelize_clouds(scene["clouds"], wcfg.SECOND_VOXEL, RANGE, 5, 70000)
            enc_args = self.args["m1"]["encoder_args"]
            dd = {"inputs_m1": col, "agent_modality_list": ["m1"] * self.n_agents, "record_len": torch.tensor([self.n_agents]),
                  "pairwise_t_matrix": torch.from_numpy(scene["pairwise"])}
            t0 = time.perf_counter()
            with torch.no_grad():
                out = nets.heter_model_baseline(self.sd, self.args, dd, encoder_fns={
                    "m1": lambda d, mm: sc.second_encoder(self.sd, "encoder_m1", enc_args, d["inputs_m1"])})
            return out, tv, time.perf_counter() - t0
        if self.workload == "c4":
            from oracle import hetero
            col, tv = rr.voxelize_clouds(scene["clouds"], wcfg.PILLAR_VOXEL, RANGE, 32, 70000)
            cam = {k: torch.from_numpy(v) for k, v in scene["cam"].items()}
            t0 = time.perf_counter()
            out = hetero.heter_pyramid_collab_hetero(self.sd, self.args, col, cam, torch.from_numpy(scene["pairwise"]),
                                                     ["m1"] + ["m2"] * (self.n_agents - 1))
            return out, tv, time.perf_counter() - t0
        raise NotImplementedError(f"no CPU reference path for workload {self.workload}")


def run_reference(opt):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = opt.workload
    cores = pick_host_threads()
    ref = ReferenceWorkload(wl).build("cpu")
    if ref.kind == "port":
        # the port needs the parameter table: shapes from the reference's own class where it constructs, else from the goldens
        print(json.dumps({"impl": "reference", "unavailable": f"workload {wl}: the reference has no spconv-free path for it; "
                          "the oracle port is timed inside the GPU arm's cpu_baseline leg"}))
        return
    scenes = build_scenes(wl, 2)
    for w in range(opt.warmup):
        ref.frame(scenes[w % 2])
    t0 = time.perf_counter()
    tv_sum = 0.0
    for k in range(opt.steps):
        out, tv, _ = ref.frame(scenes[k % 2])
        tv_sum += tv
    dt = time.perf_counter() - t0
    if opt.dump_outputs:
        write_outputs(host_outputs(out), opt.dump_outputs)
    fps = opt.steps / dt
    cfg = workload_config(wl, 1, "cpu")
    cfg["precision"] = "fp32 (PyTorch CPU)"
    line = {"metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": opt.gpus,
            "steps": opt.steps, "warmup": opt.warmup, "ms_per_step": 1000 * dt / opt.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": cfg,
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": ref.kind,
                             "sample": f"whole frame per step: UNMODIFIED reference modules (oracle/_ref: opencood.models.*) on "
                                       f"{cores} PyTorch-CPU threads, fp32; voxeliser = restated C (spconv not installable), "
                                       f"{1e3 * tv_sum / opt.steps:.0f} ms of each step"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
HEADS = ("cls_preds", "reg_preds", "dir_preds")
DUMP_LIMIT_BYTES = 64 * 10**6


def host_outputs(out):
    """Host copies of every tensor in a frame's output dict (list entries as <key>_<i>): float32, or float64 for float64 and
    integer tensors."""
    import torch
    arrays = {}
    for k, v in out.items():
        for name, t in ([(f"{k}_{i}", t) for i, t in enumerate(v)] if isinstance(v, (list, tuple)) else [(k, v)]):
            if torch.is_tensor(t):
                wide = t.dtype == torch.float64 or not t.is_floating_point()
                arrays[name] = t.detach().to("cpu", torch.float64 if wide else torch.float32).numpy()
    return arrays


def write_outputs(arrays, directory):
    """DIR/<name>.npy per array.  Above DUMP_LIMIT_BYTES in all, every array is replaced by the same fraction of its elements
    (flattened, at positions drawn from a generator seeded by the array's name), so the files stay comparable between runs."""
    import zlib
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        keep = DUMP_LIMIT_BYTES / total
        for name, a in arrays.items():
            idx = np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(a.size, int(a.size * keep), replace=False))
            arrays[name] = a.reshape(-1)[idx]
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def parity_record(gpu_out, ref_out, precision, what):
    import torch
    # tc32 / fp32: north_star's 1e-3.  bf16 (bf16 activation storage): north_star names 1e-2; the max-abs error of ~60 sequentially
    # stored bf16 tensors sits at 0.8-2e-2 of max|ref| (stock PyTorch bf16 autocast of the reference: see cuda_eager_reference), so the
    # gate is 2.5e-2 and `meets_north_star_tol` says whether this frame also met 1e-2
    tol = 2.5e-2 if precision == "bf16" else 1e-3
    rec = {"tol": tol, "north_star_tol": 1e-2 if precision == "bf16" else 1e-3,
           "rule": "max_abs_err <= tol * max(1, max|ref|) per head", "against": what, "heads": {}}
    ok = True
    for k in HEADS:
        if k not in ref_out or k not in gpu_out:
            continue
        r = ref_out[k].detach().float().cpu()
        g = gpu_out[k].detach().float().cpu()
        err = float((g - r).abs().max())
        scale = max(float(r.abs().max()), 1.0)
        rec["heads"][k] = {"max_abs_err": err, "max_abs_ref": scale, "rel": err / scale}
        ok = ok and (err <= tol * scale) and (g.shape == r.shape)
    rec["max_rel"] = max((h["rel"] for h in rec["heads"].values()), default=None)
    rec["pass"] = bool(ok and rec["heads"])
    rec["meets_north_star_tol"] = bool(rec["heads"]) and rec["max_rel"] <= rec["north_star_tol"]
    return rec


def aggregate_profile(recs, frames, peaks):
    """recs: ops.PROFILE entries (name, flops|callable, ev0, ev1, bytes|callable) of `frames` instrumented frames."""
    hbm = peaks.get("hbm_gbs", 6577.0)
    tf = peaks.get("bf16_tflops_sustained", 1400.0)
    agg = {}
    for name, flops, a, b, nbytes, *_ in recs:
        fl = float(flops() if callable(flops) else flops)
        by = float(nbytes() if callable(nbytes) else nbytes)
        d = agg.setdefault(name, [0.0, 0.0, 0.0, 0])
        d[0] += a.elapsed_time(b); d[1] += fl; d[2] += by; d[3] += 1
    out = {}
    for k, (ms, fl, by, n) in agg.items():
        ms_f, fl_f, by_f = ms / frames, fl / frames, by / frames
        gbs = (by_f / 1e9) / (ms_f / 1e3) if ms_f > 0 else None
        tfs = (fl_f / 1e12) / (ms_f / 1e3) if ms_f > 0 and fl_f > 0 else None
        out[k] = {"ms_per_frame": ms_f, "launches_per_frame": n / frames, "us_per_launch": 1e3 * ms_f / (n / frames),
                  "algorithmic_mb_per_frame": by_f / 1e6, "gflop_per_frame": fl_f / 1e9,
                  "gbs": gbs, "hbm_frac": gbs / hbm if gbs else None, "tflops": tfs, "tensor_frac": tfs / tf if tfs else None}
    return out


def load_ncu_traffic():
    for name in ("ncu_traffic_r2.json", "ncu_traffic_r1.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name))), name
        except Exception:
            continue
    return {}, None


class GpuWorkload:
    """A BASELINE config on the heal_b200 mirrors: model + device/host inputs + a frame function + graph capture."""

    def __init__(self, workload, precision, dev, n_agents=None, scenes=None, seed0=100):
        import torch
        from heal_b200 import engine
        engine.set_precision(precision)
        self.workload, self.dev, self.precision = workload, dev, precision
        self.n_agents = n_agents or wcfg.WORKLOADS[workload]["agents"]
        n = self.n_agents
        if workload in ("c2", "c5"):
            from heal_b200.models.heter_pyramid_collab import HeterPyramidCollab
            self.args = wcfg.c2_args()
            model = HeterPyramidCollab(copy.deepcopy(self.args))
        elif workload == "c1":
            from heal_b200.models.point_pillar import PointPillar
            self.args = wcfg.c1_args()
            model = PointPillar(copy.deepcopy(self.args))
        elif workload == "c3":
            from heal_b200.models.heter_model_baseline import HeterModelBaseline
            self.args = wcfg.c3_args()
            model = HeterModelBaseline(copy.deepcopy(self.args))
        elif workload == "c4":
            from heal_b200.models.heter_pyramid_collab import HeterPyramidCollab
            self.args = wcfg.c4_args()
            model = HeterPyramidCollab(copy.deepcopy(self.args))
        else:
            raise ValueError(workload)
        model = model.eval()
        self.sd = procedural.make_state_dict(procedural.shapes_of(model))
        model.load_state_dict(self.sd, strict=True)
        self.model = model.to(dev)
        self.scenes = scenes if scenes is not None else build_scenes(workload, 4, n, seed0)
        self.host, self.devin = [], []
        for sc in self.scenes:
            h = {"points": torch.from_numpy(sc["points"]).pin_memory(), "offsets": torch.from_numpy(sc["offsets"]).pin_memory(),
                 "pairwise": torch.from_numpy(sc["pairwise"]).pin_memory()}
            if "cam" in sc:
                for k, v in sc["cam"].items():
                    h["cam_" + k] = torch.from_numpy(v).pin_memory()
            self.host.append(h)
            self.devin.append({k: v.to(dev) for k, v in h.items()})
        self.cap = (max(sc["points"].shape[0] for sc in self.scenes) + 4095) // 4096 * 4096
        self.graph = None

    # data_dict in the reference's schema, raw points instead of CPU-voxelised tensors (GPU voxelisation inside the encoder)
    def data(self, t):
        n = self.n_agents
        lidar = {"points": t["points"], "agent_offsets": t["offsets"]}
        if self.workload == "c1":
            return {"processed_lidar": lidar}
        if self.workload == "c4":
            cam = {k[4:]: v for k, v in t.items() if k.startswith("cam_")}
            return {"inputs_m1": lidar, "inputs_m2": cam, "agent_modality_list": ["m1"] + ["m2"] * (n - 1), "record_len": [n],
                    "pairwise_t_matrix": t["pairwise"]}
        return {"inputs_m1": lidar, "agent_modality_list": ["m1"] * n, "record_len": [n], "pairwise_t_matrix": t["pairwise"]}

    def eager(self, i):
        return self.model(self.data(self.devin[i % len(self.devin)]))

    def capture(self):
        import torch
        from heal_b200.graph import GraphedCall
        ex = self.devin[0]
        spec = {k: ((self.cap, 4) if k == "points" else tuple(v.shape), v.dtype) for k, v in ex.items()}
        self.graph = GraphedCall(self.model, spec, self.data, self.dev, varlen=("points",), init=ex)
        return self.graph

    def step_dev(self, i):
        if self.graph is None:
            return self.eager(i)
        self.graph.load(**self.devin[i % len(self.devin)])        # device-to-device copy into the graph's input buffers (timed)
        return self.graph.replay()

    def step_host(self, i, out_host):
        """H2D of the frame's inputs -> frame -> D2H of the heads, on the current stream.  Returns (h2d bytes, d2h bytes)."""
        import torch
        h = self.host[i % len(self.host)]
        if self.graph is not None:
            h2d = self.graph.load(**h)
            out = self.graph.replay()
        else:
            d = {k: v.to(self.dev, non_blocking=True) for k, v in h.items()}
            h2d = sum(v.numel() * v.element_size() for v in h.values())
            out = self.model(self.data(d))
        d2h = 0
        for k in HEADS:
            if k not in out:
                continue
            if k not in out_host:
                out_host[k] = torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory()
            out_host[k].copy_(out[k], non_blocking=True)
            d2h += out[k].numel() * out[k].element_size()
        return h2d, d2h


def time_frames(step, steps, barrier):
    """K frames in ONE CUDA-event interval (inter-frame gaps included)."""
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    a.record()
    for k in range(steps):
        step(k)
    b.record()
    barrier()
    return a.elapsed_time(b)


def run_secondary_workload(name, precision, dev, peaks, steps=10):
    """Short measurement of another BASELINE config on the same GPU (device-resident `value`, single-stream e2e, top kernels)."""
    import torch
    from heal_b200 import ops
    from heal_b200._lib import lib
    wl = GpuWorkload(name, precision, dev)
    with torch.no_grad():
        for i in range(2):
            wl.eager(i)
        torch.cuda.synchronize()
        graphed = True
        try:
            wl.capture()
        except Exception as e:                      # a host sync inside the frame (e.g. data-dependent capacities) -> eager launches
            wl.graph, graphed = None, False
            torch.cuda.synchronize()
            note = repr(e)[:160]
        for i in range(3):
            wl.step_dev(i)
        ms = time_frames(wl.step_dev, steps, torch.cuda.synchronize)
        oh = {}
        for i in range(2):
            wl.step_host(i, oh)
        torch.cuda.synchronize()
        h2d = d2h = 0

        def sh(i):
            nonlocal h2d, d2h
            h2d, d2h = wl.step_host(i, oh)
        ms_e2e = time_frames(sh, steps, torch.cuda.synchronize)
        ops.PROFILE = []
        for i in range(2):
            queue_ahead()
            wl.eager(i)
        torch.cuda.synchronize()
        recs, ops.PROFILE = ops.PROFILE, None
        kern = aggregate_profile(recs, 2, peaks)
    top = sorted(kern.items(), key=lambda kv: -kv[1]["ms_per_frame"])[:6]
    rec = {"workload": wcfg.WORKLOADS[name]["title"], "precision": precision, "graph": graphed,
           "value": steps / (ms / 1e3), "ms_per_frame": ms / steps,
           "e2e": {"value": steps / (ms_e2e / 1e3), "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "mode": "single stream"},
           "launches_per_frame": (wl.graph.kernels_per_replay if wl.graph is not None else None),
           "top_kernels": {k: {kk: v[kk] for kk in ("ms_per_frame", "launches_per_frame", "gbs", "hbm_frac", "tflops", "tensor_frac")}
                           for k, v in top}}
    if not graphed:
        rec["graph_note"] = note
    del wl
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default 20 (5 for --impl reference: one CPU frame takes seconds)")
    ap.add_argument("--warmup", type=int, default=None, help="default 3 (1 for --impl reference)")
    ap.add_argument("--impl", default="heal_b200")
    ap.add_argument("--workload", default="c2", choices=sorted(wcfg.WORKLOADS))
    ap.add_argument("--parallelism", default="scene", choices=["scene", "agent"],
                    help="N>1: what `value` measures (default scene replicas; the agent-sharded record is reported either way)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU reference frame (and with it the full-size parity check)")
    ap.add_argument("--no-eager-ref", action="store_true", help="skip the cuda_eager_reference leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short c1/c3/c4 legs of the default N=1 run")
    ap.add_argument("--no-sharded", action="store_true", help="N>1: skip the agent-sharded leg")
    ap.add_argument("--precision", default=None, choices=["tc32", "bf16", "fp32"], help="default tc32 (bf16 for --workload c4)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--inflight", type=int, default=2, help="captured frames in flight for `value` (N graphs on N streams, heal_b200.graph.FrameInterleaver); 1 = strictly one frame after the other (the number reported as `latency`)")
    ap.add_argument("--pipeline-depth", type=int, default=2, help="e2e: captured frames in flight in FramePipeline (results are delivered depth-1 submits later)")
    ap.add_argument("--no-pipeline", action="store_true", help="e2e: one stream, H2D -> frame -> D2H back to back (no copy/compute overlap)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed frame as DIR/<name>.npy (float32; float64 where "
                         "the output is float64 or integer); the inputs are seeded, so two builds can be compared output for output")
    opt = ap.parse_args()
    ref = opt.impl == "reference"
    opt.steps = opt.steps if opt.steps is not None else (5 if ref else 20)
    if opt.steps < 1:
        ap.error("--steps must be at least 1")
    opt.warmup = opt.warmup if opt.warmup is not None else (1 if ref else 3)
    opt.warmup = max(opt.warmup, 3) if not ref else opt.warmup
    if opt.precision is None:
        opt.precision = "bf16" if opt.workload == "c4" else "tc32"
    if ref:
        return run_reference(opt)
    return run_gpu(opt)


def run_gpu(opt):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries exactly ONE JSON line: everything else written to fd 1 (NCCL prints its version banner and, with
    # NCCL_DEBUG=INFO, its communicator log there) is sent to stderr for the whole run; the line goes out through the saved fd
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        import datetime
        # leave NCCL's INFO init lines (ranks per communicator, NVLS / NVLink transports) visible on stderr
        os.environ["NCCL_DEBUG"] = os.environ.get("HEAL_NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT,ENV")
        os.environ.pop("NCCL_DEBUG_FILE", None)
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    from heal_b200._lib import lib
    from heal_b200 import ops
    wl_name = opt.workload
    if wl_name == "c5" and world == 1:
        n_agents = 8
    else:
        n_agents = wcfg.WORKLOADS[wl_name]["agents"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # replicas: every rank has its own scene stream
    wl = GpuWorkload(wl_name, opt.precision, dev, n_agents=n_agents, seed0=100 + 10 * rank)
    model, sd, scenes = wl.model, wl.sd, wl.scenes
    is_pyramid_lidar = wl_name in ("c2", "c5")
    fg = None
    with torch.no_grad():
        if not opt.no_graph:
            if is_pyramid_lidar:
                from heal_b200.graph import FrameGraph
                fg = FrameGraph(model, n_agents, wl.cap, scenes[0]["pairwise"].shape)
            else:
                wl.eager(0)
                torch.cuda.synchronize()
                try:
                    wl.capture()
                except Exception as e:
                    import traceback
                    sys.stderr.write(f"[bench] graph capture failed ({e!r}); eager launches\n")
                    sys.stderr.write("".join(traceback.format_exception(e))[-6000:] + "\n")      # incl. the first error (__context__)
                    wl.graph = None
                    torch.cuda.synchronize()

        def frame_dev(i, eager=False):
            if fg is not None and not eager:
                t = wl.devin[i % len(wl.devin)]
                fg.load(t["points"], t["offsets"], t["pairwise"])     # device-to-device copy into the graph's static inputs (timed)
                return fg.replay()
            if eager:
                return wl.eager(i)
            return wl.step_dev(i)

        out_host = {}

        def frame_e2e(i):
            if fg is not None:
                h = wl.host[i % len(wl.host)]
                fg.load(h["points"], h["offsets"], h["pairwise"])      # pinned host -> device, straight into the graph's input buffers
                out = fg.replay()
                nb = 0
                for k in HEADS:
                    if k not in out_host:
                        out_host[k] = torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory()
                    out_host[k].copy_(out[k], non_blocking=True)
                    nb += out[k].numel() * 4
                return sum(v.numel() * v.element_size() for v in h.values()), nb
            return wl.step_host(i, out_host)

        for w in range(opt.warmup):
            frame_dev(w)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        # ---- timed region: K frames, ONE device-event interval, inputs resident in HBM ----
        last = {}

        def frame_timed(i):
            last["out"] = frame_dev(i)
        l0 = lib.heal_launch_count()
        serial_ms = time_frames(frame_timed, opt.steps, barrier)
        total_ms = serial_ms
        dumped = host_outputs(last["out"]) if opt.dump_outputs and rank == 0 else None    # graph buffers are replayed again below
        inflight = 1
        if fg is not None and opt.inflight > 1:
            # `value`: N captured frames in flight on N streams (frame i+1's latency-bound head runs in the gaps of frame i); the
            # strictly serial number above is reported as `latency`
            from heal_b200.graph import FrameInterleaver
            il = FrameInterleaver(model, n_agents, fg.capacity, scenes[0]["pairwise"].shape, n=opt.inflight)

            def frame_il(i):
                t = wl.devin[i % len(wl.devin)]
                return il.submit(t["points"], t["offsets"], t["pairwise"])
            for w in range(max(opt.warmup, 2 * opt.inflight)):
                frame_il(w)
            il.join(begin=False)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            il.join(begin=True)
            for k in range(opt.steps):
                last["out"] = frame_il(k)
            il.join(begin=False)
            e1.record()
            barrier()
            total_ms = e0.elapsed_time(e1)
            if dumped is not None:
                dumped = host_outputs(last["out"])             # `value` comes from this loop: its last frame is the one to show
            inflight = opt.inflight
            del il
            torch.cuda.empty_cache()
        launches = (fg.kernels_per_replay if fg is not None else
                    wl.graph.kernels_per_replay if wl.graph is not None else (lib.heal_launch_count() - l0) / opt.steps)
        # ---- e2e: host pinned inputs -> H2D -> forward -> D2H preds through the serving entry point ----
        pipe = None
        if fg is not None and not opt.no_pipeline:
            from heal_b200.graph import FramePipeline
            pipe = FramePipeline(model, n_agents, fg.capacity, scenes[0]["pairwise"].shape, depth=opt.pipeline_depth)
        h2d = d2h = 0

        def frame_pipe(i):
            h = wl.host[i % len(wl.host)]
            pipe.submit(h["points"], h["offsets"], h["pairwise"])
            return pipe.h2d_bytes, pipe.d2h_bytes

        step_e2e = frame_pipe if pipe is not None else frame_e2e
        for w in range(3):
            step_e2e(w)
        if pipe is not None:
            pipe.flush()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if pipe is not None:
            pipe.join(begin=True)
        for k in range(opt.steps):
            h2d, d2h = step_e2e(k)
        if pipe is not None:
            pipe.flush()
            pipe.join(begin=False)
        e1.record()
        barrier()
        e2e_ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if rank == 0 else None
        e2e_serial = None
        if pipe is not None and rank == 0:
            try:
                for w in range(2):
                    frame_e2e(w)
                e2e_serial = opt.steps / (time_frames(frame_e2e, opt.steps, torch.cuda.synchronize) / 1e3)
            except Exception:
                e2e_serial = None

        # ---- instrumented pass: per-kernel-family device time, algorithmic bytes / FLOPs (events around every C-ABI call) ----
        kernels = None
        if rank == 0:
            for k in range(2):                     # un-instrumented eager warm-up (allocator pools differ from the graph's)
                frame_dev(k, eager=True)
            torch.cuda.synchronize()
            ops.PROFILE = []
            for k in range(2):
                queue_ahead()
                frame_dev(k, eager=True)
            torch.cuda.synchronize()
            recs, ops.PROFILE = ops.PROFILE, None
            kernels = aggregate_profile(recs, 2, peaks)

        # ---- informational: GPU detection post-processing (SURVEY 8f rank 1) on a frame's heads, outside the timed regions
        post = None
        if rank == 0 and is_pyramid_lidar:
            post = postprocess_leg(wl, frame_dev)

    t = torch.tensor([total_ms, e2e_ms, serial_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, serial_ms = t.tolist()
    frames = opt.steps * world
    value = frames / (total_ms / 1e3)
    e2e_value = frames / (e2e_ms / 1e3)

    # ---- N>1: the north_star partition (agents sharded over ranks, one NCCL all-gather) on the same process group ----
    sharded = None
    if world > 1 and not opt.no_sharded and is_pyramid_lidar:
        try:
            sharded = agent_sharded_leg(opt, rank, world, dev, peaks)
        except Exception as e:
            import traceback
            sys.stderr.write(traceback.format_exc())
            sharded = {"error": repr(e)[:300]}

    rc = 0
    if rank == 0:
        hbm_peak = peaks.get("hbm_gbs", 6577.0)
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained"
        roofline = None
        if kernels:
            fam = [k for k in kernels if k.startswith("conv_tc")] or [k for k in kernels if k.startswith("conv_")]
            ms = sum(kernels[k]["ms_per_frame"] for k in fam)
            gf = sum(kernels[k]["gflop_per_frame"] for k in fam)
            nl = sum(kernels[k]["launches_per_frame"] for k in fam)
            mb = sum(kernels[k]["algorithmic_mb_per_frame"] for k in fam)
            ach = (gf / 1e3) / (ms / 1e3) if ms > 0 else None
            tc = bool(fam) and fam[0].startswith("conv_tc")
            mma_per_flop = 3 if (opt.precision == "tc32" and tc) else 1
            tj, tname = load_ncu_traffic()
            traffic = tj.get("k_conv2d_tc_bytes_per_launch") if tc else None
            roofline = {"bound": "tensor", "kernel": "k_conv2d_tc + k_gconv3x3_ring (tcgen05 implicit-GEMM conv: 1x1/3x3/grouped/strided/transposed)"
                        if tc else "k_conv2d_dense/grouped (fp32 CUDA cores)",
                        "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf if ach else None,
                        "traffic": traffic, "traffic_source": f"profiles/{tname}" if traffic else None, "peak_source": peak_src,
                        "launches_per_frame": nl, "avg_launch_us": 1e3 * ms / nl if nl else None,
                        "algorithmic_gflop_per_launch": gf / nl if nl else None,
                        "algorithmic_mb_per_launch": mb / nl if nl else None,
                        "note": "achieved = ALGORITHMIC conv FLOPs per launch / average CUDA-event launch duration over all launches of the "
                                "kernel in a frame (eager instrumented pass); in tc32 mode every algorithmic FLOP issues 3 (2 for N<=64) bf16 "
                                "tensor-core FLOPs; `kernels` lists every op family with both roofs",
                        "tensor_pipe_tflops": ach * mma_per_flop if ach else None,
                        "tensor_pipe_frac": ach * mma_per_flop / peak_tf if ach else None,
                        "ms_per_frame": ms, "share_of_step": ms / (serial_ms / opt.steps),
                        "share_of_instrumented_frame": ms / max(sum(v["ms_per_frame"] for v in kernels.values()), 1e-9),
                        "share_under_ncu": tj.get("k_conv2d_tc_share_of_frame_under_ncu") if tc else None,
                        "achieved_over_whole_graph_step": (gf / 1e3) / (serial_ms / opt.steps / 1e3),
                        "share_note": "the per-family times come from an EAGER instrumented pass (events around every C-ABI call; the GPU is parked "
                                      "on a spin kernel while the host enqueues the frame, so the intervals hold device time only) and are upper "
                                      "bounds of the in-graph times (no overlap between consecutive kernels): their sum can exceed the graph step; `achieved_over_whole_graph_step` = conv "
                                      "FLOPs / the whole captured step (a lower bound of the kernel's own rate)",
                        "hbm": {"achieved": (mb / 1e3) / (ms / 1e3) if ms > 0 else None, "peak": hbm_peak, "unit": "GB/s",
                                "frac": ((mb / 1e3) / (ms / 1e3)) / hbm_peak if ms > 0 else None,
                                "note": "ALGORITHMIC conv bytes (each layer's input + weights + output + residual, once) / live launch time"},
                        "kernels": [dict(name=k, bound=("tensor" if (v["tflops"] and k.startswith("conv")) else "hbm"), **v)
                                    for k, v in sorted(kernels.items(), key=lambda kv: -kv[1]["ms_per_frame"])]}
            for rec in roofline["kernels"]:
                nb = tj.get("per_family_dram_bytes_per_frame", {}).get(rec["name"]) if tj else None
                if nb:
                    rec["ncu_dram_mb_per_frame"] = nb / 1e6
        cpu = parity = eager_ref = None
        ref_out = None
        if not opt.no_cpu_baseline and world == 1:
            try:
                cores = pick_host_threads()
                refw = ReferenceWorkload(wl_name, n_agents).build("cpu")
                refw.set_state_dict({k: v.cpu() for k, v in sd.items()})
                ref_out, tv, tn = refw.frame(scenes[1])
                what = ("UNMODIFIED reference modules (oracle/_ref)" if refw.kind == "reference" else "oracle port") + \
                    ", CPU fp32, voxeliser = restated C"
                cpu = {"value": 1.0 / (tv + tn), "unit": "frames/s", "cores": cores, "kind": refw.kind,
                       "sample": f"1 whole frame ({n_agents} agents), no warm-up: voxelize {tv*1e3:.0f} ms (restated C, 1 thread) + "
                                 f"network {tn*1e3:.0f} ms ({what.split(',')[0]}, PyTorch-CPU fp32, {cores} threads chosen by a conv "
                                 f"micro-calibration)"}
                with torch.no_grad():
                    gout = frame_dev(1, eager=True)
                    torch.cuda.synchronize()
                parity = parity_record(gout, ref_out, opt.precision, what + f"; full-size frame (scene 1 of this run, {n_agents} agents)")
                if not parity["pass"]:
                    rc = 3
            except NotImplementedError as e:
                cpu = {"unavailable": str(e)}
        if not opt.no_eager_ref and world == 1 and wl_name in ("c1", "c2", "c5"):
            try:
                eager_ref = cuda_eager_leg(wl_name, n_agents, scenes, dev, ref_out)
            except Exception as e:
                eager_ref = {"error": repr(e)[:300]}
        graphed = fg is not None or getattr(wl, "graph", None) is not None
        secondary = None
        e2e_mode = (f"FramePipeline(depth={opt.pipeline_depth}): captured frames in flight; copy-in, copy-out and two alternating compute streams" if pipe is not None
                    else "single stream: H2D -> frame -> D2H")
        if world == 1 and wl_name == "c2" and not opt.no_secondary:
            secondary = {}
            fg = pipe = None                  # release the captured graphs' pools before building the other workloads
            torch.cuda.empty_cache()
            for name in ("c1", "c3", "c4"):
                try:
                    secondary[name] = run_secondary_workload(name, "bf16" if name == "c4" else opt.precision, dev, peaks, opt.steps)
                except Exception as e:
                    import traceback
                    sys.stderr.write(traceback.format_exc())
                    secondary[name] = {"error": repr(e)[:300]}
        par_text = ("scene-replicas (1 scene stream per GPU, no collective) for `value`; `agent_sharded` = agents sharded over ranks + "
                    "1 NCCL all-gather of the BEV pyramids")
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world,
                "steps": opt.steps, "warmup": opt.warmup, "ms_per_step": total_ms / opt.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": {"tc32": "f32", "bf16": "bf16", "fp32": "f32"}[opt.precision],
                "data": "synthetic",
                "config": workload_config(wl_name, world, par_text, opt.precision),
                "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "mode": e2e_mode, "single_stream_value_rank0": e2e_serial},
                "parity": parity, "cuda_eager_reference": eager_ref, "agent_sharded": sharded,
                "latency": {"frames_in_flight_for_value": inflight, "single_frame_ms": serial_ms / opt.steps,
                            "frames_per_s_one_frame_in_flight": frames / (serial_ms / 1e3),
                            "note": "`value` overlaps consecutive captured frames on separate streams; this is the same K frames replayed strictly one after the other on one stream"},
                "postprocess": post, "other_workloads": secondary,
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
                "gflop_per_frame": frame_flops(n_agents) / 1e9 if is_pyramid_lidar else None}
        if graphed and inflight > 1:
            line["config"]["launch"] = (f"one CUDA graph replay per frame, {inflight} captured frames in flight on {inflight} streams "
                                        "(`latency` = one frame at a time); per-kernel roofline numbers come from an eager, event-instrumented pass")
        if not graphed:
            line["config"]["launch"] = "eager launches, one stream (no CUDA graph: --no-graph or the capture failed, see stderr)"
        if dumped is not None:
            write_outputs(dumped, opt.dump_outputs)
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()
    if rc:
        sys.stderr.write("[bench] PARITY FAILURE: see the `parity` key of the JSON line\n")
        sys.exit(rc)


def cuda_eager_leg(wl_name, n_agents, scenes, dev, ref_cpu_out):
    """The unmodified reference modules on the GPU through stock PyTorch/cuDNN eager: the practical bar (SURVEY 8d last row)."""
    import torch
    from oracle import ref_runner
    if not ref_runner.available():
        return {"unavailable": "oracle/_ref not present (python -m oracle.build_ref)"}
    with contextlib.redirect_stdout(sys.stderr):
        if wl_name == "c1":
            m, _ = ref_runner.build_model("point_pillar", wcfg.c1_args(), dev)
            data, _ = ref_runner.c1_data(scenes[1]["clouds"][0], dev)
        else:
            m, _ = ref_runner.build_model("heter_pyramid_collab", wcfg.c2_args(), dev)
            data, _ = ref_runner.c2_data(scenes[1], n_agents, dev)
    rec = {"protocol": "opencood/tools/profiler/params_calc.py:48-79: 50 warm-up + 200 timed forward calls between CUDA events; "
                       "inputs = CPU-voxelised tensors already on the device (the reference voxelises in DataLoader workers); "
                       "cudnn.benchmark on", "kind": "UNMODIFIED reference modules (oracle/_ref) .cuda(), PyTorch eager"}
    ms32, out32 = ref_runner.time_cuda_eager(m, data, 50, 200, allow_tf32=False)
    rec["fp32_ms"] = ms32
    mstf, _ = ref_runner.time_cuda_eager(m, data, 50, 200, allow_tf32=True)
    rec["tf32_ms"] = mstf
    try:
        msbf, _ = ref_runner.time_cuda_eager(m, data, 20, 100, allow_tf32=True, autocast_bf16=True)
        rec["bf16_autocast_ms"] = msbf
    except Exception as e:
        rec["bf16_autocast_ms"] = None
        rec["bf16_autocast_note"] = repr(e)[:120]
    if ref_cpu_out is not None:
        rec["fp32_vs_cpu_reference_max_abs"] = {k: float((out32[k].float().cpu() - ref_cpu_out[k]).abs().max()) for k in HEADS if k in out32}

        def rel(o):
            return max(float((o[k].float().cpu() - ref_cpu_out[k]).abs().max()) / max(float(ref_cpu_out[k].abs().max()), 1.0)
                       for k in HEADS if k in o)
        # how far stock PyTorch's own reduced-precision modes are from the fp32 CPU reference on this frame (context for `parity`)
        try:
            _, otf = ref_runner.time_cuda_eager(m, data, 1, 1, allow_tf32=True)
            rec["tf32_max_rel_err_vs_cpu_fp32"] = rel(otf)
            _, obf = ref_runner.time_cuda_eager(m, data, 1, 1, allow_tf32=True, autocast_bf16=True)
            rec["bf16_autocast_max_rel_err_vs_cpu_fp32"] = rel(obf)
        except Exception as e:
            rec["reduced_precision_err_note"] = repr(e)[:120]
    del m
    torch.cuda.empty_cache()
    return rec


def postprocess_leg(wl, frame_dev):
    import torch
    try:
        import math
        from heal_b200.data_utils.post_processor import build_postprocessor
        args = wl.args
        rng = list(args["lidar_range"])
        vs = args["m1"]["encoder_args"]["voxel_size"]
        pcfg = {"core_method": "VoxelPostprocessor", "gt_range": rng, "order": "hwl", "nms_thresh": 0.15,
                "anchor_args": {"cav_lidar_range": rng, "l": 3.9, "w": 1.6, "h": 1.56, "r": [0, 90], "feature_stride": 2, "num": 2,
                                "vw": vs[0], "vh": vs[1], "W": math.ceil((rng[3] - rng[0]) / vs[0]),
                                "H": math.ceil((rng[4] - rng[1]) / vs[1])},
                "target_args": {"score_threshold": 0.2}, "dir_args": args["dir_args"]}
        pp = build_postprocessor(pcfg, train=False)
        out = frame_dev(0, eager=True)
        cav = {"transformation_matrix": torch.eye(4), "anchor_box": torch.from_numpy(pp.generate_anchor_box())}
        heads = {k: out[k] for k in HEADS}
        buf = pp._decode_one(cav, heads)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            pp._decode_one(cav, heads)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            pp._decode_one(cav, heads)
        g.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        st = buf.stats.cpu().tolist()
        return {"us_per_frame": a.elapsed_time(b) * 50.0, "above_threshold": st[0], "after_filters": st[1],
                "boxes_out": int(buf.count.item()),
                "note": "heal_box_decode_nms on the frame's heads (random-init weights: far more candidates than a trained model "
                        "yields), captured graph, device time, not part of `value` / `e2e`"}
    except Exception as e:      # informational only
        return {"error": repr(e)[:200]}


def agent_sharded_leg(opt, rank, world, dev, peaks):
    """One scene, agents sharded over the ranks (heal_b200.parallel.AgentShardedFrame): latency of the whole frame as the max over
    ranks of one CUDA-event interval, the all-gather's own time / bytes / GB/s, and rank 0's single-GPU latency of the same scene."""
    import torch
    import torch.distributed as dist
    from heal_b200 import parallel
    n_agents = 8 if world >= 8 else 5
    wname = "c5" if n_agents == 8 else "c2"
    scenes = build_scenes(wname, 4, n_agents, seed0=500)              # the SAME scenes on every rank
    wl = GpuWorkload(wname, opt.precision, dev, n_agents=n_agents, scenes=scenes)
    steps = opt.steps
    with torch.no_grad():
        sf = parallel.AgentShardedFrame(wl.model, n_agents, rank, world, wl.cap, scenes[0]["pairwise"].shape, device=dev,
                                        comm=os.environ.get("HEAL_SHARD_COMM", "auto"))
        for i in range(3):
            sf.load_scene(wl.devin[i % 4]["points"], scenes[i % 4]["offsets"], wl.devin[i % 4]["pairwise"])
            sf.replay()
        torch.cuda.synchronize()
        dist.barrier()

        def step(i):
            t = wl.devin[i % 4]
            sf.load_scene(t["points"], scenes[i % 4]["offsets"], t["pairwise"])
            sf.replay()
        ms = time_frames(step, steps, lambda: (dist.barrier(), torch.cuda.synchronize()))
        # end to end: pinned host clouds of MY agents -> H2D -> frame -> D2H of the heads (every rank holds the result)
        oh = {}

        def step_host(i):
            h = wl.host[i % 4]
            sf.load_scene(h["points"], scenes[i % 4]["offsets"], h["pairwise"])
            out = sf.replay()
            for k in HEADS:
                if k not in oh:
                    oh[k] = torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory()
                oh[k].copy_(out[k], non_blocking=True)
        for i in range(2):
            step_host(i)
        ms_e2e = time_frames(step_host, steps, lambda: (dist.barrier(), torch.cuda.synchronize()))
        # the collective alone (same buffers), and the single-GPU latency of the same scene on rank 0
        ag = sf.time_allgather(20)
        out_sh = {k: sf.out[k].clone() for k in HEADS}
        ref_ms, equal = None, None
        if rank == 0:
            from heal_b200.graph import FrameGraph
            fg1 = FrameGraph(wl.model, n_agents, wl.cap, scenes[0]["pairwise"].shape)
            t = wl.devin[(steps - 1) % 4]

            def one(i):
                t2 = wl.devin[i % 4]
                fg1.load(t2["points"], t2["offsets"], t2["pairwise"])
                fg1.replay()
            for i in range(3):
                one(i)
            ref_ms = time_frames(one, steps, torch.cuda.synchronize) / steps
            fg1.load(t["points"], t["offsets"], t["pairwise"])
            o1 = fg1.replay()
            torch.cuda.synchronize()
            equal = {k: float((o1[k] - out_sh[k]).abs().max()) for k in HEADS}
    tt = torch.tensor([ms, ms_e2e, ag["ms"]], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, ms_e2e, ag_ms = tt.tolist()
    lat = ms / steps
    recv = ag["bytes_per_rank"] * (world - 1)
    return {"scene": wcfg.WORKLOADS[wname]["title"], "agents": n_agents, "ranks": world, "plan": sf.plan,
            "frame_ms": lat, "frames_per_s": 1e3 / lat, "e2e_frames_per_s": steps / (ms_e2e / 1e3),
            "single_gpu_frame_ms_rank0": ref_ms, "speedup_vs_single_gpu": (ref_ms / lat) if ref_ms else None,
            "max_abs_diff_vs_single_gpu": equal,
            "allgather": {"comm": sf.comm, "ms": ag_ms, "bytes_per_rank": ag["bytes_per_rank"], "bytes_received_per_rank": recv,
                          "gbs_received_per_rank": recv / 1e9 / (ag_ms / 1e3) if ag_ms > 0 else None,
                          "exchanges_per_frame": sf.exchanges_per_frame, "nccl_collectives_per_frame": sf.collectives_per_frame,
                          "note": "exchange of the packed per-agent BEV pyramids through the symmetric buffer, timed ALONE (no compute to "
                                  "overlap with) with CUDA events, max over ranks: comm='p2p' = heal_p2p_push of every level to all peers "
                                  "over NVLink + one flag barrier (inside the frame the pushes run on a side stream under the next "
                                  "level's convolutions); comm='nccl' = one in-place ncclAllGather.  `bytes_received` = (ranks-1) x message"},
            "tail": sf.tail_mode, "graph": True, "kernels_per_replay": sf.kernels_per_replay}


if __name__ == "__main__":
    main()
