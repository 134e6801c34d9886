#!/usr/bin/env python
"""bench.py - decoder frames/s of the wavelet-monodepth hot path on N B200s (contract: see the task brief).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the sparse wavelet decoder (SparseDepthWaveProgressiveDecoder semantics,
thresh_ratio 0.05) over one batch of synthetic encoder features.  Headline workload (BASELINE.json
north_star / configs[2],[4]): ResNet50 pyramid, 1024x320, 32 frames per GPU (weak scaling: the global batch
is 32*N, batch-sharded, one NCCL all-gather of the full-resolution depth tensor per step).  The secondary
workload of the metric (ResNet18 640x192, 16 frames/GPU, configs[1]) is reported under "also".

JSON keys beyond the base contract:
  value     frames/s with features resident in HBM (NCHW fp32, as an encoder leaves them), device-timed
  e2e       frames/s through the same public call with HOST (pinned) features: H2D of every step's inputs
            (double-buffered on a copy stream) and D2H of the step's depth output inside the timed region
  roofline  dominant kernel (by summed device time) : algorithmic bytes / CUDA-event time vs measured HBM peak,
            plus its FLOP rate; roofline_kernels lists the same for every libwmd kernel
  cpu_baseline  the oracle's port of the reference's CPU path timed on this box's host cores (bounded sample)
`--impl reference` times that CPU path as its own arm (rank 0 only under torchrun).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np   # noqa: E402
import torch         # noqa: E402

from wavelet_monodepth_b200 import synth   # noqa: E402

WORKLOADS = {
    "kitti_r50_1024x320_bs32": dict(ch=synth.RESNET50_CH, height=320, width=1024, per_gpu_batch=32),
    "kitti_r18_640x192_bs16": dict(ch=synth.RESNET18_CH, height=192, width=640, per_gpu_batch=16),
}
NYU = dict(name="nyu_d161_640x480_bs8", ch=synth.DENSENET161_CH, height=480, width=640, per_gpu_batch=8, thresh=0.1,
           heads=["wave1.conv.", "wave2.conv.", "wave3.conv."], param_seed=11, feat_seed=2000)   # configs[3]
MAIN = "kitti_r50_1024x320_bs32"
ALSO = "kitti_r18_640x192_bs16"
HEAD_KEYS = synth.KITTI_HEAD_KEYS                                                # +/- coefficient heads' 3x3 stage
SYNTH = synth.BENCH_SYNTH
THRESH = 0.05
METRIC, UNIT = "decoder_frames_per_sec", "frames/s"
FP32_SIMT_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FMA lanes x 2 flop x max SM clock
DUMP_BYTES = 64 * 1000 * 1000                                # --dump-outputs: all files together


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def synth_params(module):
    return synth.bench_kitti_params(module)


def synth_features(wl, n, first_sample, pin):
    return synth.bench_kitti_features(n, wl["height"], wl["width"], wl["ch"], first_sample, pin)


def measured_peaks():
    """(HBM GB/s, bf16 dense TFLOP/s burst, source, bf16 dense TFLOP/s sustained or None)."""
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            sus = d.get("bf16_tflops_sustained")
            return (float(d["hbm_gbs"]), float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json)",
                    float(sus) if sus else None)
        except Exception:
            pass
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md 6.65 TB/s, 1.59 PFLOP/s)", None


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.rows, self.proc = [], None
        try:
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            sel = "GPU-" + uuid if not uuid.startswith("GPU-") else uuid
        except Exception:
            sel = str(device_index)
        self.cmd = ["nvidia-smi", "-i", sel, "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"]

    def start(self):
        try:
            self.proc = subprocess.Popen(self.cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        threading.Thread(target=self._read, daemon=True).start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        hot = sorted(sm)[len(sm) // 2:] if sm else []        # upper half = samples under load
        return {"sm_mhz": float(np.median(hot)) if hot else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ roofline accounting
def _as_int(v, default):
    if v is None:
        return int(default)
    if torch.is_tensor(v):
        return int(v.reshape(-1)[0].item())
    return int(v)


def account(name, info):
    """(algorithmic bytes, flops) of one launch - SURVEY 8(d) / DESIGN.md 'algorithmic bytes'."""
    if name in ("conv_rows", "conv_rows_tc"):
        n, h, w, taps, c0, c1, cout = (info[k] for k in ("n", "h", "w", "taps", "c0", "c1", "cout"))
        total = n * h * w
        m_out = min(_as_int(info["count"], total), info["max_rows"])
        m0 = _as_int(info["m_in0"], n * (h >> info["shift0"]) * (w >> info["shift0"]) if info["count"] is None else m_out)
        m1 = _as_int(info["m_in1"], total) if c1 else 0
        by = 4 * (m0 * c0 + m1 * c1 + m_out * cout) + 4 * (taps * (c0 + c1) * cout + cout)
        by += total if info["count"] is not None else 0                 # 1-byte gate / list traffic
        return by, 2 * taps * (c0 + c1) * cout * m_out
    if name == "head_gather":
        n, h, w, g, cout = (info[k] for k in ("n", "h", "w", "groups", "cout"))
        m = min(_as_int(info["count"], n * h * w), info["max_rows"])
        return 4 * m * (9 * g + cout) + (n * h * w if info["count"] is not None else 0), 9 * g * m
    if name == "head_mlp":
        m = min(_as_int(info["count"], info["max_rows"]), info["max_rows"])
        c, n1, nz = info["c"], info["n1"], info["nz"]
        return 4 * m * (c + 56) + 4 * (n1 * c + nz * n1 + n1), 2 * m * (c * n1 + n1 * nz)
    if name == "head_conv3x3":
        n, h, w, c, cout = (info[k] for k in ("n", "h", "w", "c", "cout"))
        m = min(_as_int(info["count"], n * h * w), info["max_rows"])
        heads = 2 if info["dual"] else 1
        return 4 * (m * c * heads + m * cout) + 4 * heads * (9 * c * cout + cout), 2 * 9 * c * cout * m * heads
    if name == "head_idwt":
        px = info["n"] * info["h"] * info["w"]
        m = int(info["mask"].sum().item()) if info["mask"] is not None else px
        # ll + mask in, yh + reconstruction + disp out (+ two epilogue planes), 9 x 6 tap products per active pixel
        return px * (4 + (1 if info["mask"] is not None else 0) + 12 + 16 + 16 + (32 if info["epi"] else 0)) + m * 9 * 24, 9 * 6 * m + 14 * px
    if name == "idwt_haar":
        px = info["n"] * info["c"] * info["h"] * info["w"]
        return (32 + (16 if info["disp"] else 0)) * px, 14 * px
    if name == "idwt_bilinear":
        return 16 * info["n"] * info["c"] * info["h"] * info["w"] + 4 * info["n"] * info["c"] * info["fh"] * info["fw"], 0
    if name == "dwt_haar":
        return 8 * info["n"] * info["c"] * info["h"] * info["w"], 0
    if name == "range_thresh":
        return 4 * info["n"] * info["per"], 0
    if name == "level_masks":
        px = info["n"] * info["h"] * info["w"]
        return (12 if info["thresh"] else 0) * px + 15 * px, 0
    if name == "compact_mask":
        px = info["n"] * info["h"] * info["w"]
        m = _as_int(info["offsets"][-1:], px)
        return px + (4 * px if info["idxmap"] else 0) + (4 * m if info["pixels"] else 0), 0
    if name == "gate_map":
        return 9 * info["count"], 0
    if name == "gather_rows_list":
        m = min(_as_int(info["count"], info["max_rows"]), info["max_rows"])
        return 8 * info["c"] * m + 4 * m, 0
    if name in ("nchw_to_rows", "rows_to_nchw"):
        px = _as_int(info.get("marked"), info["n"] * info["hw"])      # gated move: only the marked pixels' rows
        return 8 * info["c"] * px + (info["n"] * info["hw"] if info.get("marked") is not None else 0), 0
    return 0, 0


def conv_layer_table(records, peak_gbs, tf32_peak, steps):
    """One line per gather-GEMM launch of a step (mean over the profiled steps): shape, active rows, time, rates.
    tensor_frac = algorithmic (fp32-equivalent) flops / tf32 peak; tensor_frac_executed counts the three tf32 MMAs
    each fp32 product costs."""
    convs = [(name, ms, info) for name, ms, info in records if name in ("conv_rows", "conv_rows_tc")]
    per_step = len(convs) // max(steps, 1)
    if per_step == 0 or per_step * steps != len(convs):
        return []
    table = []
    for k in range(per_step):
        same = convs[k::per_step]
        name, _, info = same[0]
        ms = sum(m for _, m, _ in same) / len(same)
        by, fl = account(name, info)
        rows = min(_as_int(info["count"], info["n"] * info["h"] * info["w"]), info["max_rows"])
        tf = fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        line = {"engine": ("tcgen05_f16x3" if info.get("f16") else "tcgen05_3xtf32") if name == "conv_rows_tc" else "fp32_fma",
                "taps": info["taps"],
                "cin": [info["c0"], info["c1"]], "cout": info["cout"], "grid": [info["n"], info["h"], info["w"]],
                "rows": rows, "us": round(1e3 * ms, 1), "fp32_eq_tflops": round(tf, 1),
                "hbm_frac": round(by / (ms * 1e-3) / 1e9 / peak_gbs, 3) if ms > 0 else 0.0}
        if name == "conv_rows_tc":
            line["tensor_frac"] = round(tf / tf32_peak, 3)
            line["tensor_frac_executed"] = round(3.0 * tf / tf32_peak, 3)
        else:
            line["fma_frac"] = round(tf / FP32_SIMT_PEAK_TFLOPS, 3)
        table.append(line)
    return table


def roofline_from(records, peak_gbs, peak_tf, peak_src, steps, peak_tf_sustained=None, tf32_peak=None):
    """roofline object of the dominant kernel + per-kernel table.

    Tensor-bound kernel: `achieved` = ALGORITHMIC flops (2 * taps * Cin * Cout * M_out, SURVEY 8d) / CUDA-event time and
    `frac` = achieved / tf32 peak.  The kernel executes three tf32 MMAs per fp32 product (3xTF32, needed for the 1e-4 /
    exact-mask parity bar): `frac_executed_3xtf32` = 3 * achieved / peak is the fraction of the tensor pipe it keeps busy.
    tf32 peak: measured in this process (cuBLAS TF32 GEMM 8192^3, best of 10); MEASURED_PEAKS.json's bf16 figure / 2 is
    listed beside it."""
    agg = {}
    for name, ms, info in records:
        by, fl = account(name, info)
        a = agg.setdefault(name, dict(ms=0.0, bytes=0, flops=0, launches=0))
        a["ms"] += ms; a["bytes"] += by; a["flops"] += fl; a["launches"] += 1
    total_ms = sum(a["ms"] for a in agg.values()) or 1.0
    out = {}
    for name, a in agg.items():
        gbs = a["bytes"] / (a["ms"] * 1e-3) / 1e9 if a["ms"] > 0 else 0.0
        out[name] = {
            "bound": "hbm", "achieved": round(gbs, 1), "peak": peak_gbs, "unit": "GB/s", "frac": round(gbs / peak_gbs, 4),
            "traffic": None, "avg_launch_us": round(1e3 * a["ms"] / a["launches"], 2),
            "bytes_per_launch": int(a["bytes"] / a["launches"]), "launches_per_step": a["launches"] // steps,
            "share_of_kernel_time": round(a["ms"] / total_ms, 4),
            "tflops": round(a["flops"] / (a["ms"] * 1e-3) / 1e12, 2) if a["ms"] > 0 else 0.0,
        }
    dom = max(agg, key=lambda k: agg[k]["ms"])
    hbm_view = dict(out[dom])
    tf32 = tf32_peak if tf32_peak else peak_tf / 2.0
    f16_form = any(n == "conv_rows_tc" and i.get("f16") for n, _, i in records)
    if f16_form:                       # WMD_CONV_PRECISION=f16x3: the MMAs run at the fp16 rate, so that is the peak
        tf32, tf32_peak = peak_tf, None
    if dom == "conv_rows_tc":
        alg = hbm_view["tflops"]
        main = {"bound": "tensor", "achieved": round(alg, 1), "peak": round(tf32, 1), "unit": "TFLOP/s",
                "frac": round(alg / tf32, 4), "traffic": None, "kernel": dom,
                "frac_executed_3xtf32": round(3.0 * alg / tf32, 4),
                "executed_tf32_tflops": round(3.0 * alg, 1),
                "avg_launch_us": hbm_view["avg_launch_us"],
                "launches_per_step": hbm_view["launches_per_step"], "share_of_kernel_time": hbm_view["share_of_kernel_time"],
                "bytes_per_launch": hbm_view["bytes_per_launch"],
                "hbm_view": {"achieved_gbs": hbm_view["achieved"], "peak_gbs": peak_gbs, "frac": hbm_view["frac"]},
                "peak_alternatives": {"tf32_measured_here_tflops": round(tf32_peak, 1) if tf32_peak else None,
                                      "bf16_burst_over_2": round(peak_tf / 2.0, 1),
                                      "bf16_sustained_over_2": round(peak_tf_sustained / 2.0, 1) if peak_tf_sustained else None},
                "peak_source": ("measured in this run: cuBLAS TF32 GEMM 8192^3, best of 20 (burst; each launch is timed alone "
                                "between two events)" if tf32_peak else peak_src + ": bf16_tflops / 2"),
                "operand_form": "f16x3 (fp16 pairs, opt-in)" if f16_form else "tf32x3",
                "note": "achieved = algorithmic fp32-equivalent flops (2*taps*Cin*Cout*M_out) / event time. tcgen05.mma.kind::tf32, "
                        "3 MMAs per fp32 product (hi*hi + hi*lo + lo*hi), fp32 accumulation in TMEM drained every 1024 of K; "
                        "per-layer figures in conv_layers, DESIGN.md 4"}
    else:
        main = dict(hbm_view)
        main.update(kernel=dom, peak_source=peak_src,
                    note="fp32 SIMT kernel; tflops/fp32_frac give the FMA-roof view (%.1f TFLOP/s nominal)" % FP32_SIMT_PEAK_TFLOPS,
                    fp32_frac=round(main["tflops"] / FP32_SIMT_PEAK_TFLOPS, 4))
    traffic_file = os.path.join(REPO, "profiles", "ncu_traffic.json")
    if os.path.exists(traffic_file):
        try:
            tr = json.load(open(traffic_file))
            main["traffic"] = tr.get(dom)
            for name in out:
                if tr.get(name) is not None:
                    out[name]["traffic"] = tr[name]
        except Exception:
            pass
    # whole step against the HBM roof (north_star: "fraction of the HBM roofline" for the fused decoder): the summed
    # algorithmic bytes of every launch of a step over the summed kernel time
    step_bytes = sum(a["bytes"] for a in agg.values()) / max(steps, 1)
    step_flops = sum(a["flops"] for a in agg.values()) / max(steps, 1)
    step_ms = total_ms / max(steps, 1)
    main["hbm_frac_step"] = round(step_bytes / (step_ms * 1e-3) / 1e9 / peak_gbs, 4)
    main["hbm_gbs_step"] = round(step_bytes / (step_ms * 1e-3) / 1e9, 1)
    for key, kname in (("idwt", "idwt_haar"), ("idwt_fused", "head_idwt")):
        if kname in out:
            main[key] = {"kernel": kname, "achieved_gbs": out[kname]["achieved"], "peak_gbs": peak_gbs, "frac": out[kname]["frac"],
                         "avg_launch_us": out[kname]["avg_launch_us"], "launches_per_step": out[kname]["launches_per_step"],
                         "traffic": out[kname]["traffic"]}
    main["step_view"] = {"algorithmic_bytes_per_step": int(step_bytes), "kernel_ms_per_step": round(step_ms, 3),
                         "hbm_gbs": round(step_bytes / (step_ms * 1e-3) / 1e9, 1),
                         "hbm_frac": round(step_bytes / (step_ms * 1e-3) / 1e9 / peak_gbs, 4),
                         "fp32_eq_tflops": round(step_flops / (step_ms * 1e-3) / 1e12, 1),
                         "hbm_floor_ms": round(step_bytes / (peak_gbs * 1e9) * 1e3, 3),
                         "tf32x3_floor_ms": round(3.0 * step_flops / (tf32 * 1e12) * 1e3, 3),
                         "note": "north_star target '>= 60 % of the HBM roofline on the fused decoder' presumes an HBM-bound "
                                 "decoder; at fp32-faithful precision (3 tf32 MMAs per product) the tensor-pipe floor is above "
                                 "the HBM floor (both listed), so hbm_frac_step cannot reach 0.6 with exact masks"}
    return main, out


# ------------------------------------------------------------------------------------------ CPU arm (oracle port of the reference)
_CPU_PARAMS = {}


def _affinity_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _cpu_setup(wl_name):
    from wavelet_monodepth_b200.kitti_decoders import SparseDepthWaveProgressiveDecoder
    wl = WORKLOADS[wl_name]
    if wl_name not in _CPU_PARAMS:
        _CPU_PARAMS[wl_name] = synth_params(SparseDepthWaveProgressiveDecoder(np.array(wl["ch"])))
    return wl, _CPU_PARAMS[wl_name]


def _cpu_frame(wl, sd, f, batch=None, on_frame=None):
    from oracle import kitti as okitti                     # allowed here: cpu_baseline / --impl reference legs only
    b = f % wl["per_gpu_batch"]
    if batch is not None:                                  # frame b of the step's own (host) feature batch
        feats = [t[b:b + 1].contiguous() for t in batch]
    else:
        feats = synth_features(wl, 1, b, pin=False)
    t0 = time.perf_counter()
    with torch.no_grad():
        ref = okitti.sparse_forward(sd, feats, THRESH)
    dt = time.perf_counter() - t0
    if on_frame is not None:                               # parity block: outside the timed span
        on_frame(b, ref)
    return dt


def _cpu_oracle_frame(wl_name, feats, thresh):
    """Oracle outputs of one frame at `thresh` (threshold sweep's op-count / parity check)."""
    from oracle import kitti as okitti
    _, sd = _cpu_setup(wl_name)
    with torch.no_grad():
        return okitti.sparse_forward(sd, [t.contiguous() for t in feats], thresh)


def cpu_pick_threads(wl_name):
    """The path is thousands of small ATen ops: more threads is not faster.  Probe a few intra-op thread counts up
    to every core this process may use and keep the fastest (one frame each, after one warm-up)."""
    if "threads" in _CPU_PARAMS:
        return _CPU_PARAMS["threads"]
    wl, sd = _cpu_setup(wl_name)
    cores = _affinity_cores()
    cands = sorted({c for c in (4, 8, 16, 32, cores) if c <= cores})
    torch.set_num_threads(cands[0])
    _cpu_frame(wl, sd, 0)
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        t = _cpu_frame(wl, sd, 1)
        log("[cpu arm] %d threads: %.3f s/frame" % (c, t))
        if best_t is None or t < best_t:
            best, best_t = c, t
        if t > 4 * best_t:
            break
    torch.set_num_threads(best)
    _CPU_PARAMS["threads"] = best
    return best


def cpu_frames_per_sec(wl_name, frames, budget_s=20.0, first_frame=0, batch=None, on_frame=None):
    """Times oracle.kitti.sparse_forward (the reference's batch-1 sparse path, restated) on the host cores:
    up to `frames` frames, stopping early once `budget_s` seconds of CPU work are spent.  `batch`: host feature
    tensors to take the frames from (the GPU arm's own step inputs); otherwise frames are generated one by one."""
    wl, sd = _cpu_setup(wl_name)
    torch.set_num_threads(cpu_pick_threads(wl_name))
    times = []
    for f in range(frames):
        times.append(_cpu_frame(wl, sd, first_frame + f, batch, on_frame))
        if sum(times) >= budget_s:
            break
    return len(times) / sum(times), times


def workload_config(wl_name, world, thresh=None):
    """Static description of the measured workload: identical in the native and the reference arm (the driver compares
    the two arms' `config`).  Anything measured (mask densities, op counts) or arm-specific goes elsewhere."""
    wl = WORKLOADS[wl_name]
    return {
        "workload": wl_name, "global_batch": wl["per_gpu_batch"] * world, "per_gpu_batch": wl["per_gpu_batch"],
        "encoder": "%s pyramid %s" % ("ResNet50" if wl["ch"] == synth.RESNET50_CH else "ResNet18", list(wl["ch"])),
        "resolution": "%dx%d" % (wl["width"], wl["height"]),
        "thresh_ratio": THRESH if thresh is None else thresh,
        "decoder": "SparseDepthWaveProgressiveDecoder (levels 3,2,1 sparse)",
        "parallelism": "dp%d batch-sharded, one all-gather of disp0" % world,
        "l2": "inputs larger than L2: %.2f GB of features read per step per GPU"
              % (sum(4 * c * (wl["height"] // (2 << k)) * (wl["width"] // (2 << k)) for k, c in enumerate(wl["ch"]))
                 * wl["per_gpu_batch"] / 1e9),
        "weights": "seeded random init, high-pass coefficient heads x%.0f (synth.py)" % SYNTH["head_gain"],
        "features": "seeded blocky maps, cell %d px, texture %.2f" % (SYNTH["cell"], SYNTH["texture"]),
    }


def run_reference_arm(args, rank):
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    frames_per_step = 16                                   # ~2 s of CPU work per step on the box's host cores
    cores = cpu_pick_threads(args.workload)
    per_step_budget = max(2.0, 150.0 / max(args.steps + args.warmup, 1))     # whole run stays within a few minutes
    for w in range(args.warmup):
        cpu_frames_per_sec(args.workload, 1, budget_s=per_step_budget, first_frame=w)
    t0 = time.perf_counter()
    done, spent = 0, 0.0
    for k in range(args.steps):
        _, times = cpu_frames_per_sec(args.workload, frames_per_step, budget_s=per_step_budget,
                                      first_frame=k * frames_per_step)
        done += len(times)
        spent += sum(times)
    wall = time.perf_counter() - t0
    fps = done / spent
    line = {
        "impl": "reference", "metric": METRIC, "value": round(fps, 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * spent / args.steps, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, world),
        "arm": {"frames_per_step": round(done / args.steps, 2), "wall_s": round(wall, 1),
                "note": "the reference is Python/PyTorch and cannot travel to the GPU box; this arm times the oracle's "
                        "torch-CPU port of its batch-1 sparse decoder (pinned bit-exact against the reference, "
                        "oracle/pin_against_reference.py; measured ~1.4x FASTER than the reference's own code in the "
                        "build container) on the host cores; each step is a bounded sample of the workload's frames"},
        "cpu_baseline": {"value": round(fps, 3), "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d frames in %d steps of %s, one frame at a time (reference asserts batch 1); "
                                   "intra-op threads chosen by probe out of %d usable cores"
                                   % (done, args.steps, args.workload, _affinity_cores())},
        "e2e": {"value": round(fps, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ native arm
class _Guard:
    """with _Guard(name, active, sink): a secondary section of the bench.  On one GPU an exception inside it is logged and
    recorded in `sink` instead of costing the headline line; with several ranks it propagates (a rank that skipped the
    section's collectives would hang the others)."""

    def __init__(self, name, active, sink):
        self.name, self.active, self.sink = name, active, sink

    def __enter__(self):
        return self

    def __exit__(self, et, ev, tb):
        if et is None or not self.active or not issubclass(et, Exception):
            return False
        log("[bench] section %s failed: %r" % (self.name, ev))
        self.sink[self.name] = repr(ev)[:300]
        return True


def time_device(step_fn, steps, warmup, dist, world, flush=None):
    """`steps` calls of step_fn between two CUDA events, barrier + synchronize on both sides, max over ranks.
    flush: called after the last step INSIDE the timed region (drains whatever the steps left in flight: the last
    step's op-count future and all-gather)."""
    for _ in range(warmup):
        step_fn()
    if flush:
        flush()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step_fn()
    if flush:
        flush()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def measure_tf32_peak(dev):
    """Dense TF32 tensor-core throughput of this GPU, measured the way MEASURED_PEAKS.json measures bf16: cuBLAS GEMM
    8192^3 (fp32 operands, allow_tf32), best of 20 after 10 warm-up launches, CUDA events."""
    was = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(10):                   # clocks ramp over the first launches
            torch.matmul(a, b)
        best = None
        for _ in range(20):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            t = e0.elapsed_time(e1)
            best = t if best is None or t < best else best
        del a, b
        torch.cuda.empty_cache()
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = was


class _Stepper:
    """One bench step = decoder replay (no host wait) + the rank's all-gather started asynchronously; the previous
    step's op count and gathered tensor are consumed while this one runs.  flush() drains the tail."""

    def __init__(self, run, gather, last):
        self.run, self.gather, self.last, self.pending = run, gather, last, []

    def _finish(self, item):
        fut, handle, out = item
        self.last["total_ops"] = fut.result()["total_ops"] if fut is not None else None
        self.last["ops_result"] = fut.result() if fut is not None else None
        if handle is not None:
            self.last["gathered"] = handle.wait()
        self.last["out"] = out

    def step(self):
        out = self.run()
        fut = out.get("total_ops")
        handle = self.gather.start(out[("disp", 0)]) if self.gather is not None else None
        self.pending.append((fut, handle, out))
        while len(self.pending) > 1:
            self._finish(self.pending.pop(0))

    def flush(self):
        while self.pending:
            self._finish(self.pending.pop(0))


def output_name(key):
    return "_".join(str(p) for p in key) if isinstance(key, tuple) else str(key)


def dump_outputs(out, ops_result, gathered, directory, budget_bytes=DUMP_BYTES):
    """Write one step's outputs as <directory>/<name>.npy: tensors in float32 (masks as 0 / 1), integer tensors and the
    op counts in float64.  When the whole set exceeds `budget_bytes`, the largest tensors are cut to a fixed sample of
    their flattened elements (positions drawn from a generator seeded by the output's name, sorted), so that two runs
    with the same arguments write files that compare element for element."""
    os.makedirs(directory, exist_ok=True)
    tensors = {output_name(k): v for k, v in out.items() if torch.is_tensor(v)}
    if gathered is not None:
        tensors["disp_0_gathered"] = gathered
    counts = {output_name(k): np.asarray(v, dtype=np.float64) for k, v in (ops_result or {}).items()}
    left = budget_bytes // 8 - sum(a.size for a in counts.values()) - 64 * (len(tensors) + len(counts))
    for name, a in counts.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    by_size = sorted(tensors, key=lambda n: tensors[n].numel())
    for i, name in enumerate(by_size):
        t = tensors[name]
        wide = t.dtype in (torch.int64, torch.int32, torch.float64)
        cap = left // (len(by_size) - i) * (1 if wide else 2)      # `left` counts 8-byte units
        flat = t.detach().reshape(-1)
        if flat.numel() > cap:
            pick = np.random.default_rng(zlib.crc32(name.encode())).choice(flat.numel(), cap, replace=False)
            flat = flat[torch.from_numpy(np.sort(pick)).to(flat.device)]
        left -= -(-flat.numel() // (1 if wide else 2))
        np.save(os.path.join(directory, name + ".npy"), flat.to(torch.float64 if wide else torch.float32).cpu().numpy()
                .reshape(t.shape if flat.numel() == t.numel() else (-1,)))


def run_native(args, rank, world, local_rank):
    import torch.distributed as dist
    from wavelet_monodepth_b200 import _lib, graphs, ops, shard
    from wavelet_monodepth_b200.kitti_decoders import SparseDepthWaveProgressiveDecoder

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    reserved_sms = 0
    if world > 1:
        # the persistent conv CTAs fill every SM's register file, so the previous step's all-gather kernel can only run in
        # the gaps between them.  WMD_RESERVED_SMS=n leaves n SMs to it and keeps NCCL to that many CTAs.  Off by default:
        # one sweep at 4 GPUs (10 steps) gave 4.09 / 3.92 / 4.09 ms per step for n = 0 / 4 / 8 against 3.90 for n = 0 in a
        # 20-step run - inside the noise, not enough measurements to switch it on
        reserved_sms = int(os.environ.get("WMD_RESERVED_SMS", "0"))
        if reserved_sms > 0:
            os.environ.setdefault("NCCL_MAX_CTAS", str(reserved_sms))
        dist.init_process_group("nccl", device_id=dev)
        _lib.load().wmd_conv_tc_set_reserved_sms(reserved_sms)
    peak_gbs, peak_tf, peak_src, peak_tf_sus = measured_peaks()
    tf32_peak = measure_tf32_peak(dev)
    section_errors = {}

    def setup(wl_name):
        wl = WORKLOADS[wl_name]
        n_local = wl["per_gpu_batch"]
        dec = SparseDepthWaveProgressiveDecoder(np.array(wl["ch"]))
        synth_params(dec)
        dec = dec.to(dev).eval()
        dec.count_ops = "async"            # total_ops via OpsFuture: the step never blocks the host (opsfuture.py)
        t0 = time.time()
        host = synth_features(wl, n_local, rank * n_local, pin=True)
        log("[rank %d] %s: synthetic features for %d frames in %.1fs" % (rank, wl_name, n_local, time.time() - t0))
        return wl, dec, host

    wl, dec, host = setup(args.workload)
    n_local, n_global = wl["per_gpu_batch"], wl["per_gpu_batch"] * world
    resident = [f.to(dev) for f in host]
    last = {}
    gather = shard.make_gather(n_global) if world > 1 else None

    # serving mode: the launches of one forward captured once in a CUDA graph bound to the resident feature tensors
    # (graphs.py); replay = the same kernels without the per-launch host cost.  --no-graph times the eager calls instead.
    use_graph = not args.no_graph
    graph = graphs.GraphedSparseDecoder(dec, resident, THRESH) if use_graph else None
    eager = _Stepper(lambda: dec(resident, THRESH), gather, last)
    main = _Stepper(graph.replay, gather, last) if use_graph else eager

    # ---- 1. device-resident throughput
    # clocks are sampled from before the warm-up to the end of the end-to-end pass: the two timed regions are only
    # tens of milliseconds long, nvidia-smi samples every 100 ms; the "under load" figure is the median of the upper half
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(args.warmup - 1, 0)):
        main.step()
    main.flush()
    l0 = _lib.launch_count()
    ms = time_device(main.step, args.steps, 1 if args.warmup else 0, dist, world, flush=main.flush)
    launches = _lib.launch_count() - l0
    launches -= (1 if args.warmup else 0) * (launches // (args.steps + (1 if args.warmup else 0)))
    if use_graph:
        launches = graph.launches * args.steps                       # kernel nodes replayed inside the timed region
    if args.dump_outputs and rank == 0:                              # the last timed step's outputs, before anything reuses them
        dump_outputs(last["out"], last["ops_result"], last.get("gathered"), args.dump_outputs)
    ms_eager = time_device(eager.step, args.steps, 1, dist, world, flush=eager.flush) if use_graph else ms
    value_eager = n_global * args.steps / (ms_eager * 1e-3)
    out = last["out"]
    dens = {s: round(float(out[("wavelet_mask", s)].float().mean()), 4) for s in (3, 2, 1, 0)}
    ops_per_frame = last["total_ops"] / n_local
    value = n_global * args.steps / (ms * 1e-3)
    # the step's outputs, kept on the host for the parity block of the cpu_baseline leg
    out_host = {k: v.cpu() for k, v in out.items() if torch.is_tensor(v)} if (rank == 0 and world == 1 and not args.no_cpu) else None
    if out_host is not None:
        out_host["total_ops_per_sample"] = last["ops_result"].get("total_ops_per_sample", [last["total_ops"]])

    # the collective alone (N > 1): K all-gathers of disp0 back to back, nothing else on the GPU
    allgather_ms = None
    if world > 1:
        solo = shard.make_gather(n_global)
        src = out[("disp", 0)]
        hs = []

        def ag_step():
            hs.append(solo.start(src))
            if len(hs) > 1:
                hs.pop(0).wait()

        allgather_ms = time_device(ag_step, args.steps, 2, dist, world, flush=lambda: [h.wait() for h in hs] and hs.clear()) / args.steps

    # ---- 1b. same step with the features handed over channels_last (what a channels_last cuDNN encoder leaves):
    # the decoder then uses them in place and the five NCHW->rows transposes disappear
    resident_cl = [f.contiguous(memory_format=torch.channels_last) for f in resident]
    graph_cl = graphs.GraphedSparseDecoder(dec, resident_cl, THRESH) if use_graph else None
    cl = _Stepper(graph_cl.replay if use_graph else (lambda: dec(resident_cl, THRESH)), gather, {})
    ms_cl = time_device(cl.step, args.steps, 2, dist, world, flush=cl.flush)
    value_cl = n_global * args.steps / (ms_cl * 1e-3)
    del graph_cl, resident_cl, cl
    torch.cuda.empty_cache()

    # ---- 1c. threshold sweep (BASELINE.json configs[2]: {0, 0.02, 0.05, 0.1} on one GPU; configs[4]: {0.05, 0.1} sharded)
    sweep = None
    if args.workload == MAIN and not args.no_sweep:
        sweep = []
        thr_list = (0.0, 0.02, 0.05, 0.1) if world == 1 else (0.05, 0.1)
        for thr in thr_list:
            with _Guard("sweep_%g" % thr, world == 1, section_errors):
                g = graphs.GraphedSparseDecoder(dec, resident, thr) if use_graph else None
                lst = {}
                st = _Stepper(g.replay if use_graph else (lambda thr=thr: dec(resident, thr)), gather, lst)
                ms_t = time_device(st.step, args.steps, 2, dist, world, flush=st.flush)
                o = lst["out"]
                entry = {"thresh_ratio": thr, "value": round(n_global * args.steps / (ms_t * 1e-3), 1), "unit": UNIT,
                         "ms_per_step": round(ms_t / args.steps, 3),
                         "wavelet_mask_density": {str(s_): round(float(o[("wavelet_mask", s_)].float().mean()), 4) for s_ in (3, 2, 1, 0)},
                         "total_ops_per_frame": lst["total_ops"] / n_local,
                         "frac_of_dense_ops": round(lst["total_ops"] / n_local / 17473692295, 4)}
                if rank == 0 and world == 1 and not args.no_cpu:
                    # frame 0 of the step against the oracle (the reference's counter and outputs for that frame)
                    from oracle import parity
                    ref0 = _cpu_oracle_frame(args.workload, [t[0:1] for t in host], thr)
                    got0 = parity.sample_of({**{k: v for k, v in o.items() if torch.is_tensor(v)},
                                             "total_ops_per_sample": lst["ops_result"]["total_ops_per_sample"]}, 0)
                    rep = parity.compare_kitti_sample(got0, ref0, thr)
                    entry["oracle_check_frame0"] = {"total_ops_equal": rep["total_ops_equal"], "max_rel_err": float("%.3e" % rep["max_rel_err"]),
                                                    "mask_hamming": sum(rep["mask_hamming"].values()), "failures": rep["failures"][:3]}
                sweep.append(entry)
                del g, st
                torch.cuda.empty_cache()

    # ---- 2. end to end: host features -> H2D (copy stream, double buffered) -> decode -> D2H of disp0
    # zero_copy = indices of skip maps that stay in pinned host memory and are read in place by the gated layout move
    # (only the rows under the level's upsample mask cross PCIe); the others are DMA-copied one step ahead.
    copy_stream = torch.cuda.Stream()
    disp_host = torch.empty((n_local, 1, wl["height"], wl["width"]), dtype=torch.float32).pin_memory()
    d2h_bytes = disp_host.numel() * 4 + 9 * (n_local + 1) * 4

    def run_e2e(zero_copy):
        dma = [k for k in range(len(host)) if k not in zero_copy]
        bufs = [[host[k] if k in zero_copy else torch.empty_like(host[k], device=dev) for k in range(len(host))]
                for _ in range(2)]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        state = {"i": 0}
        graphs_e2e = [graphs.GraphedSparseDecoder(dec, b, THRESH) for b in bufs] if use_graph else None
        lst = {}

        def enqueue_copy(slot):
            with torch.cuda.stream(copy_stream):
                for k in dma:
                    bufs[slot][k].copy_(host[k], non_blocking=True)
                ready[slot].record(copy_stream)

        def run():
            i = state["i"]
            slot = i % 2
            enqueue_copy(1 - slot)                                   # next step's inputs overlap this step's compute
            torch.cuda.current_stream().wait_event(ready[slot])
            o = graphs_e2e[slot].replay() if use_graph else dec(bufs[slot], THRESH)
            disp_host.copy_(o[("disp", 0)], non_blocking=True)       # the step's result back to the host
            copy_stream.wait_stream(torch.cuda.current_stream())     # slot is free for the copy after next
            state["i"] = i + 1
            return o

        st = _Stepper(run, gather, lst)
        enqueue_copy(0)
        ms_ = time_device(st.step, args.steps, 2, dist, world, flush=st.flush)
        o = lst["out"]
        h2d = sum(host[k].numel() * 4 for k in dma)
        in_place = 0
        for k in zero_copy:                                          # rows the list-based gather read from host memory
            in_place += int(o[("upsample_mask", k)].sum().item()) * host[k].shape[1] * 4
        del graphs_e2e, bufs, st
        torch.cuda.empty_cache()
        return ms_, h2d, in_place

    h2d_bytes = sum(f.numel() * 4 for f in host)
    e2e_ms, e2e_h2d, _ = run_e2e(())
    e2e_note = "pinned host features; H2D double-buffered on a copy stream; PCIe-bound"
    e2e_variants = [{"zero_copy_maps": [], "ms_per_step": round(e2e_ms / args.steps, 3), "h2d_bytes_per_step": e2e_h2d,
                     "value": round(n_global * args.steps / (e2e_ms * 1e-3), 1)}]
    e2e_dma = None
    if args.e2e_zero_copy and args.e2e_zero_copy != "off":
        # further variants: the listed skip map(s) stay in pinned host memory and the gated layout move reads only the
        # 32-pixel groups under the level's upsample mask, in place, across PCIe (graphs captured with gated_layout on)
        was = dec.gated_layout
        dec.gated_layout = was or not dec.compact_skip   # compact_skip (default) reads host maps through the list-based gather
        best = None
        try:
            for spec in args.e2e_zero_copy.split(";"):
                zc = tuple(int(k) for k in spec.split(","))
                with _Guard("e2e_zero_copy_%s" % spec, world == 1, section_errors):
                    zc_ms, zc_h2d, zc_in_place = run_e2e(zc)
                    e2e_variants.append({"zero_copy_maps": list(zc), "ms_per_step": round(zc_ms / args.steps, 3),
                                         "h2d_bytes_per_step": zc_h2d + zc_in_place, "dma_bytes": zc_h2d, "in_place_bytes": zc_in_place,
                                         "value": round(n_global * args.steps / (zc_ms * 1e-3), 1)})
                    log("[e2e] zero-copy skips %s: %.2f ms/step (%.0f MB DMA + %.0f MB in place) vs DMA-only %.2f ms/step"
                        % (zc, zc_ms / args.steps, zc_h2d / 1e6, zc_in_place / 1e6, e2e_ms / args.steps))
                    if best is None or zc_ms < best[0]:
                        best = (zc_ms, zc_h2d, zc_in_place, zc)
        finally:
            dec.gated_layout = was
        if best is not None and best[0] < e2e_ms:
            e2e_dma = {"value": round(n_global * args.steps / (e2e_ms * 1e-3), 1), "unit": UNIT,
                       "h2d_bytes_per_step": e2e_h2d * world, "ms_per_step": round(e2e_ms / args.steps, 3),
                       "note": "every feature map DMA-copied whole (the plain path)"}
            zc_ms, zc_h2d, zc_in_place, zc = best
            e2e_ms, e2e_h2d = zc_ms, zc_h2d + zc_in_place
            e2e_note = ("pinned host features; the other maps DMA-copied one step ahead on a copy stream, skip map(s) %s read in "
                        "place from pinned host memory by the list-based gather of the level's upsample-mask pixels (only "
                        "those rows cross PCIe: %.0f MB of %.0f MB, plus sector overfetch); h2d_bytes_per_step = DMA bytes + "
                        "those in-place reads; PCIe-bound" % (list(zc), zc_in_place / 1e6, sum(host[k].numel() * 4 for k in zc) / 1e6))
    e2e_value = n_global * args.steps / (e2e_ms * 1e-3)
    clocks = sampler.stop() if sampler else None

    # ---- 3. per-kernel roofline pass (same workload, CUDA events around every libwmd launch)
    prof_steps = 3
    prof = ops.Profiler()
    torch.cuda.synchronize()
    ops.set_profiler(prof)
    for _ in range(prof_steps):
        dec(resident, THRESH)
    torch.cuda.synchronize()
    ops.set_profiler(None)
    prof_records = prof.results()
    roof, roof_all = roofline_from(prof_records, peak_gbs, peak_tf, peak_src, prof_steps, peak_tf_sus, tf32_peak)
    conv_layers = conv_layer_table(prof_records, peak_gbs, tf32_peak, prof_steps)

    # ---- 4. secondary workload of the metric (device-resident only)
    also = None
    if args.workload == MAIN and not args.no_also:
        with _Guard("also", world == 1, section_errors):
            del resident
            torch.cuda.empty_cache()
            wl2, dec2, host2 = setup(ALSO)
            res2 = [f.to(dev) for f in host2]
            n2 = wl2["per_gpu_batch"] * world
            graph2 = graphs.GraphedSparseDecoder(dec2, res2, THRESH) if use_graph else None
            lst2 = {}
            st2 = _Stepper(graph2.replay if use_graph else (lambda: dec2(res2, THRESH)),
                           shard.make_gather(n2) if world > 1 else None, lst2)
            ms2 = time_device(st2.step, args.steps, max(args.warmup, 3), dist, world, flush=st2.flush)
            o2 = lst2["out"]
            also = {"workload": ALSO, "value": round(n2 * args.steps / (ms2 * 1e-3), 1), "unit": UNIT,
                    "ms_per_step": round(ms2 / args.steps, 3), "global_batch": n2,
                    "wavelet_mask_density": {str(s): round(float(o2[("wavelet_mask", s)].float().mean()), 4) for s in (3, 2, 1, 0)},
                    "total_ops_per_frame": lst2["total_ops"] / wl2["per_gpu_batch"]}
            del graph2, st2, res2

    # ---- 4b. NYUv2 workload of configs[3]: DenseNet161 pyramid 640x480, SparseDecoderWave thr 0.1, CUDA-graph replay.
    # Weak-scaled (8 frames per GPU) and, on several GPUs, as the config is written: global batch 8 sharded 1 -> 8.
    also_nyu = None
    if args.workload == MAIN and not args.no_also:
        with _Guard("also_nyu", world == 1, section_errors):
            from wavelet_monodepth_b200 import nyu_decoders
            torch.cuda.empty_cache()
            nmod = nyu_decoders.SparseDecoderWave(enc_features=list(NYU["ch"]), decoder_width=0.5)
            synth.load_random(nmod, seed=NYU["param_seed"], gains={k: SYNTH["head_gain"] for k in NYU["heads"]},
                              highpass=NYU["heads"])
            nmod = nmod.to(dev).eval()
            nmod.count_ops = "async"

            def nyu_run(nb, first):
                nfeats = [f.to(dev) for f in synth.blocky_features(
                    synth.nyu_feature_shapes(nb, NYU["height"], NYU["width"], NYU["ch"]), seed=NYU["feat_seed"] + first,
                    cell=SYNTH["cell"], texture=SYNTH["texture"])]
                n3 = nb * world
                g3 = graphs.GraphedSparseDecoder(nmod, nfeats, NYU["thresh"]) if use_graph else None
                lst3 = {}
                st3 = _Stepper(g3.replay if use_graph else (lambda: nmod(nfeats, NYU["thresh"])),
                               shard.OverlappedGather(n3) if world > 1 else None, lst3)
                ms3 = time_device(st3.step, args.steps, max(args.warmup, 3), dist, world, flush=st3.flush)
                o3 = lst3["out"]
                return {"value": round(n3 * args.steps / (ms3 * 1e-3), 1), "unit": UNIT, "ms_per_step": round(ms3 / args.steps, 3),
                        "global_batch": n3, "per_gpu_batch": nb,
                        "wavelet_mask_density": {str(s_): round(float(o3[("wavelet_mask", s_)].float().mean()), 4) for s_ in (2, 1, 0)},
                        "total_ops_per_frame": lst3["total_ops"] / nb}

            nb = NYU["per_gpu_batch"]
            also_nyu = {"workload": NYU["name"], "thresh_ratio": NYU["thresh"],
                        "launch_mode": "CUDA graph replay" if use_graph else "eager",
                        "decoder": "SparseDecoderWave (NYUv2/networks/decoders/densedepth_decoder.py:224-409), batched",
                        "dense_total_ops_per_frame": 33463546800}
            also_nyu.update(nyu_run(nb, rank * nb))
            also_nyu["scaling"] = "weak (8 frames per GPU)"
            if world > 1 and nb % world == 0:
                per = nb // world
                strong = nyu_run(per, rank * per)
                strong["scaling"] = "strong: configs[3] as written, global batch 8 sharded over %d GPUs (%d frame(s) each; latency-bound)" % (world, per)
                also_nyu["as_written_global_bs8"] = strong
            del nmod

    # ---- 5. CPU baseline + parity block (rank 0, N == 1 only)
    cpu, parity_block = None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import parity
        reports, seen = [], set()

        def on_frame(b, ref):
            if b in seen:
                return
            seen.add(b)
            reports.append(parity.compare_kitti_sample(parity.sample_of(out_host, b), ref, THRESH))

        fps, times = cpu_frames_per_sec(args.workload, args.cpu_frames, budget_s=20.0, batch=host, on_frame=on_frame)
        cpu = {"value": round(fps, 3), "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
               "sample": "%d frames of %s (the GPU arm's own %d-frame step, cycled), one at a time as the reference "
                         "requires; %.1fs of CPU work; intra-op threads chosen by probe out of %d usable cores"
                         % (len(times), args.workload, n_local, sum(times), _affinity_cores())}
        parity_block = parity.merge_reports(reports)
        parity_block["what"] = ("the timed step's own GPU outputs (every disp / wavelet plane, all five masks per scale, "
                                "total_ops) vs the oracle's outputs for the same frames, which the cpu_baseline leg computes "
                                "anyway; float bar 1e-4 relative, masks exact up to reported threshold ties (oracle/parity.py); "
                                "Haar bit-parity with pytorch_wavelets proper is unpinned (package absent), pinned algebraically")

    launches_t = torch.tensor([launches], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(launches_t)
    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, world),
            "workload_stats": {
                "wavelet_mask_density": {str(k): v for k, v in dens.items()},
                "total_ops_per_frame": ops_per_frame, "dense_total_ops_per_frame": 17473692295 if args.workload == MAIN else None,
                "timed_region": "decoder forward on NCHW fp32 features resident in HBM, incl. layout transposes, mask / "
                                "compaction kernels, the count read-back behind total_ops (asynchronous: evaluated one step "
                                "later, the last one inside the region) and (N>1) the all-gather of disp0 (started per step, "
                                "overlapped with the next step, the last one inside the region)",
                "launch_mode": "CUDA graph replay (graphs.GraphedSparseDecoder)" if use_graph else "eager",
                "head_1x1_stages": "fused (head_mlp) on levels 2, 1" if dec.fused_heads else "two gather-GEMM launches per level",
                "layout_moves": ("sparse levels %s: list-based gather of the upsample-mask pixels only (compact skip rows); other sparse "
                                 "levels: %s; dense level: whole maps" % (sorted(dec.compact_skip_levels),
                                                                        "transpose gated by the upsample mask" if dec.gated_layout else "whole maps")
                                 if dec.compact_skip else "%s, %s" % ("gated by the upsample mask" if dec.gated_layout else "whole maps",
                                                                      "side stream" if dec.overlap_layout else "in order")),
            },
            "value_eager": {"value": round(value_eager, 1), "unit": UNIT, "ms_per_step": round(ms_eager / args.steps, 3),
                            "note": "same step issued launch by launch from Python (no CUDA graph)"},
            "value_channels_last": {"value": round(value_cl, 1), "unit": UNIT, "ms_per_step": round(ms_cl / args.steps, 3),
                                    "note": "same step, encoder features in torch.channels_last: used zero-copy, no layout transposes"},
            "allgather_ms": round(allgather_ms, 3) if allgather_ms is not None else None,
            "reserved_sms": reserved_sms,
            "allgather_form": (None if gather is None else
                               "copy engines over NVLink peer memory (shard.PeerGather: one cudaMemcpyPeerAsync per peer + a 4-byte "
                               "NCCL all-reduce as the arrival barrier)" if getattr(gather, "_peer", None) not in (None, False) else
                               "NCCL all_gather_into_tensor (shard.OverlappedGather)%s" %
                               ("; peer form unavailable: %s" % gather.why_not if getattr(gather, "why_not", None) else "")),
            "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": e2e_h2d * world,
                    "d2h_bytes_per_step": d2h_bytes * world, "ms_per_step": round(e2e_ms / args.steps, 3),
                    "pcie_floor_ms": round(e2e_h2d / 57e9 * 1e3, 2),
                    "note": e2e_note + "; pcie_floor_ms = h2d bytes / 57 GB/s (what cudaMemcpyAsync from pinned memory "
                            "sustains on this box)" + ("; byte counts are the whole job's (rank 0's x %d ranks)" % world if world > 1 else "")},
            "e2e_dma": e2e_dma,
            "e2e_variants": e2e_variants,
            "gpu_launches": int(launches_t.item()),
            "clocks": clocks,
            "roofline": roof,
            "roofline_kernels": roof_all,
            "conv_layers": conv_layers,
            "sweep": sweep,
            "parity": parity_block,
            "cpu_baseline": cpu,
            "also": also,
            "also_nyu": also_nyu,
            "section_errors": section_errors or None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replay")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=MAIN, choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-frames", type=int, default=400)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-zero-copy", default=os.environ.get("WMD_E2E_ZERO_COPY", "0;0,1;0,1,2"),
                    help="';'-separated variants, each a comma list of skip-map indices that the variant leaves in pinned "
                         "host memory for the gated layout move to read in place (default: the finest map, then all three "
                         "sparse levels' maps); the fastest variant is reported as e2e; 'off' skips them")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the threshold sweep (configs[2] / configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs (rank 0's) as DIR/<name>.npy, at most 64 MB "
                         "in all: larger outputs as a fixed seeded sample of their elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if world != args.gpus:
        log("warning: --gpus %d but WORLD_SIZE=%d; using WORLD_SIZE" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device (no CPU fallback)")
    run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
