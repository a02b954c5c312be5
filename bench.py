"""bench.py - utterances/s of the speaker-conditioned mask-estimation forward pass on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp16_f8c|fp16x3|bf16x3|fp16|bf16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path (CNN -> BiLSTM -> FC -> sigmoid mask -> mask * spectrogram)
over one batch of synthetic utterances.  Workload (BASELINE.json configs[2]): `--batch` utterances per GPU of
601 frames x 257 bins + a random 256-d d-vector, random-init ("stress" flavour) weights of the
reference architecture.  Utterances are independent, so the batch is sharded across ranks with no
data-path collective (weak scaling; the only collective is the max-over-ranks of the timings).

One JSON line is printed by rank 0; keys are documented in DESIGN.md ("Measurement").  Besides the headline it carries
  train_config4   (every N)  BASELINE configs[3]: forward + Si-SNR loss chain + backward + ONE NCCL gradient all-reduce + Adam
  config2_conv_stack_b64, stock_torch_gpu_baseline, other_precisions, cpu_baseline, extras   (N = 1 only)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from voicesplit_b200 import synth  # noqa: E402

METRIC = "utterances/s (601-frame, 257-bin spectrogram) masked"
# MMA issue slots per tap-pair step relative to one fp16 pass (4 kind::f16 MMAs of K = 16 over the 64 input channels);
# an e4m3 MMA covers K = 32 in the same time, so the fp8 correction pass of fp16_f8c is one more slot-equivalent
PASS_EQUIV = {"bf16x3": 3, "fp16x3": 3, "fp16_f8c": 2, "bf16": 1, "fp16": 1}
DTYPE = {"bf16x3": "bf16x3 (split-bf16 operands hi+lo, 3 MMAs, fp32 accumulate)",
         "fp16x3": "fp16x3 (split-fp16 operands hi+lo, 3 MMAs, fp32 accumulate)",
         "fp16_f8c": "fp16 + e4m3 correction (conv stack: 4 kind::f16 + 4 kind::f8f6f4 MMAs per tap pair into one fp32 accumulator; LSTM/FC fp16x3)",
         "bf16": "bf16", "fp16": "f16", "fp32": "f32"}


# algorithmic forward FLOPs (2 x MAC) per utterance, SURVEY.md section 8(d)
def flops_per_utt(T, F, E=256, H=400, N1=600):
    P = T * F
    conv = 2 * P * (64 * 7 + 64 * 64 * 7 + 5 * 64 * 64 * 25 + 64 * 8)
    lstm_proj = 2 * T * (8 * F * 8 * H) + 2 * (E * 8 * H)
    lstm_rec = 2 * T * 2 * (H * 4 * H)
    fc = 2 * T * (2 * H * N1 + N1 * F)
    return dict(conv=conv, conv5x5_layer=2 * P * 64 * 64 * 25, lstm=lstm_proj + lstm_rec, lstm_input_proj=lstm_proj,
                lstm_recurrence=lstm_rec, fc=fc, total=conv + lstm_proj + lstm_rec + fc)


def padded_f(F):
    return (F + 2 + 7) // 8 * 8


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d["bf16_tflops_sustained"],
                    source="MEASURED_PEAKS.json (of measured)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="B200_PROFILING.md fallback (of fallback)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """Write each [B, ...] device output as out_dir/<name>.npy (float32).  When all of them together exceed DUMP_BYTES, the same
    evenly spaced utterances (always the first and the last) are kept from each, so two builds run with the same arguments can be
    compared output for output."""
    B = next(iter(arrays.values())).shape[0]
    keep = min(B, DUMP_BYTES // sum(a[0].numel() * 4 for a in arrays.values()))
    if keep < 1:
        raise SystemExit(f"--dump-outputs: one utterance's outputs exceed {DUMP_BYTES} bytes")
    idx = np.linspace(0, B - 1, keep).round().astype(np.int64)
    sel = torch.from_numpy(idx).to(next(iter(arrays.values())).device)
    os.makedirs(out_dir, exist_ok=True)
    shapes = {}
    for name, a in arrays.items():
        out = a.index_select(0, sel).float().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), out)
        shapes[name] = list(out.shape)
    return {"dir": out_dir, "shapes": shapes, "utterances": "all" if keep == B else idx.tolist()}


def _usable_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_model_name():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_throughput(dims, T, runs=5, warmup=1, batches=(1, 8), seconds_cap=150.0):
    """The reference's CPU implementation of the path - the same torch.nn ATen ops the reference module issues, restated in
    oracle/torch_port.py (/root/reference itself does not exist on the GPU box) - following BASELINE.md section 4:
    fp32, eval mode, B = 1 and B = 8 utterances of the FULL T x F, median of >= 5 runs after a warm-up, thread count the
    best of a sweep done at the full T (all cores is not always fastest for oneDNN on a many-core host).  Returns the
    cpu_baseline dict (value = the better of the two batch sizes) and the seconds of one median step."""
    from oracle import torch_port
    cores = _usable_cores()
    sd = {k: torch.from_numpy(v) for k, v in synth.make_state_dict(dims, 0, "stress").items() if v.dtype == np.float32}
    x1, e1 = synth.make_inputs(1, T, dims, 99)
    x1, e1 = torch.from_numpy(x1), torch.from_numpy(e1)
    t_start = time.perf_counter()
    # ascending, and stopped once a count is clearly past the knee: on the 128-core B200 hosts the all-cores probe takes
    # ~50 s per forward (oneDNN oversubscription, profiles/r02_bench_default_full.json) against 0.7 s at 8-32 threads
    sweep, skipped = {}, []
    for nt in sorted({cores, max(1, cores // 2), min(cores, 32), min(cores, 16), min(cores, 8)}):
        if sweep and sweep[max(sweep)] > 1.5 * min(sweep.values()):
            skipped.append(nt)
            continue
        torch.set_num_threads(nt)
        torch_port.forward(sd, x1, e1)
        t0 = time.perf_counter()
        torch_port.forward(sd, x1, e1)
        sweep[nt] = time.perf_counter() - t0
    best_t = min(sweep, key=sweep.get)
    torch.set_num_threads(best_t)
    per_batch = {}
    for bs in batches:
        x, emb = synth.make_inputs(bs, T, dims, 99)
        xt, et = torch.from_numpy(x), torch.from_numpy(emb)
        for _ in range(max(warmup, 1)):
            torch_port.forward(sd, xt, et)
        times = []
        for _ in range(max(runs, 5)):
            t0 = time.perf_counter()
            torch_port.forward(sd, xt, et)
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_start > seconds_cap and len(times) >= 3:
                break
        per_batch[bs] = dict(median_s=float(np.median(times)), runs=len(times), utt_per_s=bs / float(np.median(times)))
    best_b = max(per_batch, key=lambda b: per_batch[b]["utt_per_s"])
    return dict(value=per_batch[best_b]["utt_per_s"], unit="utterances/s", cores=best_t, kind="port",
                host=f"{cpu_model_name()}, {cores} usable cores",
                per_batch={str(b): v for b, v in per_batch.items()}, thread_sweep_s={str(k): round(v, 4) for k, v in sweep.items()},
                thread_sweep_skipped=skipped,
                sample=f"B = {', '.join(str(b) for b in batches)} utterance(s) of {T}x{dims['num_freq']} through oracle/torch_port.py (the reference's own "
                       f"torch.nn CPU ops, fp32, eval), median of {per_batch[best_b]['runs']} runs after warm-up, {best_t} of {cores} host "
                       f"threads (best of a sweep at the full T); value = B = {best_b}"), per_batch[best_b]["median_s"]


# =====================================================================================================================
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("VOICESPLIT_BENCH_PRECISION", "fp16_f8c"))
    ap.add_argument("--batch", type=int, default=256, help="utterances per GPU")
    ap.add_argument("--frames", type=int, default=601)
    ap.add_argument("--freq", type=int, default=257)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip every secondary block (training, config 2, baselines)")
    ap.add_argument("--no-train", action="store_true", help="skip the config-4 training block")
    ap.add_argument("--train-batch", type=int, default=256, help="config 4: utterances per GPU to try first (halved until it fits)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write mask.npy and masked.npy of the last timed step to DIR (rank 0; "
                                                           "evenly spaced whole utterances when all of them exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dims = synth.make_dims(args.freq, 256, 400, 600)
    T, F, B = args.frames, args.freq, args.batch
    fl = flops_per_utt(T, F)
    workload = f"full forward CNN+BiLSTM+FC+mask apply, {B} utt/GPU x {T} frames x {F} bins + 256-d d-vector (BASELINE configs[2] shape)"
    config = {"workload": workload, "per_gpu_batch": B, "frames": T, "freq_bins": F, "global_batch": B * world,
              "parallelism": f"utterance-sharded x{world}, no data-path collective",
              "l2_policy": "inputs larger than L2 (x is %.0f MB per step)" % (B * T * F * 4 / 1e6),
              "weights": "random-init stress flavour (synth.make_state_dict seed 0)"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        cb, step_s = cpu_reference_throughput(dims, T, runs=max(args.steps, 5), warmup=max(args.warmup, 1))
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"],
                "unit": "utterances/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    from voicesplit_b200 import dist as vdist
    from voicesplit_b200.engine import MaskEngine
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = vdist.init("nccl", dev)

    eng = MaskEngine(activation="mish", device=dev, **dims)
    sd = synth.make_state_dict(dims, 0, "stress")
    eng.load_state_dict_tensors({k: torch.from_numpy(v).to(dev) for k, v in sd.items() if v.dtype == np.float32})
    xnp, enp = synth.make_inputs(B, T, dims, 1234 + rank)
    xh, eh = torch.from_numpy(xnp).pin_memory(), torch.from_numpy(enp).pin_memory()
    x, emb = xh.to(dev), eh.to(dev)
    mask_h, masked_h = torch.empty_like(xh).pin_memory(), torch.empty_like(xh).pin_memory()
    prec = args.precision

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, keep_last=None):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(steps):
            if keep_last is not None and i == steps - 1:
                keep_last.append(fn())
            else:
                fn()        # earlier outputs are dropped at once, so the allocator serves every step from the same blocks
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        barrier()
        return ms

    # ---- parity evidence on utterances of the timed batch: the timed precision against (a) the CPU oracle
    # (oracle/voicesplit_oracle.c, pinned to the reference's golden vectors; one utterance, rank 0 at N = 1 only) and
    # (b) this repo's fp32 CUDA-core path on the first two utterances
    nb = min(2, B)
    ref32 = eng.forward(x[:nb], emb[:nb], precision="fp32")
    got = eng.forward(x[:nb], emb[:nb], precision=prec)
    parity = {"vs_fp32_path": {"utterances": nb, "mask_mae": float((got - ref32).abs().mean()), "mask_max_abs": float((got - ref32).abs().max())}}
    # (c) the launch that is timed - all B utterances in ONE call: first / middle / last utterance against their own
    # single-utterance runs (utterances are independent, so any difference is batch-dependent indexing, e.g. a 32-bit offset
    # into the 2.6e9-element activation planes of B = 256) and against the fp32 path
    first_of_batch, first_src = got[:1].cpu().numpy(), "a 2-utterance call"
    try:
        full = eng.forward(x, emb, precision=prec)
        picks = sorted({0, B // 2, B - 1})
        worst_self = worst_32 = 0.0
        for b in picks:
            one = eng.forward(x[b:b + 1], emb[b:b + 1], precision=prec)
            r32 = eng.forward(x[b:b + 1], emb[b:b + 1], precision="fp32")
            worst_self = max(worst_self, float((full[b:b + 1] - one).abs().max()))
            worst_32 = max(worst_32, float((full[b:b + 1] - r32).abs().max()))
        first_of_batch, first_src = full[:1].cpu().numpy(), f"the B = {B} call"
        parity["timed_batch"] = {"utterances": picks, "batch": B, "max_abs_vs_single_utterance_run": worst_self,
                                 "max_abs_vs_fp32_path": worst_32,
                                 "what": f"utterances {picks} of ONE B = {B} call in the timed precision against the same utterances run alone "
                                         "(same precision; expected 0) and against the fp32 CUDA-core path"}
        del full
    except Exception as ex:      # noqa: BLE001 - evidence only: must not cost the bench line
        parity["timed_batch"] = {"error": repr(ex)[:200]}
    if world == 1 and not args.no_extras:
        try:
            from oracle import oracle as c_oracle
            t0 = time.perf_counter()
            om = c_oracle.forward(sd, dims, xnp[:1], enp[:1])["mask"]
            d = np.abs(first_of_batch - om)
            parity["vs_cpu_oracle"] = {"utterances": 1, "what": f"utterance 0 of the timed batch (output of {first_src}), oracle/voicesplit_oracle.c (double accumulation)",
                                       "mask_mae": float(d.mean()), "mask_max_abs": float(d.max()), "oracle_seconds": round(time.perf_counter() - t0, 2)}
        except Exception as ex:      # noqa: BLE001
            parity["vs_cpu_oracle"] = {"error": repr(ex)[:200]}

    # ---- device-resident throughput ("value")
    for _ in range(args.warmup):
        eng.forward(x, emb, precision=prec, want_masked=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    eng.set_profiling(True)
    last = [] if args.dump_outputs else None
    local_ms = timed(lambda: eng.forward(x, emb, precision=prec, want_masked=True), args.steps, keep_last=last)
    kernel_ms = {}
    for name, ms in eng.profile_read():           # per-kernel times of the last timed step
        kernel_ms[name] = kernel_ms.get(name, 0.0) + ms
    launches_per_step = eng.last_launch_count()
    eng.set_profiling(False)
    dumped = dump_outputs(args.dump_outputs, dict(zip(("mask", "masked"), last[0]))) if last and rank == 0 else None
    last = None
    value, dev_ms = vdist.aggregate_throughput(B * args.steps, local_ms, dist, dev)
    # ---- end to end through the host-buffer plugin call ("e2e"): every step copies its inputs from pinned
    # host memory, runs the forward and copies mask + masked back.  The serving form of the call is
    # used (vs_forward_host_submit / _wait, two slots), so the copies of step i+1 / i-1 overlap the
    # compute of step i; the synchronous vs_forward_host is timed as well and reported next to it.
    for _ in range(min(args.warmup, 2)):
        eng.forward_host(xh, eh, mask_h, masked_h, precision=prec)
    local_sync = timed(lambda: eng.forward_host(xh, eh, mask_h, masked_h, precision=prec), max(2, args.steps // 2))
    sync_value, _ = vdist.aggregate_throughput(B * max(2, args.steps // 2), local_sync, dist, dev)
    slots = [(xh, eh, mask_h, masked_h),
             (xh.clone().pin_memory(), eh.clone().pin_memory(), torch.empty_like(xh).pin_memory(), torch.empty_like(xh).pin_memory())]

    def pipelined(steps):
        for i in range(steps):
            eng.host_submit(i & 1, *slots[i & 1], precision=prec)
            if i > 0:
                eng.host_wait((i - 1) & 1)
        eng.host_wait((steps - 1) & 1)

    pipelined(2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipelined(args.steps)           # the last host_wait blocks until the last D2H has landed
    e1.record()
    torch.cuda.synchronize()
    local_e2e = e0.elapsed_time(e1)
    barrier()
    e2e_value, e2e_ms = vdist.aggregate_throughput(B * args.steps, local_e2e, dist, dev)
    clocks = sampler.stop() if rank == 0 else None

    # ---- companion modes: the fp32-faithful fp16x3 (when the headline is fp16_f8c) and the single-pass fast mode, each with
    # its measured error (never the headline)
    def side_mode(p, note):
        g = eng.forward(x[:nb], emb[:nb], precision=p)
        for _ in range(2):
            eng.forward(x, emb, precision=p, want_masked=True)
        n = max(2, args.steps // 2)
        ms = timed(lambda: eng.forward(x, emb, precision=p, want_masked=True), n)
        v, _ = vdist.aggregate_throughput(B * n, ms, dist, dev)
        return {"precision": p, "value": v, "unit": "utterances/s", "mask_mae_vs_fp32_path": float((g - ref32).abs().mean()),
                "mask_max_abs_vs_fp32_path": float((g - ref32).abs().max()), "note": note}
    fast = faithful = None
    if prec in ("fp16x3", "bf16x3", "fp16_f8c"):
        fast = side_mode(prec[:4], "single MMA pass, 11-bit (fp16) / 8-bit (bf16) operands; error measured on stress weights")
    if prec == "fp16_f8c":
        faithful = side_mode("fp16x3", "fp32-faithful split-fp16 mode (three fp16 MMA passes): the accuracy reference among the tensor-core modes")

    del slots
    line = None
    if rank == 0:
        peaks = load_peaks()
        passes = PASS_EQUIV.get(prec)
        # dominant kernel: the five 5x5 dilated conv layers (89.5 % of the algorithmic FLOPs)
        conv_ms = [kernel_ms.get(f"cnn{i}") for i in (3, 4, 5, 6, 7)]
        roof = None
        if all(v is not None for v in conv_ms):
            avg = float(np.mean(conv_ms))
            ach = fl["conv5x5_layer"] * B / (avg / 1e3) / 1e12
            peak = peaks["bf16_tflops_sustained"]
            traffic, traffic_src = None, None
            for name in ("r02_conv_tc_summary.json", "r01_conv_tc_summary.json"):
                prof = os.path.join(ROOT, "profiles", name)
                if os.path.exists(prof) and passes:
                    pj = json.load(open(prof))
                    if pj.get("precision") == prec and pj.get("frames") == T and pj.get("freq_bins") == F:
                        traffic = pj["dram_bytes_per_launch"] / pj["batch"] * B
                        traffic_src = (f"profiles/{name} (ncu at B = {pj['batch']}: dram__bytes_read + dram__bytes_write, mean over the five 5x5 "
                                       "launches of one forward, scaled per utterance)")
                        break
            roof = {"bound": "tensor", "kernel": "k_conv_tc: dilated 5x5 conv 64->64 + BN + act (cnn3..cnn7)", "achieved": ach, "peak": peak,
                    "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["source"] + ", sustained 16-bit dense (cuBLAS bf16; fp16 runs on the same pipe)",
                    "avg_launch_ms": avg, "algorithmic_flops_per_launch": fl["conv5x5_layer"] * B,
                    "algorithmic_bytes_per_launch": B * T * padded_f(F) * 64 * 2 * (2 if (passes or 0) >= 2 else 1) * 2 if passes else None,
                    "mma_pass_equivalents": passes, "tensor_pipe_frac_incl_passes": (ach * passes / peak) if passes else None,
                    # what the tensor pipe actually executes: algorithmic flops x pass-equivalents x 6/5 (five filter taps occupy six M=128 slots)
                    "issued_tflops": (ach * passes * 1.2) if passes else None,
                    "issued_frac_of_peak": (ach * passes * 1.2 / peak) if passes else None,
                    "note": "fp32 mode runs on CUDA cores (no tensor pipe)" if prec == "fp32" else
                            "frac counts ALGORITHMIC flops; fp16_f8c issues the fp16 pass + one e4m3 pass at twice the rate (2 pass-equivalents), "
                            "fp16x3/bf16x3 three 16-bit passes; five taps occupy six M=128 slots"}
        # the BiLSTM against the same tensor roofline (north_star: ">= 60 % of the BiLSTM tensor-core roofline")
        roof_lstm = None
        if kernel_ms.get("lstm_input_proj") and kernel_ms.get("lstm_recurrence"):
            pj_ms, rc_ms = kernel_ms["lstm_input_proj"], kernel_ms["lstm_recurrence"]
            peak = peaks["bf16_tflops_sustained"]
            a_all = fl["lstm"] * B / ((pj_ms + rc_ms) / 1e3) / 1e12
            a_pj = fl["lstm_input_proj"] * B / (pj_ms / 1e3) / 1e12
            a_rc = fl["lstm_recurrence"] * B / (rc_ms / 1e3) / 1e12
            roof_lstm = {"bound": "tensor (input projection) / step latency (recurrence)", "kernel": "k_gemm_tc<GATES> + k_lstm_tc",
                         "achieved": a_all, "peak": peak, "unit": "TFLOP/s", "frac": a_all / peak,
                         "input_projection": {"ms": pj_ms, "achieved": a_pj, "frac": a_pj / peak, "frac_incl_3_passes": 3 * a_pj / peak},
                         "recurrence": {"ms": rc_ms, "achieved": a_rc, "frac": a_rc / peak, "us_per_step": rc_ms * 1e3 / T,
                                        "note": "T sequential steps; bounded by the per-step exchange latency, not by the tensor pipe"},
                         "algorithmic_flops_per_launch": fl["lstm"] * B,
                         "ncu_tensor_pipe_pct": {"input_projection": 67.7, "recurrence": 13.8,
                                                 "source": "profiles/r02_ncu_final_gates_f8c_b256_summary.txt, r02_ncu_final_lstm_f8c_b256_summary.txt (ncu --set full at B = 256)"}}
        line = {"metric": METRIC, "value": value, "unit": "utterances/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPE[prec], "data": "synthetic", "config": config,
                "e2e": {"value": e2e_value, "unit": "utterances/s", "ms_per_step": e2e_ms / args.steps,
                        "api": "vs_forward_host_submit/_wait (2 slots, copies overlap the neighbouring step's compute)",
                        "synchronous_call_value": sync_value,
                        "h2d_bytes_per_step": int(xh.numel() * 4 + eh.numel() * 4),
                        "d2h_bytes_per_step": int(mask_h.numel() * 4 + masked_h.numel() * 4)},
                "gpu_launches": launches_per_step * args.steps * 2,   # device-resident + e2e timed regions
                "launches_per_step": launches_per_step,
                "clocks": clocks, "roofline": roof, "roofline_lstm": roof_lstm, "parity": parity, "faithful_mode": faithful, "fast_mode": fast,
                "kernel_ms_last_step": {k: round(v, 4) for k, v in kernel_ms.items()},
                "gflop_per_utt": {k: v / 1e9 for k, v in fl.items()},
                "tflops_total_algorithmic": fl["total"] * value / 1e12}
        if dumped:
            line["dumped_outputs"] = dumped

    # free the inference buffers before the secondary blocks
    del eng, x, emb, xh, eh, mask_h, masked_h, ref32, got
    torch.cuda.empty_cache()

    # ---- BASELINE configs[3]: training step, every N (so the scaling run carries the 1 -> 8 training curve)
    if not args.no_extras and not args.no_train:
        try:
            tr = train_config4(dev, dist, rank, world, args.train_batch, barrier)
        except Exception as ex:      # noqa: BLE001 - a failure here must not cost the headline
            tr = {"error": repr(ex)[:300]}
        if rank == 0:
            line["train_config4"] = tr
    if rank == 0:
        if world == 1 and not args.no_extras:
            for key, fn in (("config2_conv_stack_b64", lambda: config2_conv_stack(dev, prec)),
                            ("stock_torch_gpu_baseline", lambda: stock_torch_gpu_baseline(dev, B, T)),
                            ("other_precisions", lambda: other_precisions(dev, dims, B, T, prec)),
                            ("extras", lambda: extra_measurements(dev))):
                try:
                    torch.cuda.empty_cache()
                    line[key] = fn()
                except Exception as ex:      # noqa: BLE001
                    line[key] = {"error": repr(ex)[:300]}
        if world == 1 and not args.no_cpu_baseline:
            cb, _ = cpu_reference_throughput(dims, T, runs=5, seconds_cap=60.0)
            line["cpu_baseline"] = cb
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# =====================================================================================================================
def train_config4(dev, dist, rank, world, want_batch, barrier, steps=3, warmup=2):
    """BASELINE configs[3]: forward (batch-statistics BatchNorm) + the reference's loss chain (train.py:95-108: both spectrograms
    through the Q1-faithful differentiable iSTFT, Si-SNR, one fused engine call) + backward + ONE flat NCCL gradient
    all-reduce (LSTM / FC tail overlapped with the conv backward) + Adam, at the reference-native 301 x 601, per-rank
    BatchNorm statistics (the DDP default; SyncBN is a flag, tests/test_gpu_dp.py).  Per-GPU batch: `want_batch` halved
    until the engine's workspace fits the free memory (agreed across ranks)."""
    from voicesplit_b200 import config as vconfig
    from voicesplit_b200 import dist as vdist
    from voicesplit_b200.losses import SpecSiSNRLoss
    from models.voicesplit.model import VoiceSplit
    dims = synth.make_dims(601, 256, 400, 600)
    T, F = 301, 601
    model = VoiceSplit(vconfig.AttrDict(synth.make_config_dict(dims)))
    model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in synth.make_state_dict(dims, 0, "default").items()})
    model = model.to(dev).train()
    eng = model.engine(dev)
    free, _total = torch.cuda.mem_get_info(dev)
    free += torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)
    B = want_batch
    while B > 1:
        # engine workspace + the torch-side tensors of a step (x, target, phase, mask, mask*x, their gradients, loss chain) + slack
        need = int(eng.lib.vs_train_workspace_bytes(eng.handle, B, T)) + 14 * B * T * F * 4 + (6 << 30)
        if need <= free:
            break
        B //= 2
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    crit = SpecSiSNRLoss(eng, dict(n_fft=1200, hop_length=160, win_length=400), "q1")
    # One LOCAL step (no collective in it: the data-parallel hooks are installed afterwards) proves that the batch fits on every rank;
    # the ranks then agree, so a rank that ran out of memory cannot leave the others waiting in a gradient all-reduce.
    while True:
        if dist is not None:
            t = torch.tensor([B], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            B = int(t.item())
        ok, err = 1, ""
        try:
            x, emb = synth.make_inputs(min(B, 32), T, dims, 7 + rank)
            reps = (B + x.shape[0] - 1) // x.shape[0]
            x = torch.from_numpy(np.tile(x, (reps, 1, 1))[:B]).to(dev)
            emb = torch.from_numpy(np.tile(emb, (reps, 1))[:B]).to(dev)
            x = (x + 0.01 * torch.rand_like(x)).clamp_(0, 1)         # utterances differ (tiling only bounds the host-side generation time)
            target = torch.rand(B, T, F, device=dev) * x
            phase = (torch.rand(B, T, F, device=dev) * 2 - 1) * np.pi
            seq_len = torch.full((B, 1), 160 * (T - 1), device=dev, dtype=torch.int64)
            opt.zero_grad(set_to_none=True)
            crit(model(x, emb) * x, target, phase, seq_len).backward()
            opt.step()
            torch.cuda.synchronize()
        except (torch.OutOfMemoryError, RuntimeError) as ex:
            ok, err = 0, repr(ex)[:200]
        if dist is not None:
            t = torch.tensor([ok], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok = int(t.item())
        if ok:
            break
        x = emb = target = phase = None
        opt.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
        if B <= 8:
            raise RuntimeError(f"training step does not fit at {B} utterances per GPU: {err}")
        B //= 2
    model.enable_data_parallel(dist, sync_bn=False, overlap=True)
    ar_events = []

    def step(record=False):
        opt.zero_grad(set_to_none=True)
        mask = model(x, emb)
        loss = crit(mask * x, target, phase, seq_len)
        loss.backward()
        if record:
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
        n = vdist.allreduce_gradients(model, dist)
        if record:
            a1.record()
            ar_events.append((a0, a1))
        opt.step()
        return loss, n
    for _ in range(warmup):
        loss, nred = step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, nred = step(record=True)
    e1.record()
    torch.cuda.synchronize()
    local_ms = e0.elapsed_time(e1)
    loss_val = float(loss.detach())
    ar_ms = float(np.mean([a.elapsed_time(b) for a, b in ar_events]))
    barrier()
    value, ms = vdist.aggregate_throughput(B * steps, local_ms, dist, dev)
    ar_max = vdist.max_over_ranks(ar_ms, dist, dev)
    # the collective alone: the same 75.5 MB flat buffer, all ranks entering together (right after a barrier), no backward in flight
    ar_iso = None
    flat = model.flat_gradient()
    if dist is not None and flat is not None:
        vdist.reduce_flat(flat, dist)
        iso = []
        for _ in range(5):
            barrier()
            i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            i0.record()
            vdist.reduce_flat(flat, dist)
            i1.record()
            torch.cuda.synchronize()
            iso.append(i0.elapsed_time(i1))
        ar_iso = vdist.max_over_ranks(float(np.median(iso)), dist, dev)
    peak_mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    out = {"value": value, "unit": "utterances/s", "frames_per_s": value * T, "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "per_gpu_batch": B, "global_batch": B * world, "frames": T, "freq_bins": F, "n_gpus": world, "scaling": "weak",
           "allreduce_ms": ar_iso if ar_iso is not None else ar_max, "allreduce_exposed_ms": ar_max,
           "allreduce_elements": int(nred), "allreduce_bytes": int(nred) * 4,
           "allreduce_what": "allreduce_ms = ONE in-place NCCL ReduceOp.AVG over the flat 75.5 MB gradient buffer with all ranks entering together "
                             "(median of 5, max over ranks; no gather, no copy-back); allreduce_exposed_ms = what allreduce_gradients costs inside the "
                             "step after backward (max over ranks): the LSTM/FC tail was started mid-backward on NCCL's stream, so this is the 2.3 MB "
                             "conv/BatchNorm head plus the wait for the slowest rank's backward (rank skew, not wire time)",
           "bn_statistics": "per-rank (DDP default); sync_bn=True gives the concatenated-batch statistics of the single-process reference",
           "loss_last_step": loss_val, "peak_memory_gib": round(peak_mem, 1),
           "what": "forward (batch-stat BN) + differentiable iSTFT x2 + Si-SNR (one fused engine call) + backward + flat gradient all-reduce + Adam; "
                   "conv fwd/dgrad/wgrad, LSTM input GEMMs and the iSTFT GEMMs on tcgen05 (fp16x3/bf16x3), BN / LSTM recurrence backward fp32 CUDA cores",
           "flops_per_utt_algorithmic": 3 * flops_per_utt(T, F)["total"],
           "tflops_algorithmic": 3 * flops_per_utt(T, F)["total"] * value / 1e12}
    del model, opt, crit, x, emb, target, phase
    torch.cuda.empty_cache()
    return out


def _time_gpu(fn, n, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def config2_conv_stack(dev, prec, B=64, T=601, F=257):
    """BASELINE configs[1]: the conv stack alone (8 x conv+BN+Mish and the transpose/view of model.py:70-74), B = 64, against the
    reference's `model.conv` ops (oracle/torch_port.conv_stack: F.pad/conv2d/batch_norm/Mish -> cuDNN) on the SAME GPU."""
    from oracle import torch_port
    from voicesplit_b200.engine import MaskEngine
    dims = synth.make_dims(F, 256, 400, 600)
    sdn = synth.make_state_dict(dims, 0, "stress")
    eng = MaskEngine(activation="mish", device=dev, **dims)
    eng.load_state_dict_tensors({k: torch.from_numpy(v).to(dev) for k, v in sdn.items() if v.dtype == np.float32})
    x, _ = synth.make_inputs(B, T, dims, 21)
    x = torch.from_numpy(x).to(dev)
    sd = {k: torch.from_numpy(np.array(v)).to(dev) for k, v in sdn.items()}
    out = {"batch": B, "frames": T, "freq_bins": F, "unit": "utterances/s", "gflop_per_utt": flops_per_utt(T, F)["conv"] / 1e9}
    ref = torch_port.conv_stack(sd, x[:2])
    for p in sorted({prec, "fp16x3"}):
        got = eng.conv_stack(x[:2], precision=p)
        ms = _time_gpu(lambda: eng.conv_stack(x, precision=p), 5)
        out[p] = {"value": B / (ms / 1e3), "ms": ms, "tflops_algorithmic": flops_per_utt(T, F)["conv"] * B / (ms / 1e3) / 1e12,
                  "max_abs_vs_stock_fp32": float((got - ref).abs().max()), "mean_abs_vs_stock_fp32": float((got - ref).abs().mean()),
                  "ref_abs_max": float(ref.abs().max())}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        for name, tf32 in (("stock_fp32", False), ("stock_tf32", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            ms = _time_gpu(lambda: torch_port.conv_stack(sd, x), 3)
            out[name] = {"value": B / (ms / 1e3), "ms": ms}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    out["speedup_vs_stock_fp32"] = out[prec]["value"] / out["stock_fp32"]["value"]
    out["speedup_vs_stock_tf32"] = out[prec]["value"] / out["stock_tf32"]["value"]
    return out


def stock_torch_gpu_baseline(dev, B=256, T=601, F=257):
    """The honest GPU bar (SURVEY.md 8(d)): the reference's own stock torch ops (restated in oracle/torch_port.py; the reference
    tree cannot travel) on the SAME B200 through cuDNN/cuBLAS eager, strict fp32 and TF32-allowed, at the SAME per-GPU batch
    as the headline (halved on out-of-memory, stated)."""
    from oracle import torch_port
    dims = synth.make_dims(F, 256, 400, 600)
    sd = {k: torch.from_numpy(np.array(v)).to(dev) for k, v in synth.make_state_dict(dims, 0, "stress").items()}
    try:
        # give cuDNN the LSTM weights the way nn.LSTM.cuda() holds them - one flat buffer - so that the baseline does not
        # re-compact 40 MB of weights on every call (a stock module would not either)
        lstm = torch.nn.LSTM(8 * F + dims["emb_dim"], dims["lstm_dim"], batch_first=True, bidirectional=True).to(dev)
        with torch.no_grad():
            for name, p in lstm.named_parameters():
                p.copy_(sd[f"lstm.{name}"])
        lstm.flatten_parameters()
        for name, p in lstm.named_parameters():
            sd[f"lstm.{name}"] = p.detach()
    except Exception:      # noqa: BLE001 - keep the separately allocated weights (cuDNN compacts them per call and warns)
        pass
    res = {"frames": T, "freq_bins": F, "unit": "utterances/s", "requested_batch": B,
           "what": "stock PyTorch eager (F.conv2d/batch_norm/Mish/LSTM/linear -> cuDNN/cuBLAS) on the same GPU, inputs resident"}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        while B >= 1:
            x = emb = None
            try:
                x, emb = synth.make_inputs(min(B, 32), T, dims, 11)
                reps = (B + x.shape[0] - 1) // x.shape[0]
                x = torch.from_numpy(np.tile(x, (reps, 1, 1))[:B]).to(dev)
                emb = torch.from_numpy(np.tile(emb, (reps, 1))[:B]).to(dev)
                for name, tf32 in (("fp32", False), ("tf32", True)):
                    torch.backends.cudnn.allow_tf32 = tf32
                    torch.backends.cuda.matmul.allow_tf32 = tf32
                    ms = _time_gpu(lambda: torch_port.forward(sd, x, emb), 3)
                    res[name] = B / (ms / 1e3)
                res["batch"] = B
                break
            except torch.OutOfMemoryError:
                del x, emb
                torch.cuda.empty_cache()
                B //= 2
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    return res


def other_precisions(dev, dims, B, T, headline):
    """BASELINE configs[2] names "fp32 and bf16": the same B = 256 forward in the fp32 CUDA-core mode and the bf16 modes."""
    from voicesplit_b200.engine import MaskEngine
    eng = MaskEngine(activation="mish", device=dev, **dims)
    eng.load_state_dict_tensors({k: torch.from_numpy(v).to(dev) for k, v in synth.make_state_dict(dims, 0, "stress").items() if v.dtype == np.float32})
    x, emb = synth.make_inputs(B, T, dims, 1234)
    x, emb = torch.from_numpy(x).to(dev), torch.from_numpy(emb).to(dev)
    ref = eng.forward(x[:2], emb[:2], precision="fp32")
    out = {"batch": B, "unit": "utterances/s"}
    for p, n in (("fp32", 2), ("bf16x3", 3), ("bf16", 3)):
        if p == headline:
            continue
        g = eng.forward(x[:2], emb[:2], precision=p)
        ms = _time_gpu(lambda: eng.forward(x, emb, precision=p, want_masked=True), n, warm=1)
        out[p] = {"value": B / (ms / 1e3), "ms_per_step": ms, "mask_mae_vs_fp32_path": float((g - ref).abs().mean()),
                  "mask_max_abs_vs_fp32_path": float((g - ref).abs().max())}
    return out


def extra_measurements(dev):
    """Config 5 (waveform in, separated waveform out) and d-vector extraction at the reference-native shape."""
    from voicesplit_b200.engine import MaskEngine
    out = {}
    dims = synth.make_dims(601, 256, 400, 600)
    eng = MaskEngine(activation="mish", device=dev, **dims)
    eng.load_state_dict_tensors({k: torch.from_numpy(v).to(dev) for k, v in synth.make_state_dict(dims, 0, "stress").items() if v.dtype == np.float32})
    eng.configure_audio()
    Bw = 64
    wav = torch.randn(Bw, 48000, device=dev) * 0.05
    e2 = torch.randn(Bw, 256, device=dev)
    ms = _time_gpu(lambda: eng.separate(wav, e2), 3, warm=1)
    out["audio_e2e_config5"] = {"value": Bw / (ms / 1e3), "unit": "utterances/s", "ms_per_step": ms, "batch": Bw, "samples": 48000,
                                "what": "waveform -> STFT (tcgen05 GEMM) -> CNN+BiLSTM+FC mask (fp16x3) -> mask*spec -> iSTFT (mixture phase) -> waveform"}
    from voicesplit_b200.speaker_encoder import SpeakerEncoder
    enc = SpeakerEncoder(engine=eng)
    enc.load_state_dict({k: torch.from_numpy(v) for k, v in synth.make_encoder_state_dict(1, "stress").items()})
    enc = enc.to(dev)
    ref_wav = torch.from_numpy(synth.make_reference_audio(128, 48000, 5)).to(dev)
    ms = _time_gpu(lambda: enc.embed_wav(ref_wav), 5, warm=1)
    out["dvector_extract"] = {"value": 128 / (ms / 1e3), "unit": "utterances/s", "ms_per_step": ms, "batch": 128, "samples": 48000,
                              "what": "waveform -> |STFT|^2 -> 40 mel -> log10 -> 6 windows x 3 x LSTM(768) (fp16x3 tcgen05, persistent recurrent "
                                      "kernel) -> Linear(256) -> L2 normalise -> mean"}
    return out


if __name__ == "__main__":
    sys.exit(main())
