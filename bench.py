#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: utterances/sec, ECAPA-TDNN + Fbank-80, 3 s @ 16 kHz, waveform -> 192-d
embedding (configs[1]: batch 256 x 3 s synthetic audio per GPU).

  python bench.py [--gpus N --steps K --warmup W] [--impl ours|reference] [--precision bf16x3|bf16] [--dump-outputs DIR]

One "step" = one batch of 256 utterances through the whole hot path.
  value     device-resident waveforms -> embeddings on device, CUDA events around the K timed steps, LANES batches in
            flight (PPVectorPredictor.embed_resident_stream: replica models on their own streams fill the SMs a batch's
            kernels leave idle at their tails and between dependent launches); `single_lane` = one batch at a time
  e2e       the same through PPVectorPredictor.extract_embeddings_stream: pinned host fp32 waveforms -> H2D (copy
            stream) -> hot path (LANES lanes) -> D2H embeddings, every step
  roofline  tensor-core gather-GEMM (the dominant kernel): algorithmic FLOPs / its summed launch time, measured
            with CUDA events on the launching stream around every kernel of the K steps of the single-lane pass
  cpu_baseline  the oracle (torch CPU port of the reference path; Paddle is not installable) on a bounded sample
N > 1: one process per GPU (torchrun), each rank extracts its own 256-utterance batches (weak scaling, no
data-path collective); barrier + synchronize on both sides; elapsed = max over ranks.
--impl reference: the reference's own CPU path is pure Python over paddle/paddleaudio, which cannot be installed
here (no network); the timed stand-in is the oracle port on all host cores (kind = "port").
--dump-outputs DIR: after the timed passes, rank 0 writes the embeddings of the LAST timed step as DIR/<name>.npy (float32):
  embeddings.npy      [256, 192] from the device-resident pass behind `value`
  e2e_embeddings.npy  [256, 192] from the end-to-end pass (PPVectorPredictor.extract_embeddings_stream)
Inputs and weights are seeded, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "voiceprintrecognition-paddlepaddle_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

BATCH = 256
SAMPLES = 48000
FRAMES = 298
LANES = 3  # batches in flight in the timed passes (PPVectorPredictor lanes: replica models on their own streams)
METRIC = "utterances/sec ECAPA-TDNN Fbank80 3s embed extract"


def algorithmic_flops_per_utt(T=FRAMES, F=80, C=512, scale=8, A=128, S=128, E=192, k0=5):
    """SURVEY.md §8(d): 2 x MACs of the reference graph with ASP's tiled [mean;std] folded into a bias
    (what this build executes): 2.857 GFLOP per 3 s utterance."""
    w = C // scale
    C3 = 3 * C
    per_frame = k0 * F * C + 3 * (C * C + (scale - 1) * 3 * w * w + C * C) + C3 * C3 + C3 * A + A * C3
    per_utt = 3 * (2 * C * S) + 2 * C3 * A + 2 * C3 * E
    return 2.0 * (per_frame * T + per_utt)


def synth_wave(batch, seed):
    g = torch.Generator().manual_seed(seed)
    return (0.1 * torch.randn(batch, SAMPLES, generator=g)).clamp_(-1, 1)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write {name: array} as path/<name>.npy, float64 kept as float64 and everything else as float32 (64 MB at most in all)."""
    arrays = {k: np.ascontiguousarray(a, dtype=np.float64 if a.dtype == np.float64 else np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs: {total} bytes > {DUMP_LIMIT_BYTES}"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe), polled through NVML every 50 ms in a
    thread (in-process: an nvidia-smi subprocess needs ~100 ms before its first sample); falls back to nvidia-smi -lms."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.rows = index, None, []
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self._stop = threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown if hasattr(n, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
        while not self._stop.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.mx.append(float(mx))
                r = get_reasons(self.h)
                for k, b in bits.items():
                    if r & b:
                        self.reasons.add(k)
                self.power.append(n.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.05)  # B200_PROFILING.md samples at 200 ms; a 2 ms poll from a Python thread was measured to disturb the host-paced multi-lane pass

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.t.join(timeout=1)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(self.sm),
                    "power_w_max": max(self.power) if self.power else None, "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def bench_config(world):
    """The workload description shared by both arms (the driver compares the two `config` objects)."""
    return {"workload": "ECAPA-TDNN (configs/ecapa_tdnn.yml) Fbank-80 embedding extraction, batch 256 x 3 s @ 16 kHz synthetic audio per GPU (BASELINE configs[1])",
            "batch_per_gpu": BATCH, "global_batch": BATCH * world, "samples": SAMPLES, "frames": FRAMES,
            "parallelism": f"dp{world} (independent utterance shards, no collective)",
            "l2": "two alternating input batches; per-step working set ~2.2 GB >> 126 MB L2"}


def seeded_ecapa_weights():
    """Synthetic ECAPA-TDNN weights of SURVEY.md §8(d) config 2, made by the PACKAGE (ppvector.utils.init), used by both arms."""
    from ppvector.models.ecapa_tdnn import EcapaTdnn
    from ppvector.utils.init import seeded_state_dict
    return seeded_state_dict(EcapaTdnn(input_size=80), seed=1000)


class CpuOracle:
    """The oracle port of the reference CPU path (AudioFeaturizer('Fbank') + EcapaTdnn, fp32, eval) on the host cores.
    PaddlePaddle / paddleaudio cannot be installed offline, so this is cpu_baseline.kind = "port" -- the one place bench.py
    executes oracle/ (the graph it restates is pinned to the reference's own code: tests/test_oracle_vs_reference.py)."""

    def __init__(self):
        from oracle import ecapa as oe
        from oracle import fbank as ofb
        self.oe, self.ofb = oe, ofb
        self.W = seeded_ecapa_weights()

    def step(self, wav):
        """wav: numpy [n, SAMPLES] -> embeddings; per-utterance Fbank loop (featurizer.py:94), model in chunks of 32 (predict.py:265)."""
        with torch.no_grad():
            feat = torch.from_numpy(self.ofb.audio_featurizer_fbank(wav, None, n_mels=80))
            return torch.cat([self.oe.ecapa_forward(feat[i:i + 32], self.W) for i in range(0, len(wav), 32)])

    def calibrate(self, n=16):
        """Pick the intra-op thread count that is fastest for this graph (more threads is not always faster for these small
        convolutions): generous to the baseline.  Returns (threads, utt/s)."""
        cores = os.cpu_count() or 1
        wav = synth_wave(n, 999).numpy()
        best = (cores, 0.0)
        for th in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
            torch.set_num_threads(th)
            self.step(wav[:4])
            t0 = time.perf_counter()
            self.step(wav)
            v = n / (time.perf_counter() - t0)
            if v > best[1]:
                best = (th, v)
        torch.set_num_threads(best[0])
        return best

    def timed_run(self, steps, warmup, budget_s):
        """`warmup` untimed + `steps` timed steps, each step = a bounded sample of n utterances of the 256-utterance workload,
        n chosen from the calibrated rate so that the whole run fits in `budget_s`.  Everything reported was executed."""
        threads, rate = self.calibrate()
        n = int(max(4, min(BATCH, (budget_s * rate) // max(1, steps + warmup))))
        wavs = [synth_wave(n, 1000 + i).numpy() for i in range(2)]
        for i in range(warmup):
            self.step(wavs[i % 2])
        t0 = time.perf_counter()
        for i in range(steps):
            out = self.step(wavs[i % 2])
        dt = time.perf_counter() - t0
        assert torch.isfinite(out).all()
        return {"utt_per_s": n * steps / dt, "ms_per_step": 1000.0 * dt / steps, "n": n, "threads": threads, "seconds": dt}


def run_reference(args, rank, world):
    """--impl reference: rank 0 alone times the CPU path; the other ranks exit 0 without work."""
    if rank != 0:
        return
    r = CpuOracle().timed_run(args.steps, args.warmup, budget_s=float(os.environ.get("PPV_REF_BUDGET_S", "100")))
    v = r["utt_per_s"]
    sample = (f"{r['n']} utterances x 3 s per step (bounded sample of the 256-utterance step), {args.steps} timed + {args.warmup} warm-up steps "
              f"all executed ({r['seconds']:.1f} s timed), oracle port of AudioFeaturizer+EcapaTdnn (torch CPU fp32, {r['threads']} threads); "
              "PaddlePaddle is not installable offline")
    line = {"metric": METRIC, "value": v, "unit": "utterances/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "utterances_per_step": r["n"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": bench_config(world),
            "cpu_baseline": {"value": v, "unit": "utterances/s", "cores": r["threads"], "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the embeddings of the last timed step as DIR/<name>.npy (rank 0, float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the CPU port times a calibrated, machine-dependent sample size)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import ctypes as C
    from ppvector import _lib
    from ppvector.predict import PPVectorPredictor

    assert torch.cuda.is_available(), "bench.py --impl ours needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    import yaml
    cfg = yaml.load(open(os.path.join(ROOT, "configs", "ecapa_tdnn.yml")), Loader=yaml.FullLoader)
    Wts = {k: v.numpy() for k, v in seeded_ecapa_weights().items()}
    pred = PPVectorPredictor(cfg, model_path=None, use_gpu=True, state_dict=Wts)
    pred.predictor.set_precision(args.precision)
    model, fz = pred.predictor, pred._audio_featurizer
    lib = _lib.load()

    # two distinct device-resident batches; working set per step (49 MB waveforms + ~2.2 GB activations) >> 126 MB L2
    wavs = [synth_wave(BATCH, 1000 + rank * 10 + i).to(dev) for i in range(2)]
    host = [synth_wave(BATCH, 2000 + rank * 10 + i).pin_memory() for i in range(2)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ------------------------------------------------------------------------------
    # Pass A, ONE batch at a time with a CUDA event pair around every kernel (ppv_model_profile): the per-kernel times behind `roofline`.
    # Pass B, LANES batches in flight (PPVectorPredictor.embed_resident_stream: replica models on their own streams; the kernels of one
    # batch fill the SMs another batch leaves idle at its kernel tails and between dependent launches): the `value` of the line.
    for i in range(args.warmup):
        emb = model.forward_wav(fz, wavs[i % 2])
    for _e in pred.embed_resident_stream((wavs[i % 2] for i in range(max(args.warmup, 2 * LANES))), lanes=LANES):
        pass
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    _lib.check(lib.ppv_model_profile(model._get_handle(), 1), "ppv_model_profile")
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for i in range(args.steps):
        emb = model.forward_wav(fz, wavs[i % 2])
    a1.record()
    barrier()
    ms_single = a0.elapsed_time(a1)
    g_ms, o_ms, g_n, o_n = C.c_double(), C.c_double(), C.c_int64(), C.c_int64()
    _lib.check(lib.ppv_model_profile_read(model._get_handle(), C.byref(g_ms), C.byref(o_ms), C.byref(g_n), C.byref(o_n)),
               "ppv_model_profile_read")
    _lib.check(lib.ppv_model_profile(model._get_handle(), 0), "ppv_model_profile")
    assert torch.isfinite(emb).all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for last in pred.embed_resident_stream((wavs[i % 2] for i in range(args.steps)), lanes=LANES):  # consumed and dropped: no allocator growth
        pass
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    assert torch.isfinite(last).all() and torch.equal(last, emb)  # the last batch of both passes is the same input: bitwise equal embeddings
    outputs = {}
    if args.dump_outputs and rank == 0:  # host copy outside the timed regions
        outputs["embeddings"] = last.cpu().numpy()
    del last

    # ---- end to end through the public API (host buffers) -----------------------------------------------------
    for out in pred.extract_embeddings_stream((host[i % 2] for i in range(2 * LANES)), lanes=LANES):
        pass
    barrier()
    t0 = time.perf_counter()
    for out in pred.extract_embeddings_stream((host[i % 2] for i in range(args.steps)), lanes=LANES):
        pass
    barrier()
    e2e_s = time.perf_counter() - t0
    assert np.isfinite(out.numpy()).all()
    if args.dump_outputs and rank == 0:
        outputs["e2e_embeddings"] = out.numpy().copy()
        dump_outputs(args.dump_outputs, outputs)

    times = torch.tensor([ms / 1000.0, e2e_s, ms_single / 1000.0], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_s, e2e_s, single_s = times.tolist()
    lanes_s = dev_s

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_sus = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_burst = peaks.get("bf16_tflops", 1700.0)
        # which peak applies: the timed region is short (K steps x ~3 ms); if the SM clock stayed near its maximum the cuBLAS
        # figure measured under the same conditions is the BURST one, a long (power-capped) run compares with the sustained one.
        burst = bool(clk and clk.get("sm_mhz") and clk.get("sm_max_mhz") and clk["sm_mhz"] >= 0.93 * clk["sm_max_mhz"])
        peak_tf = peak_burst if burst else peak_sus
        src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
        peak_src = (f"{src} {'bf16_tflops (burst: SM clock stayed >= 93 % of max during the timed region)' if burst else 'bf16_tflops_sustained (SM clock below 93 % of max during the timed region)'}")
        traffic, traffic_src = None, None
        try:  # per-launch DRAM bytes of the tensor-core kernels from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
            traffic, traffic_src = tj["traffic_bytes_per_launch"], tj["source"]
        except Exception:
            pass
        flops_step = algorithmic_flops_per_utt() * BATCH
        gemm_s_per_step = g_ms.value / 1000.0 / args.steps
        achieved = flops_step / gemm_s_per_step / 1e12
        # `value` is the better of the two timed passes (both are K steps of the same workload; which one wins is a runtime setting of the
        # streaming API: batches in flight).  On an oversubscribed host the multi-lane pass can lose to the single lane; the line says which.
        lanes_used = LANES
        if single_s < dev_s:
            dev_s, lanes_used = single_s, 1
        value = world * BATCH * args.steps / dev_s
        step_tf = flops_step / (dev_s / args.steps) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": "utterances/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * dev_s / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate; fp32-grade)" if args.precision == "bf16x3" else "bf16",
            "data": "synthetic",
            "config": bench_config(world),
            "e2e": {"value": world * BATCH * args.steps / e2e_s, "unit": "utterances/s",
                    "h2d_bytes_per_step": BATCH * SAMPLES * 4, "d2h_bytes_per_step": BATCH * 192 * 4,
                    "api": f"PPVectorPredictor.extract_embeddings_stream(lanes={LANES}) (pinned fp32 waveforms -> H2D on a copy stream -> {LANES} batches in the kernels on {LANES} compute lanes -> embeddings on pinned host memory; every step pays its own H2D + D2H)"},
            "gpu_launches": int(g_n.value + o_n.value),
            "lanes": lanes_used,
            "passes": {"single_lane_ms_per_step": 1000.0 * single_s / args.steps, f"lanes{LANES}_ms_per_step": 1000.0 * lanes_s / args.steps},
            "single_lane": {"value": world * BATCH * args.steps / single_s, "unit": "utterances/s", "ms_per_step": 1000.0 * single_s / args.steps,
                            "note": "one batch at a time on one stream (pass A, the pass the per-kernel events of `roofline` come from); `value` keeps "
                                    f"{LANES} batches in flight (pass B, same kernels and launch count per step, bitwise the same embeddings)"},
            "clocks": clk,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "frac_vs_burst_peak": achieved / peak_burst, "frac_vs_sustained_peak": achieved / peak_sus,
                         "whole_step_tflops": step_tf, "whole_step_frac": step_tf / peak_tf,
                         "peak_burst": peak_burst, "peak_sustained": peak_sus, "sm_mhz_observed": clk.get("sm_mhz") if clk else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "tcgen05 gather-GEMM family: gemm_tcgen05_kernel + res2chain_kernel + asp_fused_kernel (every conv / linear layer)",
                         "launches_per_step": g_n.value / args.steps, "ms_per_step_in_kernel": 1000.0 * gemm_s_per_step,
                         "timed_in": f"pass A ({args.steps} steps, one batch at a time, a CUDA event pair around every kernel on the launching stream); "
                                     "with several batches in flight the kernels of different batches share the SMs and their elapsed times overlap",
                         "other_kernels_ms_per_step": o_ms.value / args.steps,
                         "algorithmic_gflop_per_utt": algorithmic_flops_per_utt() / 1e9,
                         "executed_mma_multiple": 3 if args.precision == "bf16x3" else 1, "peak_source": peak_src},
        }
        if not args.no_cpu_baseline and world == 1:
            r = CpuOracle().timed_run(steps=3, warmup=1, budget_s=20.0)
            line["cpu_baseline"] = {"value": r["utt_per_s"], "unit": "utterances/s", "cores": r["threads"], "kind": "port",
                                    "sample": f"3 timed + 1 warm-up steps of {r['n']} utterances x 3 s ({r['seconds']:.1f} s), oracle port of "
                                              f"AudioFeaturizer+EcapaTdnn (torch CPU fp32, {r['threads']} threads); PaddlePaddle is not installable offline"}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
