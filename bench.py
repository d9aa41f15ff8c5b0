#!/usr/bin/env python
"""Benchmark of the Whisper hot path on B200:  RTFx (audio-seconds / wall-second).

    python bench.py --gpus N --steps K --warmup W                   # this repo's CUDA path, BASELINE configs[2]
    python bench.py --config c2|c3|c4 ...                            # the other single-GPU configs of BASELINE.json
    python bench.py --impl reference --gpus N --steps K --warmup W  # the reference algorithm on the host CPU
    python bench.py ... --dump-outputs DIR                           # also save the last timed step's results

Workloads (BASELINE.json `configs`):
  c3 (default)  large-v3, beam 5, batch 64 per GPU, bf16, kv-cache; one "step" = one pass of the whole hot path over
                one batch of synthetic 30-second segments: log-mel -> AudioEncoder -> cross-K/V -> prefill ->
                (decoder step, logit filters, beam update) x 224 -> finalise / rank.  EOT is suppressed so every segment
                decodes the full 224 tokens (the fixed-length mode of SURVEY.md 8d).
  c2            base.en, greedy, batch 32, fp16 - same step, GreedyDecoder.
  c4            large-v3-turbo, greedy, long-form model.transcribe() over ONE synthetic 1-hour waveform (sequential
                30-second windows, prompt conditioning, natural lengths); one "step" = one transcription of the hour.
                Also reports transcribe_batch() over the same hour cut into 16 files decoded in lock-step.

Multi-GPU (torchrun, one rank per GPU): replicated weights (rank 0 builds them, NCCL broadcast), each rank decodes
its own segments (weak scaling), results all-gathered at the end of every step.

Prints ONE JSON line on rank 0 (keys: see `emit`).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHUNK_S = 30.0
N_SAMPLES = 480000
DECODE_STEPS = 224
PRESETS = {
    # name: (model, batch, beam, dtype, mode)
    "c2": ("base.en", 32, 1, "fp16", "decode"),
    "c3": ("large-v3", 64, 5, "bf16", "decode"),
    "c4": ("turbo", 1, 1, "fp16", "transcribe"),
}
HOUR_S = 3600


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(PRESETS), help="BASELINE.json config (c3 = configs[2], the metric's)")
    ap.add_argument("--model", default=None)
    ap.add_argument("--batch", type=int, default=None, help="segments per GPU per step")
    ap.add_argument("--beam", type=int, default=None)
    ap.add_argument("--dtype", default=None, choices=["bf16", "fp16"])
    ap.add_argument("--decode-steps", type=int, default=DECODE_STEPS)
    ap.add_argument("--audio-seconds", type=int, default=HOUR_S, help="c4: length of the synthetic waveform")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--breakdown", action="store_true",
                    help="after the timed region, run one extra plain-launch step per kernel class with per-launch "
                         "CUDA events and report each class's total device time (diagnostic, not part of `value`)")
    ap.add_argument("--breakdown-ids", default="1,2,3,4,5,6,7,8", help="kernel classes for --breakdown")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64; token rows padded with -1), "
                         "so that two builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    model, batch, beam, dtype, mode = PRESETS[args.config]
    args.model = args.model or model
    args.batch = args.batch or batch
    args.beam = args.beam or beam
    args.dtype = args.dtype or dtype
    args.mode = mode
    return args


def metric_name(args):
    """BASELINE.json's metric string for configs[2]; the other configs are labelled by what they run."""
    if args.mode == "transcribe":
        return f"RTFx (audio-s/wall-s) {args.model} greedy long-form transcribe()"
    beam = f"beam={args.beam}" if args.beam > 1 else "greedy"
    return f"RTFx (audio-s/wall-s) {args.model} {beam}"


def workload_name(args):
    """ONE string for both arms (the driver compares them)."""
    if args.mode == "transcribe":
        return (f"{args.model} greedy long-form transcribe() over one synthetic {args.audio_seconds} s waveform @16 kHz, "
                f"temperature 0, condition_on_previous_text, natural lengths, random-init weights")
    beam = f"beam={args.beam}" if args.beam > 1 else "greedy"
    return (f"{args.model} {beam} batch={args.batch}/GPU synthetic 30 s @16 kHz, kv-cache, {args.decode_steps} decode "
            f"steps per segment (EOT suppressed), random-init weights")


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md 8d / BASELINE.md section 3)
# ------------------------------------------------------------------------------------------------
def algorithmic_numbers(dims, B, G, L_avg):
    d, NL, V, T = dims["n_text_state"], dims["n_text_layer"], dims["n_vocab"], dims["n_audio_ctx"]
    R = B * G
    enc_flops = (2 * 3000 * dims["n_mels"] * d * 3 + 2 * 1500 * d * d * 3
                 + dims["n_audio_layer"] * (2 * 1500 * 12 * d * d + 4 * 1500 * 1500 * d))
    out = {
        "cross_attn_bytes_per_launch": B * T * 2 * d * 2 + 2 * R * d * 2,          # K+V of one layer + q/out
        "decoder_weight_bytes_per_step": 2 * (NL * 14 * d * d + V * d),
        "cross_kv_bytes_per_step": B * NL * 2 * T * d * 2,
        "self_kv_bytes_per_step_avg": int(R * NL * 2 * L_avg * d * 2),
        "kv_append_and_logits_bytes_per_step": R * NL * 2 * d * 2 + R * V * 4,
        "encoder_flops_per_segment": enc_flops,
        "cross_kv_build_flops_per_segment": NL * 2 * (2 * 1500 * d * d),
    }
    out["decode_step_bytes"] = (out["decoder_weight_bytes_per_step"] + out["cross_kv_bytes_per_step"] +
                                out["self_kv_bytes_per_step_avg"] + out["kv_append_and_logits_bytes_per_step"])
    return out


DUMP_LIMIT_BYTES = 64 << 20


def padded_rows(rows):
    """Token lists as one float64 matrix, short rows padded with -1 (token ids are exact in float64)."""
    out = np.full((len(rows), max((len(r) for r in rows), default=0)), -1.0)
    for i, r in enumerate(rows):
        out[i, :len(r)] = r
    return out


def dump_outputs(directory, arrays):
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit; use a smaller workload")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def host_threads() -> int:
    """CPU threads this process may really use: the smallest of os.cpu_count(), the scheduler affinity
    mask and the cgroup CPU quota (the GPU boxes expose 128 logical CPUs to containers with far smaller
    quotas; 128 torch threads on such a box run ~20x slower than 16)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, int(quota / period + 0.5)))
        except Exception:
            pass
    return max(1, min(n, 32))     # torch CPU matmuls stop scaling well before 32 threads on these hosts


# ------------------------------------------------------------------------------------------------
# the reference algorithm (oracle port): bounded samples on the host CPU or, as a library baseline, in torch fp16
# on the GPU (what the reference itself would run there: model.py:44-50 -> cuBLAS, eager attention, Python loop)
# ------------------------------------------------------------------------------------------------
_ORACLE = {}


def oracle_state(model_name, device):
    from oracle import model as OM
    from whisper_b200 import synthetic

    key = (model_name, str(device))
    if key not in _ORACLE:
        dims = synthetic.dims_dict(model_name)
        cpu_key = (model_name, "cpu")
        if cpu_key not in _ORACLE:
            _ORACLE[cpu_key] = dict(dims=dims, W=OM.to_weights(synthetic.synthetic_state_dict(dims, seed=0)),
                                    audio=synthetic.synthetic_audio(1, N_SAMPLES, seed=1234, kind="noise"))
        if key != cpu_key:
            base = _ORACLE[cpu_key]
            _ORACLE[key] = dict(dims=dims, W={k: v.to(device) for k, v in base["W"].items()}, audio=base["audio"])
    return _ORACLE[key]


def oracle_sample(model_name, beam, n_decode_iters, threads, device="cpu", fp16=False, record=None, natural=False):
    """One bounded sample of the reference algorithm: log-mel + encoder on ONE segment + prefill + a few decode iterations,
    extrapolated linearly to the full 224-token window (natural=True: decode to the natural end instead)."""
    from oracle import audio as OA
    from oracle import decoding as OD
    from oracle import model as OM

    torch.set_num_threads(threads)
    st = oracle_state(model_name, device)
    dims, W = st["dims"], st["W"]
    sync = (lambda: torch.cuda.synchronize()) if str(device) != "cpu" else (lambda: None)
    t0 = time.perf_counter()
    mel = torch.from_numpy(OA.log_mel_spectrogram(st["audio"], dims["n_mels"])).to(device)
    if fp16:
        mel = mel.half()                                                   # decoding.py:645-646
    sync()
    t_mel = time.perf_counter() - t0
    t0 = time.perf_counter()
    with torch.no_grad():
        feats = OM.encoder_forward(W, dims, mel)
    sync()
    t_enc = time.perf_counter() - t0
    ids = OD.token_ids(dims["n_vocab"])
    timings = []
    opt = dict(beam_size=beam if beam > 1 else None)
    if natural:
        opt.update(sample_len=None)
    else:
        opt.update(sample_len=DECODE_STEPS, suppress_tokens=(-1, ids.eot))
    with torch.no_grad():
        res = OD.decode(W, dims, feats, OD.Options(**opt), max_steps=None if natural else 1 + n_decode_iters,
                        timings=timings, record=record)
    sync()
    t_prefill = timings[0]
    t_step = float(np.mean(timings[1:])) if len(timings) > 1 else timings[0]
    n_steps = len(timings) if natural else DECODE_STEPS
    total = t_mel + t_enc + t_prefill + (n_steps - 1) * t_step
    return {"rtfx": CHUNK_S / total, "t_mel": t_mel, "t_enc": t_enc, "t_prefill": t_prefill, "t_step": t_step,
            "wall": t_mel + t_enc + sum(timings), "feats": feats, "tokens": res[0].tokens, "n_steps": n_steps,
            "t_window": total}


def reference_value(args, threads, record=None):
    """RTFx of the reference algorithm on the host CPU for this workload, from one bounded sample."""
    if args.mode == "transcribe":
        # one 30-second window decoded to its natural end (greedy, turbo: 4 decoder layers); the window loop of
        # transcribe() is sequential, so the hour costs (number of windows) x (one window)
        s = oracle_sample(args.model, 1, 0, threads, natural=True)
        s["rtfx"] = CHUNK_S / s["t_window"]
        s["sample"] = (f"oracle port (fp32, torch CPU, {threads} threads): ONE 30 s window of the hour - log-mel + encoder + "
                       f"greedy decode to its natural end ({s['n_steps']} tokens; enc {s['t_enc']:.2f}s, prefill "
                       f"{s['t_prefill']:.2f}s, {s['t_step']:.3f}s/token), hour = windows x window")
        return s
    n_iters = 3
    s = oracle_sample(args.model, args.beam, n_iters, threads, record=record)
    what = f"beam-{args.beam}" if args.beam > 1 else "greedy"
    s["sample"] = (f"oracle port (fp32, torch CPU, {threads} threads): log-mel + encoder on 1 of {args.batch} segments + "
                   f"prefill + {n_iters} {what} iterations, extrapolated linearly to {DECODE_STEPS} (enc {s['t_enc']:.2f}s, "
                   f"prefill {s['t_prefill']:.2f}s, {s['t_step']:.3f}s/iter; {s['wall']:.1f}s of CPU work); the reference "
                   f"decodes beam-search segments one at a time (decoding.py:734,740)")
    return s


def run_reference_arm(args, rank):
    """The reference's algorithm on the host CPU (oracle port; the Python reference itself cannot travel
    to the GPU box).  Rank 0 only."""
    if rank != 0:
        return
    threads = host_threads()
    for _ in range(args.warmup):
        reference_value(args, threads)
    t0 = time.perf_counter()
    vals = [reference_value(args, threads) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    v = float(np.mean([x["rtfx"] for x in vals]))
    print(json.dumps({
        "impl": "reference", "metric": metric_name(args), "value": v, "unit": "x realtime", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * wall / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "impl_detail": "oracle port on host CPU; ms_per_step is the time "
                   "of the bounded sample, value is extrapolated from it (see cpu_baseline.sample)"},
        "cpu_baseline": {"value": v, "unit": "x realtime", "cores": threads, "kind": "port", "sample": vals[-1]["sample"]},
        "e2e": {"value": v, "unit": "x realtime", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def gpu_torch_baseline(args, dev):
    """The same port in torch eager on THIS GPU with fp16 activations (the path the reference takes on CUDA:
    fp32 parameters cast per call, cuBLAS GEMMs, eager attention, Python-driven loop with per-candidate .item() syncs)."""
    try:
        natural = args.mode == "transcribe"
        beam = 1 if natural else args.beam
        oracle_sample(args.model, beam, 2, host_threads(), device=dev, fp16=True, natural=False)      # warm-up
        s = oracle_sample(args.model, beam, 6, host_threads(), device=dev, fp16=True, natural=natural)
        v = CHUNK_S / s["t_window"]
        return {"value": v, "unit": "x realtime", "kind": "oracle port in torch eager fp16 on the same GPU (library kernels)",
                "sample": (f"1 segment: enc {s['t_enc'] * 1e3:.1f} ms, prefill {s['t_prefill'] * 1e3:.1f} ms, "
                           f"{s['t_step'] * 1e3:.2f} ms/iteration x {s['n_steps']}; segments run one at a time like the "
                           f"reference's beam search")}
    except Exception as e:                                             # a baseline must never break the bench line
        return {"value": None, "error": f"{type(e).__name__}: {e}"[:300]}
    finally:
        for k in [k for k in _ORACLE if k[1] != "cpu"]:
            del _ORACLE[k]
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------
def elapsed_by_phase(timing):
    """Sum the CUDA-event marks decode() left in model.timing into per-phase milliseconds."""
    marks = timing.get("marks", [])
    out = {}
    for (name, ev), (_, nxt) in zip(marks, marks[1:]):
        if name in ("end", "encoder_end"):
            continue
        out[name] = out.get(name, 0.0) + ev.elapsed_time(nxt)
    return out


def main():
    args = parse()
    from whisper_b200 import parallel

    if args.impl == "reference":
        run_reference_arm(args, int(os.environ.get("RANK", "0")))
        return

    import torch.distributed as dist

    import whisper_b200 as wb
    from whisper_b200 import _lib, synthetic

    rank, world, local = parallel.init_from_env("nccl" if int(os.environ.get("WORLD_SIZE", "1")) > 1 else None)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    dims = synthetic.dims_dict(args.model)
    B, G = args.batch, args.beam

    # ---- weights: rank 0 builds the synthetic checkpoint, NCCL broadcast, every rank packs its replica
    spec = [(n, s) for n, s, _ in synthetic.state_dict_spec(dims)]
    sd = synthetic.synthetic_state_dict(dims, seed=0) if rank == 0 else None
    sd_dev = parallel.broadcast_state_dict(sd, spec, dev)
    model = wb.Whisper(wb.ModelDimensions(**dims), sd_dev, device=dev, dtype=dtype)
    del sd, sd_dev
    torch.cuda.empty_cache()
    tok = wb.tokenizer.get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en",
                                     task="transcribe")
    lib = _lib.lib()

    def timed(fn, k):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(k):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    peak_src = "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s / 1400 TFLOP/s (of fallback)"

    if args.mode == "transcribe":
        return bench_transcribe(args, model, tok, dims, dev, rank, world, local, timed, lib, peak_gbs, peak_src)

    # ---- inputs: B x 30 s of synthetic 16 kHz audio per rank (pinned host copy + device copy)
    audio_host = torch.from_numpy(synthetic.synthetic_audio(B, N_SAMPLES, seed=1234 + rank, kind="noise")).pin_memory()
    audio_dev = audio_host.to(dev)
    opt_kwargs = dict(beam_size=G if G > 1 else None, sample_len=args.decode_steps, suppress_tokens=[-1, tok.eot])
    options = wb.DecodingOptions(language="en", **opt_kwargs)

    def hot_path(audio):
        mel = wb.log_mel_spectrogram(audio, dims["n_mels"], per_waveform_max=True)   # each segment = its own file
        res = model.decode(mel, options)
        return parallel.gather_results([r.tokens for r in res], [r.avg_logprob for r in res],
                                       [r.no_speech_prob for r in res], dev)

    def step_resident():
        return hot_path(audio_dev)

    def step_e2e():
        return hot_path(audio_host.to(dev, non_blocking=True))

    for _ in range(max(3, args.warmup)):
        out = step_resident()
    n_tokens = [len(t) for t in out[0]]

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    model.timing = {}
    ms, out = timed(step_resident, args.steps)
    phases = elapsed_by_phase(model.timing)
    loop_steps = sum(model.timing.get("loop_steps", [0]))
    model.timing = None
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        toks, lps, nss = out
        dump_outputs(args.dump_outputs, {"tokens": padded_rows(toks), "avg_logprob": lps, "no_speech_prob": nss})

    # roofline of the dominant kernel (decoder-step cross-attention): one more step with every launch of
    # that kernel bracketed by CUDA events on its stream.  This pass runs the decode loop as plain launches
    # (the timed steps above replay it from CUDA graphs, where per-launch events cannot be interleaved).
    lib.wb200_profile_enable(1)
    ms_prof, _ = timed(step_resident, 1)
    prof_ms, prof_n = ctypes.c_double(0), ctypes.c_int64(0)
    lib.wb200_profile_read(ctypes.byref(prof_ms), ctypes.byref(prof_n))
    lib.wb200_profile_enable(0)

    breakdown = None
    if args.breakdown:
        names = {1: "cross_attention", 2: "self_attention", 3: "gemm", 4: "encoder_attention", 5: "layernorm",
                 6: "select", 7: "log_mel", 8: "decoder_layer_fused"}
        breakdown = {}
        for kid, name in names.items():
            if str(kid) not in args.breakdown_ids.split(","):
                continue
            lib.wb200_profile_enable(kid)
            ms_k, _ = timed(step_resident, 1)
            t_k, n_k = ctypes.c_double(0), ctypes.c_int64(0)
            lib.wb200_profile_read(ctypes.byref(t_k), ctypes.byref(n_k))
            lib.wb200_profile_enable(0)
            breakdown[name] = {"ms": t_k.value, "launches": int(n_k.value), "step_ms": ms_k}

    e2e_steps = max(1, min(args.steps, 3))
    step_e2e()
    ms_e2e, _ = timed(step_e2e, e2e_steps)

    if rank != 0:
        return
    audio_s = world * B * CHUNK_S
    value = audio_s * args.steps / (ms / 1000.0)
    e2e_value = audio_s * e2e_steps / (ms_e2e / 1000.0)
    L_avg = len(tok.sot_sequence) + args.decode_steps / 2
    alg = algorithmic_numbers(dims, B, G, L_avg)
    avg_launch_ms = prof_ms.value / max(1, prof_n.value)
    achieved = alg["cross_attn_bytes_per_launch"] / (avg_launch_ms / 1000.0) / 1e9 if avg_launch_ms > 0 else 0.0
    R = B * G
    ctx = dims["n_text_ctx"]
    d2h = R * (len(tok.sot_sequence) + args.decode_steps) * 4 + R * 4 + B * 4 + 4 + \
        (B * G * ctx * 4 + 3 * B * G * 4 if G > 1 else 0)
    ms_loop_step = phases.get("decode_loop", 0.0) / max(1, loop_steps)
    step_gbs = alg["decode_step_bytes"] / (ms_loop_step / 1000.0) / 1e9 if ms_loop_step > 0 else 0.0
    ms_enc = phases.get("encoder", 0.0) / args.steps
    enc_tf = B * alg["encoder_flops_per_segment"] / (ms_enc / 1000.0) / 1e12 if ms_enc > 0 else 0.0
    line = {
        "metric": metric_name(args), "value": value, "unit": "x realtime", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {
            "workload": workload_name(args),
            "baseline_config": {"c3": "BASELINE.json configs[2]", "c2": "BASELINE.json configs[1]"}.get(args.config, "custom")
            if (args.model, G, B) == PRESETS[args.config][:3] else "custom",
            "parallelism": f"dp{world} (replicated weights, segments sharded, no per-step collective)",
            "l2": "per-step working set (cross-K/V + self-K/V) far exceeds the 126 MB L2; no flush needed",
            "tokens_per_segment": int(np.mean(n_tokens)),
            "fused_decoder_layer": os.environ.get("WB200_FUSED_LAYER", "1") != "0",
        },
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "x realtime", "h2d_bytes_per_step": B * N_SAMPLES * 4,
                "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps},
        "gpu_launches": int(launches),
        "phases_ms_per_step": {k: v / args.steps for k, v in phases.items()},
        "roofline": {
            "kernel": "cross_attention_kernel (decoder step, one launch per layer per step)",
            "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
            "frac": achieved / peak_gbs if peak_gbs else None, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg["cross_attn_bytes_per_launch"],
            "avg_launch_ms": avg_launch_ms, "launches_timed": int(prof_n.value),
            "share_of_step": (prof_ms.value / ms_prof) if ms_prof > 0 else None,
            "profiled_step_ms": ms_prof,
            "how": "CUDA events around every launch of the kernel on its stream, one extra (non-graph) step",
            "traffic": None,
        },
        # the two fractions BASELINE.json's metric names: the whole decoder step against HBM, the encoder against the
        # tensor pipe (CUDA events around the decode loop / the encoder inside the timed region)
        "roofline_decode_step": {
            "bound": "hbm", "achieved": step_gbs, "peak": peak_gbs, "unit": "GB/s", "frac": step_gbs / peak_gbs if peak_gbs else None,
            "algorithmic_bytes_per_step": alg["decode_step_bytes"], "ms_per_decode_step": ms_loop_step,
            "decode_steps_timed": int(loop_steps),
            "how": "weights + cross-K/V (once per audio) + self-K/V at the mean length + kv append + fp32 logits, divided "
                   "by the CUDA-event time of the device-resident decode loop (graph replay) per iteration"},
        "roofline_encoder": {
            "bound": "tensor", "achieved": enc_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": enc_tf / peak_tf if peak_tf else None,
            "flops": B * alg["encoder_flops_per_segment"], "ms": ms_enc,
            "how": "conv stem + 32 blocks + ln_post FLOPs (SURVEY 8d) / CUDA-event time of AudioEncoder.forward inside the "
                   "timed region; peak = sustained cuBLAS bf16"},
        "algorithmic": alg,
    }
    if breakdown is not None:
        line["breakdown"] = breakdown
    rec = {}
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        s = reference_value(args, threads, record=rec)
        line["cpu_baseline"] = {"value": s["rtfx"], "unit": "x realtime", "cores": threads, "kind": "port", "sample": s["sample"]}
        if not args.no_parity:
            line["parity_check"] = parity_check(args, model, wb, audio_dev, dims, opt_kwargs, rec, s, dtype)
    if world == 1 and not args.no_gpu_baseline:
        line["gpu_torch_baseline"] = gpu_torch_baseline(args, dev)
    print(json.dumps(line))


def parity_check(args, model, wb, audio_dev, dims, opt_kwargs, rec, sample, dtype):
    """Segment 0 of the timed batch against the oracle sample the CPU baseline just ran: encoder features, then the
    decoder teacher-forced along the oracle's trajectory (device logits of every iteration, exact tokens / beam
    parents / score sums), then free-running with the measured-error gate (oracle/parity.py)."""
    from oracle import parity

    tol = {torch.float16: 5e-3, torch.bfloat16: 4e-2}[dtype]
    out = {"segment": 0, "logit_tol": tol}
    try:
        mel = wb.log_mel_spectrogram(audio_dev[:1], dims["n_mels"], per_waveform_max=True)
        g_feats = model.embed_audio(mel)
        err = (g_feats.float().cpu() - sample["feats"].float()).abs()
        out.update(feature_err_max=float(err.max()), feature_err_mean=float(err.mean()))
        rec["options"] = __import__("oracle.decoding", fromlist=["Options"]).Options(
            beam_size=opt_kwargs["beam_size"], sample_len=opt_kwargs["sample_len"], suppress_tokens=tuple(opt_kwargs["suppress_tokens"]))
        forced = parity.teacher_forced(model, opt_kwargs, 1, g_feats, rec, tol)
        out.update(iterations=forced["steps"], beam_reorders=forced["reorders"], logit_rel_err_max=forced["worst_rel_logit_err"],
                   tokens_parents_scores_exact=True)
        free = parity.free_running(model, opt_kwargs, 1, g_feats, rec, dims)
        out.update(free_running_asserted=free["asserted_steps"], ok=True)
    except AssertionError as e:
        out.update(ok=False, error=str(e)[:300])
    return out


def bench_transcribe(args, model, tok, dims, dev, rank, world, local, timed, lib, peak_gbs, peak_src):
    """c4: model.transcribe() over one synthetic hour (sequential windows) + transcribe_batch() over the same hour cut
    into 16 files (lock-step).  Replicas only across GPUs: every rank transcribes its own hour."""
    import whisper_b200 as wb
    from whisper_b200 import _lib, synthetic

    n = args.audio_seconds * 16000
    audio_host = torch.from_numpy(synthetic.synthetic_audio(1, n, seed=1234 + rank, kind="speechlike")[0]).pin_memory()
    audio_dev = audio_host.to(dev)
    kw = dict(temperature=0.0, condition_on_previous_text=True, language="en")

    def run(audio):
        return model.transcribe(audio, **kw)

    for _ in range(max(1, min(args.warmup, 3))):
        res = run(audio_dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    model.timing = {}
    ms, res = timed(lambda: run(audio_dev), args.steps)
    phases = elapsed_by_phase(model.timing)
    loop_steps = sum(model.timing.get("loop_steps", [0]))
    n_decodes = len(model.timing.get("loop_steps", []))
    model.timing = None
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        segs = res["segments"]
        dump_outputs(args.dump_outputs, {"tokens": padded_rows([s["tokens"] for s in segs]),
                                         **{k: [s[k] for s in segs] for k in ("seek", "start", "end", "temperature",
                                                                             "avg_logprob", "compression_ratio",
                                                                             "no_speech_prob")}})
    e2e_steps = max(1, min(args.steps, 2))
    ms_e2e, _ = timed(lambda: run(audio_host.to(dev, non_blocking=True)), e2e_steps)
    # lock-step over 16 files of the same total duration
    n_files = 16
    piece = n // n_files
    files = [audio_dev[i * piece:(i + 1) * piece] for i in range(n_files)]
    model.transcribe_batch = lambda a: wb.transcribe_batch(model, a, **kw)
    model.transcribe_batch(files)
    ms_b, res_b = timed(lambda: model.transcribe_batch(files), max(1, min(args.steps, 2)))
    ms_b /= max(1, min(args.steps, 2))
    if rank != 0:
        return
    windows = len({s["seek"] for s in res["segments"]})
    tokens = sum(len(s["tokens"]) for s in res["segments"])
    value = world * args.audio_seconds * args.steps / (ms / 1000.0)
    line = {
        "metric": metric_name(args), "value": value, "unit": "x realtime", "n_gpus": world, "steps": args.steps,
        "warmup": max(1, min(args.warmup, 3)), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": workload_name(args), "baseline_config": "BASELINE.json configs[3]",
                   "parallelism": f"replicas only x{world} (one file's window loop is sequential: transcribe.py:272-508)",
                   "decode_calls_per_hour": n_decodes // max(1, args.steps), "windows_with_segments": windows,
                   "tokens_per_hour": tokens, "decoder_iterations_per_hour": loop_steps // max(1, args.steps),
                   "l2": "batch-1 decode: the working set (weights 0.3 GB + one audio's K/V) exceeds L2; no flush needed"},
        "clocks": clocks,
        "e2e": {"value": world * args.audio_seconds * e2e_steps / (ms_e2e / 1000.0), "unit": "x realtime",
                "h2d_bytes_per_step": n * 4, "d2h_bytes_per_step": int(tokens * 4 + n_decodes / max(1, args.steps) * 64),
                "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps},
        "gpu_launches": int(launches),
        "phases_ms_per_step": {k: v / args.steps for k, v in phases.items()},
        "transcribe_batch": {"files": n_files, "seconds_each": piece / 16000.0, "value": args.audio_seconds / (ms_b / 1000.0),
                             "unit": "x realtime", "ms": ms_b, "rounds": res_b[0].get("rounds"),
                             "note": "the same hour as 16 files advanced in lock-step (SURVEY 8f.1)"},
    }
    # HBM roofline of the batch-1 decoder iteration: every iteration streams the decoder's weights, the logits matrix and
    # the window's cross K/V once; the mean self-attention history is tokens / decode call / 2
    iters = loop_steps / max(1, args.steps)
    alg = algorithmic_numbers(dims, 1, 1, max(1.0, tokens / max(1, n_decodes / max(1, args.steps)) / 2.0))
    loop_ms = phases.get("decode_loop", 0.0) / args.steps
    ach = alg["decode_step_bytes"] * iters / (loop_ms / 1000.0) / 1e9 if loop_ms > 0 else None
    line["roofline"] = {"kernel": "decoder iteration (one audio, greedy): 3 fused-layer launches + 2 attention launches per layer, "
                                  "logits GEMM, selection", "bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s",
                        "frac": (ach / peak_gbs) if ach else None, "peak_source": peak_src, "traffic": None,
                        "algorithmic_bytes_per_iteration": alg["decode_step_bytes"],
                        "us_per_iteration": 1000.0 * loop_ms / max(1.0, iters),
                        "how": "weights of the decoder layers + logits matrix + the window's cross K/V + mean self K/V, x iterations, "
                               "divided by the CUDA-event time of the device-resident decode loops of the hour"}
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        s = reference_value(args, threads)
        line["cpu_baseline"] = {"value": s["rtfx"], "unit": "x realtime", "cores": threads, "kind": "port", "sample": s["sample"]}
    if world == 1 and not args.no_gpu_baseline:
        line["gpu_torch_baseline"] = gpu_torch_baseline(args, dev)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
