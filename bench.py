#!/usr/bin/env python
"""bench.py -- the reference's headline metric on the reference's headline config (BASELINE.json):
real-time factor (RTFx = audio seconds / wall seconds, Sources/Tools/mlx-audio-swift-tts/App.swift:204)
of Orpheus-3B TTS, batch 8 x 64-token prompt -> 512 audio tokens -> SNAC decode, per B200; beside it, in the same
JSON line, BASELINE.json's other half of the metric (Whisper-base STT, config 3) and the SNAC decode (config 2).

A "step" is one pass of the hot path over one batch: 8 prompts -> prefill -> 512 decode steps (EOS masked so
work is fixed) -> parseOutput / 7-token de-interleave -> SNAC decode -> 8 waveforms.  The synthetic 64-token prompt
ends with START_OF_SPEECH (128257, the first token a real checkpoint emits), so parseOutput crops the prompt as it
does in a real run and the audio is BASELINE.md's 512 tokens -> 73 frames -> 6.229 s per utterance.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--scaling weak|strong] [--dump-outputs DIR]
    torchrun ... bench.py --gpus N ...          (one rank per GPU; utterances shard)

Every block times K steps.  --dump-outputs DIR writes, after the timed steps, what each timed device path returned to its caller
in its last step on rank 0 (DIR/<name>.npy: floating outputs as float32, integer ones as float64).  Inputs and weights are seeded,
so two builds run with the same arguments can be compared output for output (DESIGN.md 5: which outputs repeat bit for bit).

`value` : inputs already resident in HBM, waveforms left in HBM (b2a_tts_generate_dev).
`e2e`   : same metric through the host-buffer C ABI call a user makes (b2a_tts_generate): pinned host ids
          in, waveforms copied back to pinned host memory, inside the timed region.
`whisper` / `snac` : secondary blocks with their own value / e2e / roofline (and cpu_baseline for Whisper at N=1).
Timed with CUDA events on the stream the library launches on; max over ranks; rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

ORPHEUS = dict(hidden_size=3072, num_hidden_layers=28, intermediate_size=8192, num_attention_heads=24,
               num_key_value_heads=8, head_dim=128, vocab_size=156940, rms_norm_eps=1e-5, rope_theta=500000.0,
               tie_word_embeddings=True,
               rope_scaling={"rope_type": "llama3", "factor": 32.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                             "original_max_position_embeddings": 8192})
BATCH, PROMPT_LEN, GEN_TOKENS = 8, 64, 512
METRIC, UNIT = "orpheus3b_tts_rtfx_batch8", "x_realtime(audio_s/s)"


def workload_name(cfg=ORPHEUS):
    return (f"Orpheus-3B bf16 (hidden {cfg['hidden_size']} x {cfg['num_hidden_layers']} layers, vocab {cfg['vocab_size']}), "
            f"{PROMPT_LEN}-token prompt, {GEN_TOKENS} audio tokens, batch {BATCH}, SNAC-24kHz decode")


def frames_per_utterance(n_gen: int = GEN_TOKENS) -> int:
    # parseOutput crops everything up to the last 128257 (the prompt's final token), keeps the generated codes:
    # floor(G / 7) frames (LlamaTTS.swift:383-434) -> BASELINE.md: 512 tokens -> 73 frames
    return n_gen // 7


def audio_seconds_per_utterance(n_gen: int = GEN_TOKENS) -> float:
    return frames_per_utterance(n_gen) * 4 * 512 / 24000.0            # 2048 samples per frame at 24 kHz: 6.229 s


def make_prompts(rank: int, rows: int = BATCH) -> np.ndarray:
    """[SOH] body [EOT, EOH] as prepareInputIds frames it (LlamaTTS.swift:446-553), then START_OF_SPEECH -- the first token a
    real checkpoint generates -- so that parseOutput crops the prompt exactly as in a real run (VERDICT r1 / ADVICE r1)."""
    rng = np.random.default_rng(3 + rank)
    ids = np.empty((rows, PROMPT_LEN), dtype=np.int32)
    ids[:, 0] = 128259
    ids[:, 1:-3] = rng.integers(0, 128000, size=(rows, PROMPT_LEN - 4), dtype=np.int32)
    ids[:, -3], ids[:, -2], ids[:, -1] = 128009, 128260, 128257
    return ids


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thr = index, [], None, None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "400"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        self.thr = threading.Thread(target=self._read, daemon=True)
        self.thr.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s: the sustained figure (the encoder / prefill GEMMs run inside a long step)."""
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        if "bf16_tflops_sustained" in d:
            return float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1450.0, "fallback (B200_PROFILING.md sustained cuBLAS bf16)"


def weight_bytes(cfg) -> int:
    H, I, hd = cfg["hidden_size"], cfg["intermediate_size"], cfg["head_dim"]
    nq, nkv, L, V = cfg["num_attention_heads"], cfg["num_key_value_heads"], cfg["num_hidden_layers"], cfg["vocab_size"]
    per_layer = (nq + 2 * nkv) * hd * H + H * nq * hd + 3 * I * H
    return 2 * (L * per_layer + V * H)        # every matrix once + the tied lm head; bf16


KV_ELEM_BYTES_BUILT = 4      # the cache this library keeps is fp32 (DESIGN.md 3.3); SURVEY.md 8(d) counts a bf16 cache


def kv_bytes(cfg, batch, ctx, elem_bytes: int = 2) -> int:
    """K and V read by one decode step at context ctx.  elem_bytes = 2 is SURVEY.md 8(d)'s definition (bf16 cache): the roofline
    numerator uses THAT, so the fp32 cache's extra traffic is not credited as useful bytes."""
    return 2 * batch * cfg["num_key_value_heads"] * ctx * cfg["head_dim"] * elem_bytes * cfg["num_hidden_layers"]


# dram__bytes_read.sum + dram__bytes_write.sum over the 144 launches of ONE decode step (batch 8, context 320), from
# `ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none python tools/profile_step.py 320 3`
# on the B200 (profiles/r02_decode_step_dram.csv, summary profiles/r02_decode_step_dram.md)
MEASURED_STEP_DRAM_BYTES = {"context": 320, "batch": 8, "bytes": 7244129280}


# ------------------------------------------------------------------------------------------------- CPU legs
def usable_cpus() -> int:
    """Hardware threads this process may really run on: the scheduler affinity mask capped by the cgroup CPU quota.
    (os.cpu_count() reports the HOST's count; inside a quota-limited container, asking torch for that many threads
    oversubscribes the cores it actually has and slows the CPU arm down many times over.)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                                     # cgroup v2: "max 100000" or "<quota> <period>"
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.999)))
    except (OSError, ValueError):
        try:                                                 # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and per > 0:
                n = min(n, max(1, (q + per - 1) // per))
        except (OSError, ValueError):
            pass
    return max(1, n)


class CpuReference:
    """The reference path restated on the CPU (oracle/, kind "port"), as a BOUNDED sample per call.
    Weights (full width, 4 layers + the tied embedding) are built once.  One sample times: the prefill on a 16-token prompt
    (x 4 = 64 tokens, linear in tokens) and one decode step, each on a 2- and a 4-layer model to separate the per-layer cost from
    the lm head, extrapolated to 28 layers x (64-token prefill + 512 steps); and the SNAC decode of a quarter of one utterance's
    frames (x 4 x 8 utterances, linear in frames)."""

    PREFILL_TOKENS, SNAC_DIV = 16, 4

    def __init__(self, cfg, threads: int):
        """threads = the most the process may use (usable_cpus()); the count actually used is the fastest of a short calibration
        over {threads, threads/2, threads/4, ...} on the decode step (see calibrate) and is what `cores` reports."""
        import torch
        from oracle import llama as ol
        from oracle import snac as osn
        torch.set_num_threads(threads)
        self.cfg, self.threads, self.ol, self.osn, self.torch = cfg, threads, ol, osn, torch
        self.max_threads, self.calibration = threads, ""
        g = torch.Generator().manual_seed(0)
        H, I, hd = cfg["hidden_size"], cfg["intermediate_size"], cfg["head_dim"]
        nq, nkv, V = cfg["num_attention_heads"], cfg["num_key_value_heads"], cfg["vocab_size"]

        def lin(o, i):
            return torch.randn(o, i, generator=g) * 0.02      # fp32 (bf16-valued weights pre-widened once)

        W = {"model.embed_tokens.weight": lin(V, H), "model.norm.weight": torch.ones(H)}
        for l in range(4):
            p = f"model.layers.{l}."
            W[p + "self_attn.q_proj.weight"] = lin(nq * hd, H)
            W[p + "self_attn.k_proj.weight"] = lin(nkv * hd, H)
            W[p + "self_attn.v_proj.weight"] = lin(nkv * hd, H)
            W[p + "self_attn.o_proj.weight"] = lin(H, nq * hd)
            W[p + "mlp.gate_proj.weight"] = lin(I, H)
            W[p + "mlp.up_proj.weight"] = lin(I, H)
            W[p + "mlp.down_proj.weight"] = lin(H, I)
            W[p + "input_layernorm.weight"] = torch.ones(H)
            W[p + "post_attention_layernorm.weight"] = torch.ones(H)
        self.W = W
        self.scfg = osn.SNACConfig()
        self.SW = osn.init_weights(self.scfg, 1234)
        self.calibrate()

    def calibrate(self):
        """Pick the thread count that makes the CPU arm FASTEST: the decode step (the dominant term, 512 of them) of the 2-layer
        model is timed at max, max/2, max/4, ... threads (down to 4) and the best count is kept for everything."""
        torch = self.torch
        cands, n = [], self.max_threads
        while n >= 4:
            cands.append(n)
            n //= 2
        if not cands:
            cands = [self.max_threads]
        mo = self.ol.LlamaOracle(self._build(2), self.W, round_acts=True)
        ids = torch.as_tensor(make_prompts(0)[:, :2], dtype=torch.long)
        nxt = mo.forward(ids)[:, -1].argmax(-1, keepdim=True)
        best, seen = None, []
        for c in cands:
            torch.set_num_threads(c)
            mo.forward(nxt)                                   # settle the pool at this size
            ts = []
            for _ in range(3):                                # median of three: one timing is too noisy on a shared host
                t0 = time.perf_counter()
                mo.forward(nxt)
                ts.append(time.perf_counter() - t0)
            dt = float(np.median(ts))
            seen.append(f"{c}: {dt * 1e3:.0f}ms")
            if best is None or dt < best[1]:
                best = (c, dt)
        self.threads = best[0]
        torch.set_num_threads(self.threads)
        self.calibration = f"thread count chosen by timing one 2-layer decode step at {{{', '.join(seen)}}} of {self.max_threads} usable"

    def _build(self, nl):
        c = self.cfg
        return self.ol.LlamaConfig(hidden_size=c["hidden_size"], num_hidden_layers=nl, intermediate_size=c["intermediate_size"],
                                   num_attention_heads=c["num_attention_heads"], num_key_value_heads=c["num_key_value_heads"],
                                   head_dim=c["head_dim"], vocab_size=c["vocab_size"])

    STEP_REPS, PREFILL_REPS = 5, 2

    def sample(self, light: bool = False):
        """-> (RTFx, total seconds extrapolated, description).  light=True (warm-up samples): one decode step only.
        Every timing inside a sample is a MEDIAN (decode step: 5 repeats, prefill: 2) at the fixed, calibrated thread count, so the
        reference arm does not move 2x between runs on a shared host (VERDICT r1 weak #8)."""
        torch, ol, osn = self.torch, self.ol, self.osn
        L_full = self.cfg["num_hidden_layers"]
        ids = torch.as_tensor(make_prompts(0)[:, :self.PREFILL_TOKENS], dtype=torch.long)
        # two DIRECT measurements, no difference of near-equal numbers (that made the round-1 arm move 2x between runs):
        #   layers: the 4-layer model with the lm head switched off (head_positions=[])  -> per-layer cost = t / 4
        #   head  : a 0-layer model (embedding, final norm, tied lm head on every position, as the reference's graph evaluates it)
        def timed_pair(nl, head):
            mo = ol.LlamaOracle(self._build(nl), self.W, round_acts=True)
            kw = {} if head else {"head_positions": []}
            pre_ids = ids if not light else ids[:, :2]
            tp = []
            for _ in range(1 if light else self.PREFILL_REPS):
                mo.reset()
                t0 = time.perf_counter()
                mo.forward(pre_ids, **kw)
                tp.append(time.perf_counter() - t0)
            nxt = pre_ids[:, -1:]
            td = []
            for _ in range(1 if light else self.STEP_REPS):
                t0 = time.perf_counter()
                mo.forward(nxt, **kw)
                td.append(time.perf_counter() - t0)
            return float(np.median(tp)) * (PROMPT_LEN / pre_ids.shape[1]), float(np.median(td))

        lay_pre, lay_dec = timed_pair(4, head=False)
        head_pre, head_dec = (0.0, 0.0) if light else timed_pair(0, head=True)
        per_layer_pre, per_layer_dec = lay_pre / 4, lay_dec / 4
        res = {4: (lay_pre + head_pre, lay_dec + head_dec)}
        t_prefill = L_full * per_layer_pre + head_pre
        t_step = L_full * per_layer_dec + head_dec
        frames = frames_per_utterance()
        fsub = max(frames // self.SNAC_DIV, 1) if not light else 1
        osn.DTYPE = torch.float32
        codes = osn.synth_codes(self.scfg, 1, 4 * fsub, seed=2)
        t0 = time.perf_counter()
        osn.decode(self.scfg, self.SW, codes, None)
        t_snac1 = (time.perf_counter() - t0) * frames / fsub
        osn.DTYPE = torch.float64
        total = t_prefill + GEN_TOKENS * t_step + BATCH * t_snac1
        audio = BATCH * audio_seconds_per_utterance()
        desc = (f"oracle port (torch-CPU fp32 math on bf16-valued weights, {self.threads} threads fixed, {self.calibration}): full-width 4-layer stack (lm head off) and 0-layer model (embedding + norm + tied lm head) timed directly, "
                f"every timing a median (decode step x{self.STEP_REPS}, prefill x{self.PREFILL_REPS}) "
                f"(prefill of {self.PREFILL_TOKENS} of {PROMPT_LEN} prompt tokens x batch {BATCH}: {res[4][0]:.2f}s scaled / decode step "
                f"{res[4][1]*1e3:.0f}ms at 4 layers + head), per-layer + lm-head cost extrapolated linearly to {L_full} layers x "
                f"({PROMPT_LEN}-token prefill + {GEN_TOKENS} steps); SNAC decode timed on {fsub} of {frames} frames of 1 of {BATCH} "
                f"utterances ({t_snac1:.2f}s scaled) x {BATCH}")
        return audio / total, total, desc


def cpu_reference_sample(cfg, threads: int, n: int = 3):
    """-> (RTFx, total seconds, description, threads actually used): the MEDIAN of n bounded samples."""
    ref = CpuReference(cfg, threads)
    ref.sample(light=True)
    out = sorted((ref.sample() for _ in range(n)), key=lambda r: r[0])
    v, tot, desc = out[len(out) // 2]
    return v, tot, desc + f"; median of {n} samples", ref.threads


def bench_config(cfg, world: int, scaling: str, tiny: bool = False) -> dict:
    rows = BATCH if scaling == "weak" else max(1, BATCH // world)
    return {"workload": workload_name(cfg) + (" [TINY plumbing run -- not a bench number]" if tiny else ""),
            "global_batch": rows * world, "rows_per_gpu": rows, "parallelism": f"utterance-dp{world}",
            "sampling": "T=0.6 top_p=0.8 rep_penalty=1.3/20 (reference defaults), EOS masked",
            "prompt": "64 tokens: [SOH] 60 ids [EOT, EOH, START_OF_SPEECH]; parseOutput crops it, audio = 512 // 7 = 73 frames = 6.229 s per utterance (BASELINE.md)",
            "l2": "inputs larger than L2: every decode step streams %.2f GB of weights" % (weight_bytes(cfg) / 1e9),
            "audio_s_per_step": audio_seconds_per_utterance() * rows * world}


def cpu_whisper_sample(threads: int):
    """Whisper-base (config 3) on the CPU port: ONE 30 s clip -- log-mel, 6-layer encoder, 4-token prefix + 64 greedy steps
    (EOT masked) -- timed once after a light warm-up; x16 clips (batched == serial, linear in clips)."""
    import torch
    from oracle import dsp
    from oracle import whisper as ow
    torch.set_num_threads(threads)
    cfg = ow.WhisperConfig(**{k: v for k, v in WHISPER_BASE.items() if k in ow.WhisperConfig.__dataclass_fields__})
    W = ow.init_weights(cfg, 1234)
    x = dsp.synth_audio(480000, 0)
    ow.transcribe_tokens(ow.WhisperOracle(cfg, W), x[:32000], ow.build_prompt_tokens(), max_tokens=2, mask_eot=True)
    t0 = time.perf_counter()
    ow.transcribe_tokens(ow.WhisperOracle(cfg, W), x, ow.build_prompt_tokens(), max_tokens=WH_STEPS, mask_eot=True)
    dt = time.perf_counter() - t0
    return 30.0 / dt, f"oracle port (torch-CPU fp32), {threads} threads: 1 of {WH_BATCH} clips timed ({dt:.2f} s), x{WH_BATCH} (linear in clips)"


def run_reference_arm(args, rank: int, world: int):
    if rank != 0:
        return
    ref = CpuReference(ORPHEUS, usable_cpus())    # weights built once; every step is one bounded sample (see CpuReference)
    threads = ref.threads                          # the calibrated count (the fastest for this arm), fixed from here on, reported as `cores`
    vals, totals, sample = [], [], ""
    for i in range(args.warmup + args.steps):
        v, tot, sample = ref.sample(light=i < args.warmup)     # warm-up samples: threads / allocator only (one decode step)
        if i >= args.warmup:
            vals.append(v); totals.append(tot)
    v = float(np.median(vals))                     # median over the timed samples (each sample is itself built from medians)
    sample += f"; value = median of {len(vals)} samples (min {min(vals):.3f}, max {max(vals):.3f})"
    cfg = bench_config(ORPHEUS, world, args.scaling)
    cfg["reference_arm"] = ("CPU restatement of the reference path (the Swift/MLX reference cannot be built in this image); always the "
                            "batch-8 workload on rank 0's host cores, extrapolated from a bounded sample")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.median(totals)) * 1e3, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    try:
        wv, wdesc = cpu_whisper_sample(threads)
        line["whisper"] = {"metric": "whisper_base_stt_rtfx_batch16", "value": wv, "unit": UNIT, "cpu_baseline": {"value": wv, "unit": UNIT, "cores": threads, "kind": "port", "sample": wdesc}}
    except Exception as e:      # the headline line must still print
        line["whisper"] = {"unavailable": repr(e)[:200]}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------- GPU arm
WHISPER_BASE = dict(vocab_size=51865, num_mel_bins=80, d_model=512, encoder_layers=6, encoder_attention_heads=8, encoder_ffn_dim=2048,
                    max_source_positions=1500, decoder_layers=6, decoder_attention_heads=8, decoder_ffn_dim=2048, max_target_positions=448)
WH_BATCH, WH_STEPS, WH_SAMPLES = 16, 64, 480000
SNAC_BATCH, SNAC_T = 8, 1024


def whisper_encoder_flops() -> float:
    """Dense FLOPs of the Whisper-base encoder for one 30 s clip (SURVEY.md 8a row a14: ~87 GFLOP)."""
    d, f, T = WHISPER_BASE["d_model"], WHISPER_BASE["encoder_ffn_dim"], 1500
    conv = 2 * (3000 * 80 * 3 * d + T * d * 3 * d)
    layer = 2 * (4 * T * d * d + 2 * T * T * d + 2 * T * d * f)
    return float(conv + WHISPER_BASE["encoder_layers"] * layer)


DUMP_BYTES_MAX = 64 << 20


def write_outputs(directory, arrays: dict) -> None:
    """DIR/<name>.npy for every array: float32 and narrower floats as float32, everything else (integers exactly) as float64."""
    out = {}
    for k, v in arrays.items():
        v = np.asarray(v)
        out[k] = v.astype(np.float32 if v.dtype.kind == "f" and v.itemsize <= 4 else np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_BYTES_MAX:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES_MAX}-byte budget")
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    for k, a in out.items():
        np.save(d / f"{k}.npy", a)


def synth_clip(n: int, seed: int) -> np.ndarray:
    """SURVEY.md 8(d): x = 0.5 sin(2 pi 220 t) + 0.1 N(0, 1), clipped, 16 kHz."""
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float64) / 16000.0
    return np.clip(0.5 * np.sin(2 * np.pi * 220.0 * t) + 0.1 * rng.standard_normal(n), -1.0, 1.0).astype(np.float32)


class GpuTimer:
    """CUDA events on the library's own stream (torch.cuda.Event only sees the stream it is recorded on), barrier + synchronize on
    both sides, max over ranks."""

    def __init__(self, torch, dist, m):
        self.torch, self.dist, self.m = torch, dist, m

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def __call__(self, fn, stream, steps, warmup):
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = self.m.launch_count()
        e0.record(stream)
        outs = [fn() for _ in range(steps)]
        e1.record(stream)
        self.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item()), self.m.launch_count() - n0, outs


def whisper_block(m, torch, timer, rank, world, local, steps, warmup, dump=None):
    """BASELINE config 3: Whisper-base, 16 x 30 s synthetic clips per GPU, greedy, 64 forced decode steps (EOT masked)."""
    wm = m.WhisperModel.random_init(WHISPER_BASE, device=local, max_batch=WH_BATCH)
    stream = torch.cuda.ExternalStream(wm.stream, device=torch.device("cuda", local))
    pcm_host = torch.from_numpy(np.stack([synth_clip(WH_SAMPLES, 100 * rank + i) for i in range(WH_BATCH)])).pin_memory()
    pcm_dev = pcm_host.cuda()
    P = m.STTGenerateParameters(max_tokens=WH_STEPS, mask_eot=True)
    toks = torch.zeros((WH_BATCH, WH_STEPS), dtype=torch.int32).pin_memory()
    ntok = torch.zeros(WH_BATCH, dtype=torch.int32).pin_memory()
    ms_dev, launches, outs = timer(lambda: wm.generate_dev(pcm_dev, P, toks.numpy(), ntok.numpy()), stream, steps, warmup)
    if dump is not None:
        dump["whisper_tokens"], dump["whisper_token_counts"] = toks.numpy().copy(), ntok.numpy().copy()
    pcm_np = pcm_host.numpy()                       # a view of the pinned buffer: the C ABI copies host -> device from it
    ms_e2e, _, _ = timer(lambda: wm.generate(pcm_np, P), stream, steps, 1)
    assert int(ntok.min()) == WH_STEPS, "whisper benchmark produced too few tokens"
    audio = WH_BATCH * 30.0 * world
    enc_s = float(np.median([o.encode_time for o in outs]))
    dec_s = float(np.median([o.decode_time for o in outs]))
    peak, peak_src = measured_tensor_peak()
    ach = whisper_encoder_flops() * WH_BATCH / enc_s / 1e12
    alg_mel = WH_BATCH * (4 * WH_SAMPLES + 4 * 3000 * 80)
    return {"metric": "whisper_base_stt_rtfx_batch16", "unit": UNIT, "value": audio * steps / (ms_dev * 1e-3),
            "ms_per_step": ms_dev / steps,
            "config": {"workload": f"Whisper-base (d_model 512, 6+6 layers, vocab 51865) random-init bf16, {WH_BATCH} x 30 s synthetic 16 kHz clips per GPU, "
                                   f"greedy, 4-token prefix + {WH_STEPS} forced decode steps (EOT masked)", "clips_per_gpu": WH_BATCH},
            "e2e": {"value": audio * steps / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": int(pcm_host.numel() * 4), "d2h_bytes_per_step": int(toks.numel() * 4 + ntok.numel() * 4)},
            "gpu_launches": int(launches), "stages_s": {"encode(log-mel + encoder + cross K/V)": enc_s, "decode": dec_s},
            "roofline": {"kernel": "encoder (log-mel, conv stem, 6 x [LN, qkv gemm, attention, o gemm, LN, fc1+GELU, fc2], cross K/V projections); "
                                   "dominant kernels tc_gemm_kernel<128> + the encoder attention kernel", "bound": "tensor",
                         "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                         "flops_per_clip": whisper_encoder_flops(), "note": "useful dense FLOPs of the encoder / host-timed encode stage "
                         "(includes the log-mel kernel and the cross-K/V projections); log-mel algorithmic bytes %d per step" % alg_mel}}


def snac_block(m, torch, timer, rank, world, local, codec, steps, warmup, dump=None):
    """BASELINE config 2: SNAC-24kHz decode, batch 8 x 1024 latent steps -> 8 x 524 288 samples (21.85 s each)."""
    stream = torch.cuda.ExternalStream(codec.stream, device=torch.device("cuda", local))
    rng = np.random.default_rng(2 + rank)
    codes_host = [torch.from_numpy(rng.integers(0, 4096, size=(SNAC_BATCH, SNAC_T // s), dtype=np.int32)).pin_memory() for s in (4, 2, 1)]
    codes_dev = [c.cuda() for c in codes_host]
    wave_dev = torch.empty((SNAC_BATCH, 1, SNAC_T * 512), device="cuda")
    ms_dev, launches, _ = timer(lambda: codec.decode_dev(codes_dev, wave_dev, seed=1, stream=codec.stream), stream, steps, warmup)
    if dump is not None:
        dump["snac_waveforms"] = wave_dev.cpu().numpy()
    codes_np = [c.numpy() for c in codes_host]
    wave_np = torch.empty((SNAC_BATCH, 1, SNAC_T * 512), dtype=torch.float32).pin_memory().numpy()
    ms_e2e, _, outs = timer(lambda: codec.decode(codes_np, out=wave_np), stream, steps, 1)
    assert outs[-1].shape[-1] == SNAC_T * 512 and np.isfinite(outs[-1]).all()
    audio = SNAC_BATCH * SNAC_T * 512 / 24000.0 * world
    peak, peak_src = measured_peaks()
    fused = 441.5e6 * SNAC_BATCH               # SURVEY.md 8(d): every DecoderBlock boundary activation written once + read once, fp32
    minimum = SNAC_BATCH * (7168 + 2097152) + 52.5e6
    ach = fused / (ms_dev / steps * 1e-3) / 1e9
    return {"metric": "snac24k_decode_rtfx_batch8", "unit": UNIT, "value": audio * steps / (ms_dev * 1e-3), "ms_per_step": ms_dev / steps,
            "config": {"workload": f"SNAC-24kHz decode, batch {SNAC_BATCH} x {SNAC_T} latent steps (codes [8,256] [8,512] [8,1024]) -> 8 x 524288 samples, "
                                   "NoiseBlock noise drawn on the device"},
            "e2e": {"value": audio * steps / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": int(sum(c.numel() for c in codes_host) * 4), "d2h_bytes_per_step": int(wave_dev.numel() * 4)},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "whole decode (RVQ lookup, 4 DecoderBlocks, final conv); dominant kernels cg::conv_gemm_kernel + rf::ru_fused_kernel",
                         "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                         "bytes_definition": "SURVEY.md 8(d) per-block-fused bound, fp32 activations: 441.5 MB per utterance",
                         "algorithmic_minimum_bytes": minimum, "frac_vs_algorithmic_minimum": minimum / (ms_dev / steps * 1e-3) / 1e9 / peak}}


Q3_ROWS, Q3_FRAMES, Q3_CHUNK = 4, 1024, 64


def qwen3_block(m, torch, timer, rank, world, local, steps, warmup, dump=None):
    """BASELINE config 5: Qwen3-TTS-0.6B geometry (talker 1024 x 28, code predictor 1024 x 5, 16 code groups; random-init bf16 -- an
    8-bit checkpoint is expanded to bf16 at load, DESIGN.md 3.9), batch 32 over 8 GPUs = 4 utterances per GPU, 1024 frames each
    (81.9 s of audio), the codes decoded by the speech-tokenizer decoder (the model's vocoder) in streaming chunks of 64 frames."""
    import importlib
    codec = importlib.import_module("mlx_audio_swift_b200.qwen3_tts_codec")
    tcfg = m.Qwen3TalkerConfig()
    talker = m.Qwen3TTSTalker.random_init(tcfg, device=local, max_batch=Q3_ROWS, max_context=Q3_FRAMES + 32, std=0.02, seed=77 + rank)
    dcfg = codec.Qwen3TTSTokenizerDecoderConfig()
    dec = codec.Qwen3TTSSpeechTokenizerDecoder(dcfg, weights=codec.random_init_weights(dcfg, 5), device=local, max_batch=Q3_ROWS,
                                                 max_cache_frames=Q3_FRAMES + 8)
    rng = np.random.default_rng(9 + rank)
    H = tcfg.hidden_size
    embeds = (0.05 * rng.standard_normal((Q3_ROWS, 10, H))).astype(np.float32)          # the prompt rows prepareGenerationInputs builds (L = 10)
    trailing = (0.05 * rng.standard_normal((Q3_ROWS, 24, H))).astype(np.float32)
    pad = (0.05 * rng.standard_normal(H)).astype(np.float32)
    P = m.Qwen3GenerateParameters(max_tokens=Q3_FRAMES, temperature=0.9, top_k=50, top_p=1.0, repetition_penalty=1.05, seed=rank, mask_eos=True)
    stream = torch.cuda.ExternalStream(talker.stream, device=torch.device("cuda", local))
    stages, last = {}, {}

    def step():
        t0 = time.perf_counter()
        codes, info = talker.generate_codes(embeds, list(trailing), pad, P)
        t1 = time.perf_counter()
        c = np.ascontiguousarray(np.stack(codes).transpose(0, 2, 1))                    # [B, 16, frames]
        dec.reset_streaming_state()
        audio = [dec.streaming_step(c[:, :, f0:f0 + Q3_CHUNK]) for f0 in range(0, Q3_FRAMES, Q3_CHUNK)]
        stages["talker"], stages["decoder"] = t1 - t0, time.perf_counter() - t1
        assert sum(a.shape[-1] for a in audio) == Q3_FRAMES * 1920 and all(len(x) == Q3_FRAMES for x in codes)
        last["codes"], last["audio"] = c, audio
        return info

    ms, launches, infos = timer(step, stream, steps, warmup)           # every call ends synchronised (codes / audio copied to the host)
    if dump is not None:
        dump["qwen3_codes"], dump["qwen3_audio"] = last["codes"], np.concatenate(last["audio"], axis=-1)
    audio = Q3_ROWS * Q3_FRAMES * 1920 / 24000.0 * world
    frame_ms = float(np.median([i.generate_time for i in infos])) / Q3_FRAMES * 1e3
    return {"metric": "qwen3tts_0.6b_rtfx_batch4_per_gpu", "unit": UNIT, "value": audio * steps / (ms * 1e-3), "ms_per_step": ms / steps,
            "config": {"workload": f"Qwen3-TTS-0.6B geometry random-init bf16, {Q3_ROWS} utterances per GPU (batch 32 on 8 GPUs), 10 prompt rows, {Q3_FRAMES} "
                                   f"frames x 16 code groups each, sampled (T 0.9, top-k 50, rep 1.05, EOS masked), speech-tokenizer decoder in "
                                   f"{Q3_CHUNK}-frame streaming chunks", "rows_per_gpu": Q3_ROWS},
            "e2e": {"value": audio * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
                    "h2d_bytes_per_step": int(embeds.nbytes + trailing.nbytes + pad.nbytes + Q3_ROWS * 16 * Q3_FRAMES * 4),
                    "d2h_bytes_per_step": int(Q3_ROWS * Q3_FRAMES * (16 * 4 + 1920 * 4)),
                    "note": "the only entry points are host-buffer calls (b2a_qwen3_talker_generate, b2a_speech_tokenizer_streaming_step): value == e2e"},
            "gpu_launches": int(launches), "stages_s": dict(stages), "ms_per_frame": frame_ms,
            "roofline": {"kernel": "one frame = one CUDA graph (talker step + 16 code-predictor passes + 16 sampler launches)", "bound": "hbm",
                         "achieved": (0.88e9 + 16 * 0.15e9 + 15 * 2 * 2048 * 1024 * 2) / (frame_ms * 1e-3) / 1e9, "peak": measured_peaks()[0], "unit": "GB/s",
                         "frac": (0.88e9 + 16 * 0.15e9 + 15 * 2 * 2048 * 1024 * 2) / (frame_ms * 1e-3) / 1e9 / measured_peaks()[0], "traffic": None,
                         "note": "bytes = talker weights once + predictor weights 16 times + 15 heads/embeddings per frame (bf16); the frame is launch-latency bound, not HBM bound"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 8 utterances per GPU; strong: the fixed batch of 8 split 8/G per GPU (SURVEY.md 8e)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the whisper / snac blocks")
    ap.add_argument("--tiny", action="store_true", help="small model (plumbing check only; NOT a bench number)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what each timed device path returned in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import mlx_audio_swift_b200 as m

    assert m.device_count() > 0, "bench.py needs a CUDA device: libb200audio has no CPU fallback"
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":      # NCCL prints its version banner on STDOUT, ahead of the JSON line
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    timer = GpuTimer(torch, dist, m)

    cfg = dict(ORPHEUS)
    if args.tiny:
        cfg.update(hidden_size=512, num_hidden_layers=2, intermediate_size=1024, num_attention_heads=4, num_key_value_heads=2)
    rows = BATCH if args.scaling == "weak" else max(1, BATCH // world)
    assert args.scaling == "weak" or BATCH % world == 0, "strong scaling splits the batch of 8: use 1, 2, 4 or 8 GPUs"
    codec = m.SNAC(weights=m.SNAC.random_init_weights(1234), device=local)
    tts = m.LlamaTTSModel.random_init(cfg, snac=codec, device=local, max_batch=BATCH, max_context=PROMPT_LEN + GEN_TOKENS + 16,
                                      std=0.02, seed=1234 + (rank if args.scaling == "weak" else 0))
    params = m.GenerateParameters(max_tokens=GEN_TOKENS, temperature=0.6, top_p=0.8, repetition_penalty=1.3,
                                  repetition_context_size=20, seed=rank, mask_eos=True, wrap_codes=True)
    wave_len = frames_per_utterance() * 2048
    audio_s = rows * wave_len / 24000.0

    all_prompts = make_prompts(rank) if args.scaling == "weak" else make_prompts(0)[rank * rows:(rank + 1) * rows]
    ids_host = torch.from_numpy(np.ascontiguousarray(all_prompts)).pin_memory()
    toks_host = torch.zeros((rows, GEN_TOKENS), dtype=torch.int32).pin_memory()
    ntok_host = torch.zeros(rows, dtype=torch.int32).pin_memory()
    wave_host = torch.zeros((rows, wave_len), dtype=torch.float32).pin_memory()
    wlen_host = torch.zeros(rows, dtype=torch.int64)
    ids_dev = ids_host.cuda(non_blocking=False)
    wave_dev = torch.zeros((rows, wave_len), dtype=torch.float32, device="cuda")
    gathered = torch.zeros((world, rows, wave_len), dtype=torch.float32, device="cuda") if world > 1 else None
    stream = torch.cuda.ExternalStream(tts.stream, device=torch.device("cuda", local))
    dump = {} if args.dump_outputs and rank == 0 else None
    last = {}

    def step_dev():
        wl, info = tts.generate_dev(ids_dev, params, wave_dev, wave_len)
        if dist is not None:      # the ONE collective of the path: re-join decoded waveforms
            with torch.cuda.stream(stream):
                dist.all_gather_into_tensor(gathered, wave_dev)
        last["wave_lengths"] = wl
        return info

    def step_e2e():
        return tts.generate_into(ids_host, params, toks_host, ntok_host, wave_host, wlen_host)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, launches, infos = timer(step_dev, stream, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if dump is not None:
        dump["orpheus_waveforms"], dump["orpheus_wave_lengths"] = wave_dev.cpu().numpy(), last["wave_lengths"]
    ms_e2e, _, _ = timer(step_e2e, stream, args.steps, max(1, min(args.warmup, 1)))
    assert int(wlen_host[0]) == wave_len and bool(torch.isfinite(wave_host).all()), "benchmark produced no / bad audio"

    # roofline of the dominant kernel group: the captured decode step (weights streamed once + KV read), timed INSIDE the measured
    # loop: generate_time covers the GEN_TOKENS - 1 graph replays after the prefill (incl. the host's poll every 16 tokens)
    ctx = PROMPT_LEN + GEN_TOKENS // 2              # mean context over the loop; KV bytes are linear in it
    step_ms = float(np.median([i.generate_time for i in infos])) / (GEN_TOKENS - 1) * 1e3
    graph_ms = tts.time_steps(rows, ctx, 24)        # the same graph replayed back to back, greedy, no host polling (for reference)
    peak, peak_src = measured_peaks()
    alg_bytes = weight_bytes(cfg) + kv_bytes(cfg, rows, ctx, 2)
    built_bytes = weight_bytes(cfg) + kv_bytes(cfg, rows, ctx, KV_ELEM_BYTES_BUILT)
    achieved = alg_bytes / (step_ms * 1e-3) / 1e9

    secondary = {}
    if not args.no_secondary and not args.tiny:
        del tts
        torch.cuda.empty_cache()
        secondary["whisper"] = whisper_block(m, torch, timer, rank, world, local, args.steps, 3, dump)
        secondary["snac"] = snac_block(m, torch, timer, rank, world, local, codec, args.steps, 3, dump)
        try:
            secondary["qwen3"] = qwen3_block(m, torch, timer, rank, world, local, args.steps, 1, dump)
        except Exception as e:      # row N1 is the newest path: the headline line must still print
            secondary["qwen3"] = {"unavailable": repr(e)[:300]}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    value = world * audio_s * args.steps / (ms_dev * 1e-3)
    e2e = world * audio_s * args.steps / (ms_e2e * 1e-3)
    traffic = MEASURED_STEP_DRAM_BYTES["bytes"] if (rows == MEASURED_STEP_DRAM_BYTES["batch"] and not args.tiny) else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": bench_config(cfg, world, args.scaling, args.tiny),
        "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(ids_host.numel() * 4), "d2h_bytes_per_step": int(wave_host.numel() * 4 + toks_host.numel() * 4)},
        "gpu_launches": int(launches),
        "stages_s": {"prefill": float(np.median([i.prefill_time for i in infos])), "decode": float(np.median([i.generate_time for i in infos])),
                     "codec": float(np.median([i.codec_time for i in infos]))},
        # host-clock prefill + decode + codec of every timed step: a host-side stall between or inside steps shows up as an outlier here
        # (ms_per_step is the CUDA-event time of all steps / steps and includes such stalls)
        "steps_host_s": [float(i.prefill_time + i.generate_time + i.codec_time) for i in infos],
        "roofline": {"kernel": "decode step (CUDA graph of 144 launches: embed, norm, 28 x [qkv tcgen05 gemm (rstd in the epilogue), 2-CTA-cluster "
                               "attention, o cluster split-K gemm (+ residual + norm 2), gate/up gemm + swiglu, down cluster split-K gemm (+ residual + "
                               "next norm)], lm-head gemm, sampler); dominant kernels tc_gemm_kernel<16> / tc_gemm_splitk_kernel", "bound": "hbm",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "traffic_source": "sum of dram__bytes_read.sum + dram__bytes_write.sum over the launches of one step at context 320, batch 8 "
                                       "(ncu, profiles/r02_decode_step_dram.csv / .md)",
                     "algorithmic_bytes_per_step": alg_bytes, "bytes_definition": "SURVEY.md 8(d): every weight once (bf16, tied lm head) + bf16 K/V read at the mean context",
                     "kv_cache_dtype_built": "f32", "built_bytes_per_step": built_bytes,
                     "ms_per_decode_step": step_ms, "ms_per_decode_step_source": "median generate_time / 511 graph replays inside the timed loop",
                     "ms_per_graph_replay_back_to_back": graph_ms, "context": ctx},
        "clocks": clocks,
    }
    line.update(secondary)
    if not args.no_cpu_baseline and world == 1 and not args.tiny:
        v, tot, sample, threads = cpu_reference_sample(cfg, usable_cpus())
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
        if "whisper" in line:
            try:
                wv, wdesc = cpu_whisper_sample(threads)
                line["whisper"]["cpu_baseline"] = {"value": wv, "unit": UNIT, "cores": threads, "kind": "port", "sample": wdesc}
            except Exception as e:
                line["whisper"]["cpu_baseline"] = {"unavailable": repr(e)[:200]}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
