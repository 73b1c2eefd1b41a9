#!/usr/bin/env python
"""bench.py -- the headline measurement (contract: task brief "Measurement").

Workload = BASELINE.json configs[2], the configuration its metric is quoted on: the FULL TURN of the cascade on one GPU,
    Whisper-small STT (10 s / 16 kHz utterance, 128 tokens)  ->  Llama-3-8B bf16 (64-token prompt, 128-token reply)
    ->  Qwen3-TTS (talker + code predictor + codec decoder; the reply spoken: 20-token first sentence + the other 108 tokens)
with S conversation sessions per GPU in flight together (sessions batch inside the GPU; ranks shard sessions, SURVEY.md 8e).
Weights: seeded random-init at the exact / published geometries (no checkpoints offline); timing is value independent.
One STEP = one wave: every one of the S sessions of a rank completes one full turn.

metric   "concurrent real-time sessions": a live session repeats [user speaks AUDIO_IN_S -> turn -> assistant speaks the
         reply]; a GPU that completes S turns in T seconds sustains S * cycle_s / T such sessions, cycle_s = AUDIO_IN_S + the
         seconds of speech generated per turn; "real-time" additionally needs every session's TTS real-time factor >= 1 in the
         wave (reported; the line says so when it fails).  The p50 audio-in -> first-audio-out latency (VADAudio.created_at_s ->
         first int16 block, the interval the reference logs, S/TTS/qwen3_tts_handler.py:867-878) is reported beside it for one
         session on an idle GPU and for the sessions of the loaded wave.
value    device-timed: inputs resident in HBM, engine-level launch sequence of the wave, CUDA events.
e2e      the same wave through the three HANDLER classes (B200WhisperSTTHandler -> B200LanguageModelHandler ->
         B200Qwen3TTSHandler): one thread per session, host PCM in, int16 blocks on the host out, shared engines + batchers.
roofline the kernel with the largest share of the step (measured per stage with CUDA events): algorithmic bytes / time.
cpu_baseline / --impl reference: the reference's CPU path for the same turn on the host cores (transformers Whisper-small
         fp32 in full + a stated, scaled sample of Llama-3-8B; faster-whisper and faster-qwen3-tts are unavailable).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 1 --warmup 0
    python bench.py --gpus 1 --steps 3 --warmup 3 --dump-outputs DIR     # + what the last timed wave computed, as DIR/*.npy
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import queue
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the benchmark leaves the tree as it found it (it may be read-only)

MODEL = "small"
AUDIO_S = 10.0
N_SAMPLES = 160000
MAX_NEW = 128                     # STT tokens and LLM reply tokens
LLM_PROMPT = 64
FIRST_SENTENCE = 20               # reply tokens that make the first TTS input (stream_batch_sentences=1)
SEC_PER_TOKEN = 0.30              # speech seconds per reply token (~2.6 words/s, the handler's own estimate, :60)
FRAMES_PER_S = 12.5
CHUNK = 8                         # the reference's streaming chunk (qwen3_tts_handler.py:49)
LEFT_CTX = 25
TTS_GEOM = "qwen3-tts-12hz"
PREFIX = [50258, 50259, 50359, 50363]
SUPPRESS = [1, 2, 7, 8, 9, 10, 14, 25, 26, 27, 28, 29, 31, 58, 59, 60, 61, 62, 63, 90, 91, 92, 93, 359, 503, 522, 542,
            873, 893, 902, 918, 922, 931, 1350, 1853, 1982, 2460, 2627, 3246, 3253, 3268, 3536, 3846, 3961, 4183, 4667,
            6585, 6647, 7273, 9061, 9383, 10428, 10929, 11938, 12033, 12331, 12562, 13793, 14157, 14635, 15265, 15618,
            16553, 16604, 18362, 18956, 20075, 21675, 22520, 26130, 26161, 26435, 28279, 29464, 31650, 32302, 32470,
            36865, 42863, 47425, 49870, 50254, 50258, 50358, 50359, 50360, 50361, 50362]
BEGIN_SUPPRESS = [220, 50257]
METRIC = "concurrent real-time sessions (full turn: Whisper-small -> Llama-3-8B 128-tok reply -> Qwen3-TTS); p50 audio-in->first-audio-out ms"


def frames_for(tokens: int) -> int:
    return int(round(tokens * SEC_PER_TOKEN * FRAMES_PER_S))


F1, F2 = frames_for(FIRST_SENTENCE), frames_for(MAX_NEW - FIRST_SENTENCE)     # 75 + 405 frames = 38.4 s of speech
REPLY_S = (F1 + F2) / FRAMES_PER_S
CYCLE_S = AUDIO_S + REPLY_S


def workload_config(world: int, sessions_per_gpu: int) -> dict:
    """The SAME dict on both arms (the driver compares them)."""
    return {"workload": "full turn, BASELINE configs[2]: whisper-small STT (10 s utterance, 128 tokens) -> llama-3-8b (64-token "
                        "prompt, 128-token reply) -> qwen3-tts 12 Hz (reply spoken: 75 + 405 codec frames = 38.4 s)",
            "audio_in_s": AUDIO_S, "reply_audio_s": REPLY_S, "cycle_s": CYCLE_S, "stt_tokens": MAX_NEW, "llm_prompt": LLM_PROMPT,
            "llm_reply_tokens": MAX_NEW, "tts_frames": F1 + F2, "tts_chunk_frames": CHUNK, "tts_left_context": LEFT_CTX,
            "sessions_per_gpu": sessions_per_gpu, "parallelism": f"session-shard dp{world}",
            "gates": "speculative_reopen 0, smart_turn off, stream_batch_sentences 1 (BASELINE.md section 3)",
            "weights": "seeded random-init, exact / published geometries"}


def decode_bytes_whisper(g, n_prefix, max_new, B) -> float:
    d, L, f, V, T = g.d_model, g.dec_layers, g.ffn, g.vocab, g.max_source_positions
    w_layer = (3 * d * d + 3 * d * d + 2 * f * d) * 2
    cross_kv = L * T * 2 * d * 2
    steps = n_prefix - 1 + max_new
    self_kv = sum(L * 2 * (p + 1) * d * 2 for p in range(steps))
    return steps * (L * w_layer + B * cross_kv) + max_new * V * d * 2 + B * self_kv


def decode_bytes_llama(g, n_steps, B, past) -> float:
    d, L, f, V = g.d_model, g.layers, g.ffn, g.vocab
    qd, kvd = g.heads * g.head_dim, g.kv_heads * g.head_dim
    w_layer = ((qd + 2 * kvd) * d + d * qd + 3 * f * d) * 2
    kv = sum(L * 2 * (past + s + 1) * kvd * 2 for s in range(n_steps))
    return n_steps * (L * w_layer + V * d * 2) + B * kv


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# =============================================================================================== reference arm (CPU)
def build_hf_whisper(g):
    import torch
    from transformers import WhisperConfig, WhisperForConditionalGeneration
    cfg = WhisperConfig(vocab_size=g.vocab, num_mel_bins=g.n_mels, d_model=g.d_model, encoder_layers=g.enc_layers,
                        decoder_layers=g.dec_layers, encoder_attention_heads=g.heads, decoder_attention_heads=g.heads,
                        encoder_ffn_dim=g.ffn, decoder_ffn_dim=g.ffn, max_source_positions=g.max_source_positions,
                        max_target_positions=g.max_target_positions, pad_token_id=0, bos_token_id=0, eos_token_id=0,
                        decoder_start_token_id=PREFIX[0], suppress_tokens=None, begin_suppress_tokens=None)
    torch.manual_seed(0)
    return WhisperForConditionalGeneration(cfg).eval()


def run_reference_stt(model, fe, audio):
    """What WhisperSTTHandler.process does on device='cpu', torch_dtype float32 (S/STT/whisper_stt_handler.py:83-87, 243)."""
    import torch
    feats = fe(audio, sampling_rate=16000, return_tensors="pt").input_features
    with torch.no_grad():
        return model.generate(feats, decoder_input_ids=torch.tensor([PREFIX]), max_new_tokens=MAX_NEW, min_new_tokens=MAX_NEW,
                              num_beams=1, do_sample=False, suppress_tokens=SUPPRESS, begin_suppress_tokens=BEGIN_SUPPRESS,
                              return_timestamps=False)


LLM_SAMPLE_LAYERS, LLM_SAMPLE_TOKENS = 2, 8


def cpu_turn(n_turns: int, threads: int) -> dict:
    """The reference's CPU implementation of the turn on `threads` host threads: transformers Whisper-small generate fp32 (in
    full: the call WhisperSTTHandler makes) + the transformers Llama decoder stack at the Llama-3-8B layer geometry, a bounded
    sample (2 of 32 layers, the 64-token prompt + 8 of 128 reply tokens through the KV cache, fp32) scaled by 32/2 x 128/8;
    embedding and lm_head are left out of the sample, which flatters the CPU arm.  TTS: n/a (faster-qwen3-tts is not installed
    anywhere; SURVEY.md 8d), so the CPU turn is STT + LLM only -- again in the CPU arm's favour."""
    import logging
    import torch
    from oracle import weights as W
    torch.set_num_threads(threads)
    logging.getLogger("transformers").setLevel(logging.ERROR)
    from transformers import LlamaConfig, LlamaModel, WhisperFeatureExtractor
    g = W.WHISPER_GEOMETRIES[MODEL]
    model = build_hf_whisper(g)
    fe = WhisperFeatureExtractor(feature_size=g.n_mels)
    lg = W.LLAMA_GEOMETRIES["llama-3-8b"]
    cfg = LlamaConfig(vocab_size=1024, hidden_size=lg.d_model, intermediate_size=lg.ffn, num_hidden_layers=LLM_SAMPLE_LAYERS,
                      num_attention_heads=lg.heads, num_key_value_heads=lg.kv_heads, head_dim=lg.head_dim, rms_norm_eps=lg.rms_eps,
                      rope_theta=lg.rope_theta)
    torch.manual_seed(1)
    llm = LlamaModel(cfg).eval()
    prompt = torch.randint(0, 1024, (1, LLM_PROMPT))
    run_reference_stt(model, fe, W.synthetic_audio(0, N_SAMPLES))          # warm-up
    stt_s, llm_s = [], []
    for i in range(n_turns):
        a = W.synthetic_audio(100 + i, N_SAMPLES)
        t = time.perf_counter()
        run_reference_stt(model, fe, a)
        stt_s.append(time.perf_counter() - t)
        with torch.no_grad():
            out = llm(prompt, use_cache=True)                               # prefill (not timed: the GPU arm's prefill is small too)
            kv, tok = out.past_key_values, prompt[:, -1:]
            t = time.perf_counter()
            for _ in range(LLM_SAMPLE_TOKENS):
                out = llm(tok, past_key_values=kv, use_cache=True)
                kv = out.past_key_values
            llm_s.append(time.perf_counter() - t)
    stt, llm_sample = sum(stt_s) / len(stt_s), sum(llm_s) / len(llm_s)
    llm_full = llm_sample * (32 / LLM_SAMPLE_LAYERS) * (MAX_NEW / LLM_SAMPLE_TOKENS)
    turn = stt + llm_full
    return {"value": CYCLE_S / turn, "unit": "sessions", "cores": threads, "kind": "reference",
            "turn_s": turn, "stt_s": stt, "llm_s_scaled": llm_full,
            "sample": f"{n_turns} turn(s): transformers {__import__('transformers').__version__} WhisperForConditionalGeneration.generate fp32 "
                      f"in full ({stt:.2f} s) + LlamaModel fp32 decode {LLM_SAMPLE_LAYERS}/32 layers x {LLM_SAMPLE_TOKENS}/128 tokens "
                      f"({llm_sample:.2f} s, scaled to {llm_full:.1f} s; embedding / lm_head not counted); TTS n/a; torch.set_num_threads({threads}) "
                      f"of {os.cpu_count()} cpus; faster-whisper unavailable, transformers CPU path timed instead; faster-qwen3-tts unavailable"}


def host_threads() -> int:
    """CPU threads of the reference arm: the cores this process may run on (affinity / cgroup aware), at most 64 -- the same
    count whatever the launcher's OMP_NUM_THREADS says (torchrun sets it to 1) and without oversubscribing a box whose
    os.cpu_count() exceeds its quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(n, os.cpu_count() or n, 64))


def cpu_baseline_subprocess(turns: int, timeout_s: float = 240.0) -> dict:
    """The CPU turn in a child process (fresh OpenMP runtime, no CUDA context, hard time limit): `bench.py --impl reference`."""
    import subprocess as sp
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        r = sp.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(max(1, turns)), "--warmup", "0"],
                   capture_output=True, text=True, timeout=timeout_s, env=env)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                line = json.loads(ln)
                if line.get("cpu_baseline"):
                    return line["cpu_baseline"]
                return {"value": None, "unit": "sessions", "cores": 0, "kind": "reference", "sample": "failed: " + str(line.get("error"))}
        return {"value": None, "unit": "sessions", "cores": 0, "kind": "reference", "sample": "failed: no output; " + r.stderr[-300:]}
    except sp.TimeoutExpired:
        return {"value": None, "unit": "sessions", "cores": host_threads(), "kind": "reference",
                "sample": f"not finished within {timeout_s:.0f} s on this host (bounded sample aborted)"}


def reference_arm(args, rank, world):
    """--impl reference: rank 0 alone, a fixed thread count whatever the launcher's OMP_NUM_THREADS says."""
    if rank != 0:
        return
    threads = host_threads()
    line = {"metric": METRIC, "unit": "sessions", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": "reference", "config": workload_config(world, args.sessions)}
    try:
        cb = cpu_turn(max(1, args.steps), threads)
        line.update({"value": cb["value"], "ms_per_step": 1e3 * cb["turn_s"], "cpu_baseline": cb,
                     "e2e": {"value": cb["value"], "unit": "sessions", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "latency_ms_p50": 1e3 * cb["turn_s"]})
    except Exception as e:
        line.update({"value": None, "error": f"{type(e).__name__}: {e}"})
    print(json.dumps(line), flush=True)


# =============================================================================================== B200 arm
_T0 = time.perf_counter()


def log(msg: str) -> None:
    """Progress on stderr (the JSON line is the only thing on stdout)."""
    print(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


class Stack:
    """The three engines of one lane of one GPU, shared by the lane's sessions.  A lane is an SM partition (engine.get_context):
    with L lanes the persistent decode kernels of lane i run on num_sms // L CTAs, concurrently with the other lanes'."""

    def __init__(self, E, W, dev: int, S: int, lane: int = 0, lanes: int = 1):
        import torch
        from speech_to_speech_b200.tts_model import B200Qwen3TTS
        self.E, self.W, self.dev, self.S, self.lane, self.lanes = E, W, dev, S, lane, lanes
        self.wg = W.WHISPER_GEOMETRIES[MODEL]
        self.lg = W.LLAMA_GEOMETRIES["llama-3-8b"]
        self.whisper = E.WhisperEngine(self.wg.to_dict(), dtype="float16", max_batch=min(16, S), device=dev, lane=lane, lanes=lanes)
        self.whisper.init_random(1234)
        self.llm = E.LlamaEngine(self.lg.to_dict(), dtype="bfloat16", max_sessions=S, max_positions=LLM_PROMPT + MAX_NEW + 8,
                                 max_prefill=LLM_PROMPT * 8, device=dev, lane=lane, lanes=lanes)
        self.llm.init_random(7)
        self.tts = B200Qwen3TTS.from_random(TTS_GEOM, seed=11, dtype="bfloat16", device=dev, max_sessions=S,
                                            max_positions=max(F1, F2) + 32, max_text=128, lane=lane, lanes=lanes)
        self.opts = E.WhisperDecodeOptions(prefix=PREFIX, eos_id=-1, max_new_tokens=MAX_NEW, suppress=SUPPRESS,
                                           begin_suppress=BEGIN_SUPPRESS)
        mb = self.llm.max_decode_batch()
        self.llm_b = -(-S // (-(-S // mb)))          # balanced launches: 16 sessions, 12 per launch at most -> 8 + 8
        self.tts_b = self.tts.engine.max_batch()
        self.prompt = np.random.default_rng(0).integers(0, self.lg.vocab, LLM_PROMPT).tolist()
        from speech_to_speech_b200.handlers.qwen3_tts_postproc import TTSPostProcessor
        self.post = TTSPostProcessor(dev)
        self.torch = torch


class TtsProfileWindow:
    """cudaProfilerStart/Stop around chunks [first, first + n) of the second utterance's frame loop (all lanes): an ncu launch
    list of the whole region is ~42k launches at ~0.2 s each, the per-chunk kernel mix is what the list is for."""

    def __init__(self, torch, lanes: int, n: int, first: int = 2):
        self.torch, self.lanes, self.n, self.first = torch, lanes, n, first
        self.lock, self.started, self.stopped = threading.Lock(), 0, 0

    def chunk_begin(self, ci: int) -> None:
        if ci == self.first:
            with self.lock:
                self.started += 1
                if self.started == 1:
                    self.torch.cuda.cudart().cudaProfilerStart()

    def chunk_end(self, ci: int) -> None:
        if ci == self.first + self.n - 1:
            self.torch.cuda.current_stream().synchronize()
            with self.lock:
                self.stopped += 1
                if self.stopped == self.lanes:
                    self.torch.cuda.cudart().cudaProfilerStop()


def wave_device(st: Stack, pcm_dev, ev, tts_prof: "TtsProfileWindow | None" = None, out: "dict | None" = None) -> None:
    """One wave of S full turns as an engine-level launch sequence; stage boundaries marked with CUDA events.  `out`, when given,
    collects the device tensors the wave returns (token ids, codec codes, int16 audio) for wave_outputs()."""
    torch, S = st.torch, st.S
    keep = out is not None
    if keep:
        out.update(stt=[], llm_first=[], llm=[], tts=[])
    dev = f"cuda:{st.dev}"
    ev["t0"].record()
    for b0 in range(0, S, 16):                                           # ---- STT
        nb = min(16, S - b0)
        st.whisper.logmel(pcm_dev[b0:b0 + nb], [N_SAMPLES] * nb)
        st.whisper.encode(nb)
        wa, wb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wa.record()
        ids, _ = st.whisper.decode(nb, st.opts)
        wb_.record()
        if keep:
            out["stt"].append(ids)
        ev["whisper_mark"].append((wa, wb_))
    ev["stt"].record()
    firsts = []
    for b0 in range(0, S, 8):                                             # ---- LLM prefill: 8 prompts per pass over the weights
        sl = list(range(b0, min(S, b0 + 8)))
        for s in sl:
            st.llm.reset(s)
        firsts.append(st.llm.prefill_batch(sl, [st.prompt] * len(sl)))
    ev["prefill"].record()
    first = torch.cat(firsts)
    for b0 in range(0, S, st.llm_b):                                      # ---- LLM decode, llm_b sessions per launch
        sl = list(range(b0, min(S, b0 + st.llm_b)))
        ids, _ = st.llm.decode(sl, first[b0:b0 + len(sl)].contiguous(), MAX_NEW - 1)
        if keep:
            out["llm"].append(ids)
    if keep:
        out["llm_first"].append(first)
    ev["llm"].record()
    eng = st.tts.engine
    text1, text2 = [3] * FIRST_SENTENCE, [5] * (MAX_NEW - FIRST_SENTENCE)
    for text, frames in ((text1, F1), (text2, F2)):                       # ---- TTS: two utterances per turn
        for s in range(S):
            eng.prefill(s, text, 2301)
        if keep:
            out["tts"].append([])                                         # per chunk: (codes of each launch, audio of each session)
        done, ci = 0, 0
        while done < frames:
            n = min(CHUNK, frames - done)
            if tts_prof is not None and text is text2:
                tts_prof.chunk_begin(ci)
            codes = [eng.decode_frames(list(range(b0, min(S, b0 + st.tts_b))), n) for b0 in range(0, S, st.tts_b)]
            ev["frames_mark"].append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
            a, b = ev["frames_mark"][-1]
            a.record()
            audio = [st.post.to_int16_device(wav) for b0 in range(0, S, st.tts_b)
                     for wav in eng.decode_audio_batch(list(range(b0, min(S, b0 + st.tts_b))), n, LEFT_CTX)]
            b.record()
            if keep:
                out["tts"][-1].append((codes, audio))
            if tts_prof is not None and text is text2:
                tts_prof.chunk_end(ci)
            done += n
            ci += 1
    ev["tts"].record()


def run_wave(stacks, pcm_dev, evs, tts_prof=None, outs=None):
    """One wave on every lane at once: a host thread per lane issues the lane's launch sequence on the lane's stream; the step is
    timed on the calling stream, from an event every lane waits for to an event that waits for every lane.  outs: one dict per
    lane for wave_device's `out`."""
    outs = outs or [None] * len(stacks)
    torch = stacks[0].torch
    cur = torch.cuda.current_stream()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(cur)
    if len(stacks) == 1:
        wave_device(stacks[0], pcm_dev, evs[0], tts_prof, outs[0])
    else:
        errs, Sl = [], stacks[0].S

        def run(i):
            try:
                st = stacks[i]
                torch.cuda.set_device(st.dev)
                with st.E.lane_context(st.dev, st.lane, st.lanes):
                    torch.cuda.current_stream().wait_event(start)
                    wave_device(st, pcm_dev[i * Sl:(i + 1) * Sl], evs[i], tts_prof, outs[i])
                    evs[i]["done"].record()
            except BaseException as e:  # noqa: BLE001
                errs.append(e)
        ths = [threading.Thread(target=run, args=(i,), daemon=True) for i in range(len(stacks))]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if errs:
            raise errs[0]
        for e in evs:
            cur.wait_event(e["done"])
    end.record(cur)
    return start, end


def e2e_wave(handlers, auds, S, offsets=None) -> dict:
    """The wave through the three handler classes, one thread per session (the reference's thread-per-unit shape).  offsets[i]:
    seconds after the start of the wave at which session i stops speaking (default: all at once, the worst case)."""
    from speech_to_speech_b200.host import resolve
    api = resolve()
    lat, rtf, t_done = [None] * S, [None] * S, [None] * S
    errs = []

    def session(i):
        try:
            stt, llm, tts = handlers[i]
            if offsets is not None:
                time.sleep(offsets[i])
            vad = api.VADAudio(audio=auds[i], mode="final", turn_id=f"t{i}", turn_revision=0)
            out = list(stt.process(vad))
            tr = out[-1]
            first_audio, speech_s, t_tts0 = None, 0.0, None
            sentences: "queue.Queue" = queue.Queue()

            def generate():
                """The LLM stage of the unit: its own thread, like the reference's handler threads -- it keeps generating while
                the TTS stage speaks the first sentence (sentences travel through a queue, LLM/language_model.py -> TTS)."""
                try:
                    sent_first = False
                    for _piece in llm.generate_text_stream(llm_prompt, max_new_tokens=MAX_NEW):
                        if not sent_first and len(llm.streamer.generated) >= FIRST_SENTENCE:
                            sentences.put((FIRST_SENTENCE, F1))
                            sent_first = True
                    sentences.put((MAX_NEW - FIRST_SENTENCE, F2))
                except BaseException as e:  # noqa: BLE001
                    sentences.put(e)
                finally:
                    sentences.put(None)

            def speak(n_tokens, frames):
                nonlocal first_audio, speech_s, t_tts0
                tts.max_new_tokens = frames
                tts.streaming_chunk_size = CHUNK
                if t_tts0 is None:
                    t_tts0 = time.perf_counter()
                item = api.TTSInput(text="x" * n_tokens, speech_stopped_at_s=tr.speech_stopped_at_s)
                for blk in tts.process(item):
                    if first_audio is None:
                        first_audio = time.perf_counter()
                    speech_s += len(blk) / 16000.0
            gen_thread = threading.Thread(target=generate, daemon=True)
            gen_thread.start()
            while True:
                it = sentences.get()
                if it is None:
                    break
                if isinstance(it, BaseException):
                    raise it
                speak(*it)
            gen_thread.join()
            t_end = time.perf_counter()
            lat[i] = 1e3 * (first_audio - vad.created_at_s)
            rtf[i] = speech_s / max(1e-9, t_end - t_tts0)
            t_done[i] = t_end
        except Exception as e:  # noqa: BLE001
            errs.append(f"session {i}: {type(e).__name__}: {e}")

    llm_prompt = np.random.default_rng(0).integers(0, 128256, LLM_PROMPT).tolist()
    ths = [threading.Thread(target=session, args=(i,), daemon=True) for i in range(S)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    deadline = t0 + 240.0                      # a stuck session must not hang the bench: report it instead
    for t in ths:
        t.join(max(0.0, deadline - time.perf_counter()))
    stuck = sum(t.is_alive() for t in ths)
    if stuck:
        errs.append(f"{stuck} session thread(s) still running after 240 s")
    wall = time.perf_counter() - t0
    ok = [x for x in lat if x is not None]
    return {"wall_s": wall, "latency_ms": ok, "rtf": [x for x in rtf if x is not None], "errors": errs[:3]}


DUMP_AUDIO_SAMPLES = 1 << 21      # --dump-outputs: int16 samples kept of the wave's audio (all of it is 78 MB as float32)


def wave_outputs(outs: list) -> dict:
    """What one wave returned (wave_device's `out` of every lane), sessions in order lane by lane, as float32 arrays: the STT and
    LLM token ids, the codec codes of both TTS utterances, and a fixed, seeded sample of the 16 kHz int16 audio of every session
    (the utterances one after the other) with its (session, sample) index."""
    import torch
    cat = torch.cat
    res = {"stt_token_ids": cat([t for o in outs for t in o["stt"]]),
           "llm_token_ids": cat([cat([cat(o["llm_first"])[:, None], cat(o["llm"])], 1) for o in outs])}
    for u, name in enumerate(("first_sentence", "rest")):
        res[f"tts_codes_{name}"] = cat([cat([cat(codes) for codes, _ in o["tts"][u]], 1) for o in outs])
    audio = cat([torch.stack([cat([a[j] for chunks in o["tts"] for _, a in chunks]) for j in range(o["llm_first"][0].numel())])
                 for o in outs]).cpu().numpy()
    res = {k: v.cpu().numpy() for k, v in res.items()}
    pick = np.sort(np.random.default_rng(0).choice(audio.size, min(audio.size, DUMP_AUDIO_SAMPLES), replace=False))
    res["tts_audio_int16_sample"] = audio.reshape(-1)[pick]
    res["tts_audio_int16_sample_index"] = np.stack(np.unravel_index(pick, audio.shape), 1)
    return {k: v.astype(np.float32) for k, v in res.items()}


LLM_STREAM_CHUNK = 4     # tokens per decode launch in the handler path: the TTS stage sees a sentence at most 4 steps late, and a
                         # first-sentence TTS request waits behind at most 4 LLM steps on the lane's stream


def make_handlers(S: int, dev: int, lanes: int = 1):
    """S pipeline units' worth of handler instances; the units of a lane share one engine per stage (gen_kwargs / kwargs of the
    reference slots)."""
    from queue import Queue
    from threading import Event
    from speech_to_speech_b200.handlers.language_model_handler import B200LanguageModelHandler
    from speech_to_speech_b200.handlers.qwen3_tts_handler import B200Qwen3TTSHandler
    from speech_to_speech_b200.handlers.whisper_stt_handler import B200WhisperSTTHandler
    out = []
    Sl = S // lanes
    for i in range(S):
        lane = i // Sl
        stt = B200WhisperSTTHandler(Event(), queue_in=Queue(), queue_out=Queue(),
                                    setup_kwargs=dict(model_name=f"random:{MODEL}:1234", device=f"cuda:{dev}", torch_dtype="float16",
                                                      language="en", gen_kwargs={"max_new_tokens": MAX_NEW}, max_batch=min(16, Sl),
                                                      lane=lane, lanes=lanes))
        stt.tokens.eos = -1                   # random-init weights: every utterance decodes its full 128 tokens (both arms do)
        llm = object.__new__(B200LanguageModelHandler)   # the load hook only: the request lifecycle needs the reference's Chat types
        llm.device = f"cuda:{dev}"
        B200LanguageModelHandler._load_model(llm, "random:llama-3-8b:7", f"cuda:{dev}", "bfloat16",
                                             {"max_new_tokens": MAX_NEW, "max_sessions": Sl, "max_positions": LLM_PROMPT + MAX_NEW + 8,
                                              "stream_chunk_tokens": LLM_STREAM_CHUNK, "lane": lane, "lanes": lanes})
        llm.eos_ids = []                      # random-init weights: never stop early, every reply has 128 tokens
        llm.streamer.eos_ids = set()
        tts = B200Qwen3TTSHandler(Event(), queue_in=Queue(), queue_out=Queue(), setup_args=(Event(),),
                                  setup_kwargs=dict(model_name=f"random:{TTS_GEOM}", device=f"cuda:{dev}", speaker="Aiden",
                                                    max_sessions=Sl, lane=lane, lanes=lanes, gen_kwargs={"seed": 11}))
        out.append((stt, llm, tts))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sessions", type=int, default=32, help="conversation sessions in flight per GPU (one wave = one turn of each)")
    ap.add_argument("--lanes", type=int, default=2,
                    help="SM partitions per GPU: each lane runs sessions/lanes sessions through its own engines; the lanes' persistent "
                         "decode launches run concurrently on num_sms/lanes CTAs each")
    ap.add_argument("--cpu-baseline-turns", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profile-tts-chunks", type=int, default=0,
                    help="cudaProfilerStart/Stop around this many 8-frame chunks (frames + codec + post-processing) of the TTS stage only")
    ap.add_argument("--profile-region", action="store_true",
                    help="cudaProfilerStart/Stop around the device-timed region (use with ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's sessions) as DIR/<name>.npy, float32, under 64 MB; "
                         "the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from oracle import weights as W
    from speech_to_speech_b200 import engine as E, shard

    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    dev = f"cuda:{local_rank}"
    S, L = args.sessions, max(1, args.lanes)
    assert S % L == 0, "--sessions must be a multiple of --lanes"
    stacks = [Stack(E, W, local_rank, S // L, lane, L) for lane in range(L)]
    st = stacks[0]
    log(f"engines built: {L} lane(s) x {S // L} sessions, llm max batch {st.llm_b}, tts max batch {st.tts_b}")

    # ---- session-shard split: the ingest rank (0) holds every session's PCM and scatters each rank its shard over NCCL -------
    layout = shard.shard_layout(world * S, world)
    full = None
    if rank == 0:
        full = torch.stack([torch.from_numpy(W.synthetic_audio(sid, N_SAMPLES)) for r in range(world) for sid in layout[r]]).to(dev)
    if world > 1:   # the first collective of a process group builds the NCCL communicator: keep that out of the exchange timing
        shard.scatter_from_ingest(full, S, (N_SAMPLES,), torch.float32, dev)
        shard.gather_to_ingest(torch.zeros((S, 64), dtype=torch.int32, device=dev))
        torch.cuda.synchronize()
    xe = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    xe[0].record()
    pcm_dev = shard.scatter_from_ingest(full, S, (N_SAMPLES,), torch.float32, dev)
    xe[1].record()
    torch.cuda.synchronize()
    scatter_ms = xe[0].elapsed_time(xe[1])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def new_events():
        names = ("t0", "stt", "prefill", "llm", "tts", "done")
        out = []
        for _ in range(L):
            ev = {n: torch.cuda.Event(enable_timing=True) for n in names}
            ev["frames_mark"] = []
            ev["whisper_mark"] = []
            out.append(ev)
        return out

    for i in range(args.warmup):
        run_wave(stacks, pcm_dev, new_events())
        torch.cuda.synchronize()
        log(f"warm-up wave {i} done")

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    E.launch_count(local_rank, reset=True)
    evs, spans = [], []
    barrier()
    if args.profile_region:
        torch.cuda.cudart().cudaProfilerStart()
    t_wall = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)                 # L2 flush between timed steps (not timed)
        ev = new_events()
        prof = TtsProfileWindow(torch, L, args.profile_tts_chunks) if args.profile_tts_chunks > 0 and i == 0 else None
        outs = [{} for _ in stacks] if args.dump_outputs and rank == 0 and i == args.steps - 1 else None
        spans.append(run_wave(stacks, pcm_dev, ev, prof, outs))
        evs.append(ev[0])                     # stage boundaries: lane 0's (the lanes run the same sequence side by side)
    barrier()
    if args.profile_region:
        torch.cuda.cudart().cudaProfilerStop()
    wall_s = time.perf_counter() - t_wall
    launches = E.launch_count(local_rank, reset=True)
    log(f"timed region done: {wall_s:.2f} s for {args.steps} wave(s), {launches} launches")
    if args.dump_outputs and rank == 0:
        dumped = wave_outputs(outs)
        assert sum(a.nbytes for a in dumped.values()) <= 64 << 20
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
        log(f"outputs of the last timed wave written to {args.dump_outputs}: " + ", ".join(f"{k} {list(a.shape)}" for k, a in dumped.items()))
        del dumped, outs

    def stage(ev, a, b):
        return ev[a].elapsed_time(ev[b])
    step_ms = [a.elapsed_time(b) for a, b in spans]
    stages = {"stt_ms": statistics.mean(stage(e, "t0", "stt") for e in evs),
              "llm_prefill_ms": statistics.mean(stage(e, "stt", "prefill") for e in evs),
              "llm_decode_ms": statistics.mean(stage(e, "prefill", "llm") for e in evs),
              "tts_ms": statistics.mean(stage(e, "llm", "tts") for e in evs)}
    codec_ms = statistics.mean(sum(a.elapsed_time(b) for a, b in e["frames_mark"]) for e in evs)
    stages["tts_codec_postproc_ms"] = codec_ms
    stages["stt_decode_ms"] = statistics.mean(sum(a.elapsed_time(b) for a, b in e["whisper_mark"]) for e in evs)
    stages["tts_talker_predictor_ms"] = stages["tts_ms"] - codec_ms
    total_ms = sum(step_ms)

    # ---- results back to the ingest rank (first codec chunk's int16 audio + ids are what a client needs first): gather ----
    res = torch.zeros((S, 64), dtype=torch.int32, device=dev)
    ge = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    ge[0].record()
    shard.gather_to_ingest(res)
    ge[1].record()
    torch.cuda.synchronize()
    gather_ms = ge[0].elapsed_time(ge[1])

    # ---- single-session latency on an idle GPU + the loaded wave, through the handler classes (host PCM in, int16 out) ----
    e2e = None
    if not args.no_e2e:
        try:
            # ~70 Python threads (two per session + the batchers' engine threads) hand work to each other through the GIL: the
            # default 5 ms switch interval is longer than a whole batch window
            sys.setswitchinterval(0.0005)
            handlers = make_handlers(S, local_rank, L)
            log("handler instances built and warmed up")
            auds = [pcm_dev[i].cpu().numpy() for i in range(S)]
            e2e_wave(handlers[:1], auds, 1)                                    # warm-up
            single = [e2e_wave(handlers[:1], auds, 1) for _ in range(2)]
            log(f"single-session e2e: {[round(w['wall_s'], 2) for w in single]} s, errors {single[-1]['errors']}")
            e2e_wave(handlers, auds, S)                                        # warm-up of the loaded path
            log("loaded e2e warm-up wave done")
            barrier()

            def batcher_stats():
                out = {}
                for name, get in (("stt", lambda h: h[0].bundle.batcher), ("llm", lambda h: h[1].bundle.batcher), ("tts", lambda h: h[2].model.batcher)):
                    bs = {id(get(h)): get(h) for h in handlers if get(h) is not None}
                    out[name] = (sum(b.batches_run for b in bs.values()), sum(b.items_run for b in bs.values()))
                return out
            bs0 = batcher_stats()
            loaded = [e2e_wave(handlers, auds, S) for _ in range(2 if args.steps >= 4 else 1)]
            bs1 = batcher_stats()
            barrier()
            # latency under a steady load: the sessions' turns end evenly spread, at 70 % of the arrival rate the loaded wave sustained
            spacing = statistics.mean(w["wall_s"] for w in loaded) / S / 0.7
            order = np.random.default_rng(3).permutation(S)          # lanes interleaved, not lane 0 first
            staggered = e2e_wave(handlers, auds, S, offsets=[float(spacing * int(np.where(order == i)[0][0])) for i in range(S)])
            log(f"staggered wave (one turn end every {1e3 * spacing:.0f} ms): p50 latency {statistics.median(staggered['latency_ms']) if staggered['latency_ms'] else None}")
            # and at 30 %: the other end of the latency-vs-load curve (half the sessions keep the run short)
            spacing30 = statistics.mean(w["wall_s"] for w in loaded) / S / 0.3
            half = [int(i) for i in order[: max(2, S // 2)]]
            light = e2e_wave([handlers[i] for i in half], [auds[i] for i in half], len(half), offsets=[float(spacing30 * k) for k in range(len(half))])
            log(f"staggered wave (one turn end every {1e3 * spacing30:.0f} ms): p50 latency {statistics.median(light['latency_ms']) if light['latency_ms'] else None}")
            e2e = {"single": single, "loaded": loaded, "staggered": staggered, "staggered_spacing_s": spacing,
                   "light": light, "light_spacing_s": spacing30,
                   "batching": {k: {"launch_groups": bs1[k][0] - bs0[k][0], "requests": bs1[k][1] - bs0[k][1],
                                    "mean_batch": round((bs1[k][1] - bs0[k][1]) / max(1, bs1[k][0] - bs0[k][0]), 2)} for k in bs1}}
            log(f"loaded e2e waves: {[round(w['wall_s'], 2) for w in loaded]} s")
            for hs in handlers:
                for h in hs:
                    try:
                        h.cleanup()
                    except Exception:
                        pass
        except Exception as ex:  # never lose the headline line because of the handler-level section
            e2e = {"error": f"{type(ex).__name__}: {ex}"}
    clocks = sampler.stop() if rank == 0 else None

    e2e_wall = statistics.mean(w["wall_s"] for w in e2e["loaded"]) if e2e and "loaded" in e2e else float("nan")
    total_ms, e2e_wall_max = shard.max_over_ranks([total_ms, e2e_wall if e2e_wall == e2e_wall else 0.0], device=dev)

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = world * S * CYCLE_S / (ms_per_step / 1e3)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        # dominant stage of the step and its kernel's roofline
        shares = {k: v / ms_per_step for k, v in stages.items() if k in ("stt_ms", "llm_prefill_ms", "llm_decode_ms", "tts_talker_predictor_ms", "tts_codec_postproc_ms")}
        Sl = S // L                                                   # sessions of one lane
        n_llm_launch = (Sl + st.llm_b - 1) // st.llm_b                # per lane; the L lanes' launches run side by side
        llm_bytes = decode_bytes_llama(st.lg, MAX_NEW - 1, min(Sl, st.llm_b), LLM_PROMPT)
        llm_ms = stages["llm_decode_ms"] / n_llm_launch
        ach_llm_launch = llm_bytes / 1e9 / (llm_ms / 1e3)
        ach_llm = L * ach_llm_launch
        n_w_launch = (Sl + 15) // 16
        wb = decode_bytes_whisper(st.wg, len(PREFIX), MAX_NEW, min(Sl, 16))
        ach_w = L * wb / 1e9 / (stages["stt_decode_ms"] / n_w_launch / 1e3)
        lane_ctas = torch.cuda.get_device_properties(local_rank).multi_processor_count // L
        # the TTS frame loop: the same persistent kernel on the talker (1 step) and the code predictor (15 steps) per frame
        from speech_to_speech_b200.tts_model import TTS_GEOMETRIES
        tg = TTS_GEOMETRIES[TTS_GEOM]

        def _w(g):   # bf16 weight bytes of one decode step (all layers + one output head)
            qd, kvd = g["heads"] * g["head_dim"], g["kv_heads"] * g["head_dim"]
            return (g["layers"] * ((qd + 2 * kvd) * g["d_model"] + g["d_model"] * qd + 3 * g["ffn"] * g["d_model"]) + g["vocab"] * g["d_model"]) * 2
        frame_bytes = _w(tg["talker"]) + (tg["n_groups"] - 1) * _w(tg["predictor"])
        n_frame_launch = (Sl + st.tts_b - 1) // st.tts_b
        frame_ms = stages["tts_talker_predictor_ms"] / (F1 + F2) / n_frame_launch
        ach_tts = L * frame_bytes / 1e9 / (frame_ms / 1e3)
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("llama_decode", {}).get("dram_bytes_per_launch")
        roofline = {"kernel": f"llama_decode_kernel (persistent, {min(Sl, st.llm_b)} sessions x {MAX_NEW - 1} steps per launch, Llama-3-8B bf16; "
                              f"{L} launch(es) run concurrently, one per lane of {lane_ctas} CTAs)",
                    "bound": "hbm", "achieved": ach_llm, "peak": peak, "unit": "GB/s", "frac": ach_llm / peak, "traffic": traffic,
                    "achieved_note": f"sum over the {L} concurrent launches (each streams its own copy of the weights): "
                                     f"{L} x algorithmic_bytes_per_launch / launch_ms; achieved_per_launch is one launch alone",
                    "achieved_per_launch": ach_llm_launch, "concurrent_launches": L,
                    "algorithmic_bytes_per_launch": llm_bytes, "launch_ms": llm_ms, "launches_per_step": L * n_llm_launch,
                    "peak_source": peak_src, "share_of_step": shares["llm_decode_ms"], "stage_shares": shares}
        line = {
            "metric": METRIC, "value": value, "unit": "sessions", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 (Whisper, codec-decoder contractions) / bf16 (Llama, talker, code predictor) operands, f32 accumulate and residual streams", "data": "synthetic",
            "config": workload_config(world, S),
            "l2": "flushed between timed steps (256 MiB write); every stage streams > 126 MB of weights per launch",
            "lanes": {"per_gpu": L, "ctas_per_lane": lane_ctas, "sessions_per_lane": Sl,
                      "note": "SM partitions with their own engines and CUDA streams; stage_ms are lane 0's (all lanes run the same "
                              "sequence side by side), ms_per_step spans all lanes"},
            "turn_gpu_ms_per_session": ms_per_step / S, "stage_ms": stages, "wall_s_timed_region": wall_s,
            "gpu_launches": int(launches), "roofline": roofline, "clocks": clocks,
            "session_shard_exchange": {"collective": "torch.distributed scatter (PCM from the ingest rank) + gather (results), NCCL send/recv",
                                       "scatter_ms": scatter_ms, "gather_ms": gather_ms,
                                       "bytes_in_per_session": N_SAMPLES * 4, "bytes_out_per_session": 64 * 4},
            "whisper_decode_roofline": {"kernel": f"whisper_decode_kernel (persistent, {min(Sl, 16)} sessions per launch, {L} concurrent)",
                                        "bound": "hbm", "algorithmic_bytes_per_launch": wb, "launches_per_step": L * n_w_launch,
                                        "achieved": ach_w, "peak": peak, "unit": "GB/s", "frac": ach_w / peak},
            "tts_frame_roofline": {"kernel": f"llama_decode_kernel on the talker (1 step) + code predictor ({tg['n_groups'] - 1} steps), "
                                             f"{min(Sl, st.tts_b)} sessions per launch, {L} concurrent", "bound": "hbm",
                                   "algorithmic_bytes_per_frame": frame_bytes, "ms_per_frame": frame_ms, "achieved": ach_tts, "peak": peak,
                                   "unit": "GB/s", "frac": ach_tts / peak,
                                   "note": "latency-bound: ~630 grid-barrier phases of 5-10 us per frame (profiles/r2/tts_phase_trace.txt); "
                                           "weights are KV-free attention-light (<= 512 positions), KV bytes not counted"},
            "stt_only_sessions": world * S * AUDIO_S / (stages["stt_ms"] / 1e3),
        }
        if e2e and "loaded" in e2e:
            lat_loaded = [x for w in e2e["loaded"] for x in w["latency_ms"]]
            rtf_loaded = [x for w in e2e["loaded"] for x in w["rtf"]]
            lat_single = [x for w in e2e["single"] for x in w["latency_ms"]]
            e2e_val = world * S * CYCLE_S / e2e_wall_max if e2e_wall_max > 0 else None
            realtime = bool(rtf_loaded) and min(rtf_loaded) >= 1.0
            line["e2e"] = {"value": e2e_val, "unit": "sessions", "h2d_bytes_per_step": S * N_SAMPLES * 4,
                           "d2h_bytes_per_step": S * int((F1 + F2) * 1920 * 2 / 3) * 2,
                           "wall_s_per_wave": e2e_wall_max, "path": "B200WhisperSTTHandler -> B200LanguageModelHandler -> B200Qwen3TTSHandler, "
                           "per session an LLM thread feeding a TTS thread through a queue (the reference's thread-per-stage shape), "
                           "shared engines + session batchers per lane",
                           "tts_rtf_min": min(rtf_loaded) if rtf_loaded else None, "tts_rtf_p50": statistics.median(rtf_loaded) if rtf_loaded else None,
                           "real_time": realtime, "errors": [e for w in e2e["loaded"] for e in w["errors"]][:3],
                           "batching": e2e.get("batching")}
            line["latency_ms_p50"] = statistics.median(lat_loaded) if lat_loaded else None
            line["latency_ms_p50_single_session"] = statistics.median(lat_single) if lat_single else None
            lat_st = sorted(e2e.get("staggered", {}).get("latency_ms", []))
            if lat_st:
                line["latency_ms_at_70pct_load"] = {"p50": statistics.median(lat_st), "p90": lat_st[min(len(lat_st) - 1, int(0.9 * len(lat_st)))],
                                                    "turn_end_every_ms": 1e3 * e2e["staggered_spacing_s"], "sessions": len(lat_st),
                                                    "errors": e2e["staggered"]["errors"]}
            lat_30 = sorted(e2e.get("light", {}).get("latency_ms", []))
            if lat_30:
                line["latency_ms_at_30pct_load"] = {"p50": statistics.median(lat_30), "p90": lat_30[min(len(lat_30) - 1, int(0.9 * len(lat_30)))],
                                                    "turn_end_every_ms": 1e3 * e2e["light_spacing_s"], "sessions": len(lat_30),
                                                    "errors": e2e["light"]["errors"]}
            line["latency_note"] = ("audio-in (VADAudio.created_at_s) -> first int16 block out of the TTS handler; 'single' = one session on an "
                                    "idle GPU (on its lane's SM partition), 'latency_ms_p50' = the S sessions of a wave that all stop speaking at the same instant (worst case), "
                                    "'latency_ms_at_70pct_load' / 'latency_ms_at_30pct_load' = turn ends evenly spread at 70 % / 30 % of the rate the loaded wave sustains")
        elif e2e:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            log("cpu baseline (child process)")
            line["cpu_baseline"] = cpu_baseline_subprocess(args.cpu_baseline_turns)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
