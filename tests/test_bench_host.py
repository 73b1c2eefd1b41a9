"""Host-side pieces of bench.py that run without a GPU: the workload description both arms print, the byte models behind the
roofline numbers, the ncu window over TTS chunks, the lane fan-out of a wave, and the arrays --dump-outputs writes."""
import importlib.util
import os
import subprocess
import sys
import threading
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_cli_parses_and_documents_the_contract_flags():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--sessions", "--lanes", "--dump-outputs"):
        assert flag in out.stdout


def test_workload_is_baseline_config_2_and_identical_for_both_arms(bench):
    a, b = bench.workload_config(1, 32), bench.workload_config(1, 32)
    assert a == b and a["sessions_per_gpu"] == 32 and "l2" not in a and "lanes" not in a      # arm-specific keys live outside `config`
    assert bench.F1 + bench.F2 == a["tts_frames"] == 480 and abs(a["cycle_s"] - 48.4) < 1e-9
    assert a["stt_tokens"] == 128 and a["llm_reply_tokens"] == 128 and a["tts_chunk_frames"] == 8 and a["tts_left_context"] == 25


def test_byte_models_match_the_published_geometries(bench):
    from oracle import weights as W
    g = W.LLAMA_GEOMETRIES["llama-3-8b"]
    per_step = bench.decode_bytes_llama(g, 1, 1, 0)
    assert 15.0e9 < per_step < 15.2e9            # 15.0 GB of bf16 weights per token (SURVEY.md Appendix A) + one KV row
    eight = bench.decode_bytes_llama(g, 127, 8, 64)
    assert 1.92e12 < eight < 1.93e12             # the figure the roofline uses; ncu measured 1.958 TB of DRAM traffic
    wg = W.WHISPER_GEOMETRIES["small"]
    assert 1.5e11 < bench.decode_bytes_whisper(wg, 4, 128, 16) < 1.6e11


def test_tts_profile_window_brackets_the_chosen_chunks_of_all_lanes(bench):
    events = []
    cudart = types.SimpleNamespace(cudaProfilerStart=lambda: events.append("start"), cudaProfilerStop=lambda: events.append("stop"))
    stream = types.SimpleNamespace(synchronize=lambda: events.append("sync"))
    torch = types.SimpleNamespace(cuda=types.SimpleNamespace(cudart=lambda: cudart, current_stream=lambda: stream))
    w = bench.TtsProfileWindow(torch, lanes=2, n=2, first=2)

    def lane():
        for ci in range(6):
            w.chunk_begin(ci)
            w.chunk_end(ci)
    ths = [threading.Thread(target=lane) for _ in range(2)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    assert events.count("start") == 1 and events.count("stop") == 1 and events.count("sync") == 2
    assert events[0] == "start" and events[-1] == "stop"


def test_e2e_wave_runs_the_stages_in_their_own_threads_and_honours_offsets(bench):
    """bench.e2e_wave with fake handlers: STT -> LLM thread -> queue -> TTS thread per session; a sentence is spoken as soon as the
    LLM has produced it (the LLM keeps generating meanwhile); offsets stagger the turn ends; a failing session is reported."""
    import time
    import numpy as np
    t_wave = time.perf_counter()
    started = {}

    class STT:
        def __init__(self, i):
            self.i = i

        def process(self, vad):
            started[self.i] = time.perf_counter() - t_wave
            yield types.SimpleNamespace(text="hi", speech_stopped_at_s=getattr(vad, "created_at_s", None))

    class LLM:
        def __init__(self, fail=False):
            self.streamer = types.SimpleNamespace(generated=[])
            self.fail = fail

        def generate_text_stream(self, prompt, max_new_tokens=128):
            self.streamer.generated = []
            for k in range(max_new_tokens // 4):
                time.sleep(0.001)
                self.streamer.generated += [1, 2, 3, 4]
                if self.fail and k == 3:
                    raise RuntimeError("boom")
                yield "x"

    class TTS:
        def __init__(self):
            self.spoken = []

        def process(self, item):
            self.spoken.append((len(item.text), self.max_new_tokens))
            for _ in range(3):
                time.sleep(0.002)
                yield np.zeros(512, np.int16)

    hs = [(STT(i), LLM(fail=(i == 2)), TTS()) for i in range(3)]
    auds = [np.zeros(1600, np.float32)] * 3
    r = bench.e2e_wave(hs, auds, 3, offsets=[0.0, 0.05, 0.1])
    assert len(r["latency_ms"]) == 2 and all(0 < x < 2000 for x in r["latency_ms"])        # sessions 0 and 1; session 2 failed
    assert len(r["errors"]) == 1 and "boom" in r["errors"][0]
    assert started[1] >= 0.045 and started[2] >= 0.09                                         # the offsets were slept before the turn end
    for i in (0, 1):
        assert hs[i][2].spoken == [(bench.FIRST_SENTENCE, bench.F1), (bench.MAX_NEW - bench.FIRST_SENTENCE, bench.F2)]
    assert all(x > 0 for x in r["rtf"])


def test_wave_outputs_put_every_session_in_order_as_float32(bench, monkeypatch):
    """bench.wave_outputs on what wave_device collects for 2 lanes x 3 sessions (two LLM / TTS launches per lane, two TTS
    utterances of 2 and 1 chunks): every value names its session, so the order across lanes, launches and chunks is checked."""
    import numpy as np
    import torch
    monkeypatch.setattr(bench, "DUMP_AUDIO_SAMPLES", 50)

    def lane(l):
        sid = torch.arange(3, dtype=torch.int32) + 3 * l
        ids = lambda rows, n: sid[rows, None].repeat(1, n)
        chunk = lambda n: ([ids(slice(0, 2), n * 16).view(2, n, 16), ids(slice(2, 3), n * 16).view(1, n, 16)],
                           [torch.full((4 * n,), int(s), dtype=torch.int16) for s in sid])
        return {"stt": [ids(slice(0, 3), 128)], "llm_first": [sid], "llm": [ids(slice(0, 2), 127), ids(slice(2, 3), 127)],
                "tts": [[chunk(8), chunk(2)], [chunk(5)]]}
    out = bench.wave_outputs([lane(0), lane(1)])
    assert all(a.dtype == np.float32 for a in out.values())
    col = np.arange(6, dtype=np.float32)[:, None]
    assert np.array_equal(out["stt_token_ids"], np.repeat(col, 128, 1))
    assert np.array_equal(out["llm_token_ids"], np.repeat(col, 128, 1))
    assert out["tts_codes_first_sentence"].shape == (6, 10, 16) and out["tts_codes_rest"].shape == (6, 5, 16)
    assert (out["tts_codes_first_sentence"] == col[:, :, None]).all() and (out["tts_codes_rest"] == col[:, :, None]).all()
    idx = out["tts_audio_int16_sample_index"]
    assert idx.shape == (50, 2) and idx[:, 1].max() < 4 * 15 and len({tuple(r) for r in idx.tolist()}) == 50
    assert np.array_equal(out["tts_audio_int16_sample"], idx[:, 0])
    again = bench.wave_outputs([lane(0), lane(1)])
    assert np.array_equal(again["tts_audio_int16_sample_index"], idx)          # a fixed sample: runs compare element for element
