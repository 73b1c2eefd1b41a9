"""CPU: the drop-in boundary.  With the reference (the upstream `speech_to_speech` package, oracle/upstream.py) importable our handlers must
subclass ITS base classes, register in ITS backend registry and honour ITS process() contract; the device work is
replaced by a fake engine exactly the way the reference's own tests fake their models
(T/test_whisper_language_detection.py:52-141).  Without the reference the same contract is checked on the mirror."""
from queue import Queue
from threading import Event, Thread
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import upstream

HAVE_REF = upstream.importable()

from speech_to_speech_b200.host import resolve  # noqa: E402
from speech_to_speech_b200.handlers import whisper_stt_handler as WH  # noqa: E402


class FakeEngine:
    def __init__(self):
        self.calls = []

    def transcribe(self, audio, opts):
        self.calls.append(("transcribe", len(audio[0]), list(opts.prefix), opts.max_new_tokens))
        return [[11, 22, 33, opts.eos_id] for _ in audio]

    detect_result = "third"   # "third": lang_ids[2]; an int: that id; None: an id outside the table; an Exception: raised

    def detect_language_host(self, audio, sot, lang_ids):
        self.calls.append(("detect", sot, len(audio)))
        if isinstance(self.detect_result, Exception):
            raise self.detect_result
        if self.detect_result is None:
            return -1
        return lang_ids[2] if self.detect_result == "third" else self.detect_result

    def transcribe_auto(self, audio, sot, lang_ids, make_opts):
        """Detection + decode on one encoder pass (engine.WhisperEngine.transcribe_auto): a real engine always answers with
        one of lang_ids; `None` models an id outside the handler's table."""
        langs = [self.detect_language_host(a, sot, lang_ids) for a in audio]
        opts = make_opts(langs)
        rows = opts.prefix_rows
        for a, row in zip(audio, rows):
            self.calls.append(("transcribe", len(a), list(row), opts.max_new_tokens))
        return [[11, 22, 33, opts.eos_id] for _ in audio], langs

    def close(self):
        self.calls.append(("close",))


def make_handler(language="en", gen_kwargs=None, max_batch=1, engine=None):
    """Bypass setup() (model load) like the reference's tests do; wire the attributes process() reads."""
    api = resolve()
    h = object.__new__(WH.B200WhisperSTTHandler)
    h.stop_event, h.queue_in, h.queue_out = Event(), Queue(), Queue()
    h.pipeline_index, h._times = None, []
    h.speculative_turns = None
    h.device, h.device_index, h.torch_dtype = "cuda", 0, "float16"
    h.gen_kwargs = dict(gen_kwargs or {"max_new_tokens": 128, "task": "transcribe"})
    h.start_language = language
    h.last_language = language if language != "auto" else None
    if h.last_language is not None:
        h.gen_kwargs["language"] = h.last_language
    from speech_to_speech_b200 import _lib

    class _E:  # the two names process() takes from the engine module
        WhisperDecodeOptions = __import__("speech_to_speech_b200.engine", fromlist=["x"]).WhisperDecodeOptions if False else None

    from dataclasses import dataclass

    @dataclass
    class Opts:
        prefix: list
        eos_id: int
        max_new_tokens: int = 128
        suppress: tuple = ()
        begin_suppress: tuple = ()
        prefix_rows: object = None

    h._E = SimpleNamespace(WhisperDecodeOptions=Opts)
    h.max_batch, h.batch_wait_s, h._shared_key = max_batch, 0.2, None
    h.bundle = WH._EngineBundle(h._E, engine or FakeEngine(), WH.TokenTable.synthetic(51865), lambda ids: " ".join(map(str, ids)),
                                max_batch, 0.2)
    h.engine, h.tokens, h._decode_text = h.bundle.engine, h.bundle.tokens, h.bundle.decode_text
    h.processor = None
    return api, h


def vad(api, mode="final", n=16000):
    return api.VADAudio(audio=np.zeros(n, np.float32), mode=mode, turn_id="t1", turn_revision=3)


def test_base_classes_come_from_the_reference_when_present():
    api = resolve()
    assert api.source == ("reference" if HAVE_REF else "mirror")
    assert issubclass(WH.B200WhisperSTTHandler, api.BaseSTTHandler)
    assert issubclass(WH.B200WhisperSTTHandler, api.BaseHandler)


def test_process_yields_transcription_with_reference_fields():
    api, h = make_handler("en")
    item = vad(api)
    out = list(h.process(item))
    assert len(out) == 1 and isinstance(out[0], api.Transcription)
    t = out[0]
    assert t.text == "11 22 33" and t.language_code == "en" and t.turn_id == "t1" and t.turn_revision == 3
    assert t.speech_stopped_at_s == item.created_at_s
    kind, n, prefix, max_new = h.engine.calls[-1]
    tok = h.tokens
    assert kind == "transcribe" and prefix == [tok.sot, tok.lang_to_id["en"], tok.transcribe, tok.no_timestamps] and max_new == 128


def test_progressive_mode_yields_partial():
    api, h = make_handler("en")
    out = list(h.process(vad(api, mode="progressive")))
    assert len(out) == 1 and isinstance(out[0], api.PartialTranscription) and out[0].text == "11 22 33"


def test_absent_mode_still_yields_transcription():
    """Items without a `mode` attribute are final segments (reference tests/test_whisper_progressive_transcription.py:215)."""
    api, h = make_handler("en")
    item = SimpleNamespace(audio=np.zeros(8000, np.float32), turn_id="t9", turn_revision=1, created_at_s=12.5)
    out = list(h.process(item))
    assert len(out) == 1 and isinstance(out[0], api.Transcription) and out[0].speech_stopped_at_s == 12.5


def test_auto_language_detects_then_forces_and_marks_auto():
    api, h = make_handler("auto")
    out = list(h.process(vad(api)))
    detected = h.tokens.id_to_lang[list(h.tokens.lang_to_id.values())[2]]
    assert out[0].language_code == detected + "-auto"
    kinds = [c[0] for c in h.engine.calls]
    assert kinds == ["detect", "transcribe"]
    assert h.engine.calls[-1][2][1] == h.tokens.lang_to_id[detected]
    assert h.last_language == (detected if detected in WH.SUPPORTED_LANGUAGES else None)


# ---- the language bookkeeping scenarios of the reference's tests/test_whisper_language_detection.py, on this handler ----
def test_detection_does_not_mutate_gen_kwargs():
    api, h = make_handler("auto", gen_kwargs={"task": "transcribe"})
    list(h.process(vad(api)))
    assert h.gen_kwargs == {"task": "transcribe"}


def test_unsupported_detected_language_is_reported_not_retranscribed():
    """A detected language outside SUPPORTED_LANGUAGES is forced for this utterance and reported, one transcription
    only, and does not become the sticky fallback (reference :287-306)."""
    api, h = make_handler("auto")
    h.last_language = "de"
    h.engine.detect_result = h.tokens.lang_to_id["ru"]
    out = list(h.process(vad(api)))[0]
    assert out.language_code == "ru-auto" and h.last_language == "de"
    calls = [c for c in h.engine.calls if c[0] == "transcribe"]
    assert len(calls) == 1 and calls[0][2][1] == h.tokens.lang_to_id["ru"]


def test_no_detection_falls_back_to_last_language_then_english():
    api, h = make_handler("auto")
    h.engine.detect_result = None                      # the detector returns nothing usable
    h.last_language = "de"
    assert list(h.process(vad(api)))[0].language_code == "de-auto"
    h.last_language = None
    out = list(h.process(vad(api)))[0]
    assert out.language_code == "en-auto"
    assert [c[0] for c in h.engine.calls].count("transcribe") == 2   # one generate per utterance, no retry


def test_detect_language_failure_is_survivable():
    api, h = make_handler("auto")
    h.last_language = "de"
    h.engine.detect_result = RuntimeError("no kernel")
    out = list(h.process(vad(api)))[0]
    assert out.text == "11 22 33" and out.language_code == "de-auto"
    assert [c[0] for c in h.engine.calls].count("transcribe") == 1


def test_language_code_has_no_auto_suffix_when_start_language_is_not_auto():
    api, h = make_handler("en")
    assert list(h.process(vad(api)))[0].language_code == "en"


def test_runs_inside_the_stage_thread_loop_and_survives_errors():
    api, h = make_handler("en")
    th = Thread(target=h.run)
    th.start()
    h.queue_in.put(vad(api))
    first = h.queue_out.get(timeout=5)
    assert isinstance(first, api.Transcription)
    boom = vad(api)
    h.engine.transcribe = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("device error"))
    h.queue_in.put(boom)  # logged + dropped by the loop (S/baseHandler.py:162-163)
    h.queue_in.put(api.PIPELINE_END)
    assert h.queue_out.get(timeout=5) == api.PIPELINE_END
    th.join(timeout=5)
    assert not th.is_alive() and ("close",) in h.engine.calls


def test_cpu_device_is_rejected_no_fallback():
    api = resolve()
    with pytest.raises(ValueError, match="no CPU fallback"):
        WH.B200WhisperSTTHandler(Event(), queue_in=Queue(), queue_out=Queue(),
                                 setup_kwargs={"model_name": "random:micro", "device": "cpu"})


def test_token_table_from_generation_config():
    gc = SimpleNamespace(decoder_start_token_id=50258, eos_token_id=50257, task_to_id={"transcribe": 50359, "translate": 50358},
                         no_timestamps_token_id=50363, lang_to_id={"<|en|>": 50259, "<|de|>": 50261, "<|yue|>": 50358},
                         suppress_tokens=[1, 2], begin_suppress_tokens=[220, 50257])
    t = WH.TokenTable.from_generation_config(gc)
    assert t.lang_to_id == {"en": 50259, "de": 50261, "yue": 50358} and t.suppress == [1, 2] and t.eos == 50257


@pytest.mark.skipif(not HAVE_REF, reason="the upstream speech_to_speech package is not available")
def test_registers_in_the_reference_backend_registry():
    import speech_to_speech_b200.registry as r
    specs = r.register()
    from speech_to_speech.backend_registry import LLM_BACKENDS, STT_BACKENDS
    from speech_to_speech.arguments_classes.whisper_stt_arguments import WhisperSTTHandlerArguments
    assert STT_BACKENDS["b200-whisper"] is specs["b200-whisper"] and "b200-transformers" in LLM_BACKENDS
    cfg = specs["b200-whisper"].normalize(WhisperSTTHandlerArguments(stt_model_name="random:small"))
    assert cfg["model_name"] == "random:small" and cfg["device"] == "cuda" and cfg["gen_kwargs"]["max_new_tokens"] == 128


@pytest.mark.skipif(not HAVE_REF, reason="the upstream speech_to_speech package is not available")
def test_tts_spec_and_overrides_cover_all_three_slots():
    """`b200-qwen3` reuses the reference's Qwen3TTSHandlerArguments / prefix; install_overrides() swaps the classes behind the
    unchanged names whisper / transformers / qwen3 (the lazy factories resolve to our modules, nothing is imported yet)."""
    import dataclasses
    import speech_to_speech_b200.registry as r
    import speech_to_speech.backend_registry as br
    from speech_to_speech.arguments_classes.qwen3_tts_arguments import Qwen3TTSHandlerArguments
    saved = (dict(br.STT_BACKENDS), dict(br.LLM_BACKENDS), dict(br.TTS_BACKENDS))
    try:
        specs = r.register()
        tts = specs["b200-qwen3"]
        assert br.TTS_BACKENDS["b200-qwen3"] is tts and tts.kind == "tts" and tts.config_type is Qwen3TTSHandlerArguments
        cfg = tts.normalize(Qwen3TTSHandlerArguments(qwen3_tts_model_name="random:micro", qwen3_tts_speaker="Aiden"))
        assert cfg["model_name"] == "random:micro" and cfg["speaker"] == "Aiden" and cfg["blocksize"] == 512
        before = {k: br.TTS_BACKENDS[k].create_handler for k in ("qwen3",)}
        r.install_overrides()
        assert br.TTS_BACKENDS["qwen3"].create_handler is not before["qwen3"]
        assert br.TTS_BACKENDS["qwen3"].config_type is Qwen3TTSHandlerArguments
        assert br.LLM_BACKENDS["transformers"].name == "transformers" and br.STT_BACKENDS["whisper"].name == "whisper"
        for spec in (br.STT_BACKENDS["whisper"], br.LLM_BACKENDS["transformers"], br.TTS_BACKENDS["qwen3"]):
            assert dataclasses.is_dataclass(spec) and callable(spec.create_handler)
    finally:
        for d, s in zip((br.STT_BACKENDS, br.LLM_BACKENDS, br.TTS_BACKENDS), saved):
            d.clear(); d.update(s)


@pytest.mark.skipif(not HAVE_REF, reason="the upstream speech_to_speech package is not available")
def test_llm_handler_implements_the_reference_hooks():
    from speech_to_speech_b200.handlers import language_model_handler as LH
    from speech_to_speech.LLM.language_model import BaseLanguageModelHandler
    assert issubclass(LH.B200LanguageModelHandler, BaseLanguageModelHandler)
    assert not getattr(LH.B200LanguageModelHandler, "__abstractmethods__", None)


def test_token_streamer_chunks_and_stops_at_eos():
    from speech_to_speech_b200.handlers.language_model_handler import TokenStreamer, _IdTokenizer
    import torch

    class FakeLlama:
        device = "cpu"
        cfg = SimpleNamespace(max_prefill=4)

        def __init__(self):
            self.script = list(range(100, 120)) + [7]  # 7 = eos
            self.pos = 0
            self.prefills = []

        def reset(self, slot):
            self.pos = 0

        def prefill(self, slot, ids):
            self.prefills.append(list(ids))
            return torch.tensor([self.script[0]]), None

        def decode(self, slots, first, n, eos_id=-1):
            self.pos += 1 if self.pos == 0 else 0
            out = self.script[self.pos:self.pos + n]
            self.pos += n
            ln = len(out)
            if eos_id in out:
                ln = out.index(eos_id) + 1
            return torch.tensor([out + [eos_id] * (n - len(out))]), torch.tensor([ln])

    import speech_to_speech_b200.handlers.language_model_handler as LH
    eng = FakeLlama()
    real_tensor = torch.tensor
    tok = _IdTokenizer(1000)
    st = TokenStreamer(eng, lambda ids: tok.decode(ids), [7], chunk=5)
    torch_tensor = torch.tensor
    try:
        torch.tensor = lambda data, dtype=None, device=None: real_tensor(data, dtype=dtype)  # no CUDA on the CPU box
        text = "".join(st.stream(list(range(10)), max_new_tokens=64))
    finally:
        torch.tensor = torch_tensor
    assert eng.prefills == [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]]  # chunked prefill
    assert st.generated == list(range(100, 120)) and text == tok.decode(range(100, 120))
