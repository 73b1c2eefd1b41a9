"""CPU contract tests of the B200 TTS handler slot with a fake model object (the reference's own test strategy: bypass the
device, inject fakes -- T/test_qwen3_tts_handler_backend.py:18-19, 756-762).  Both base classes are exercised: the reference's
Qwen3TTSHandler when the upstream `speech_to_speech` package is importable (oracle/upstream.py), and the mirror used without it."""
import importlib
import os
import sys
import zlib
from queue import Queue
from threading import Event

import numpy as np
import pytest

from oracle import upstream

HAVE_UPSTREAM = upstream.importable()
LONG = " ".join(["This is a deliberately long sentence for the Qwen3 TTS budget estimator."] * 12)
CJK_SHORT = "我懂，心情不好时会让人特别疲惫。"
CJK_LONG = ("上海是一座充满活力的现代化大都市，既有繁华的金融中心和摩天大楼，也有老城厢的弄堂风情"
            "和江南水乡的韵味。这里交通便利，餐饮选择丰富，从精致西餐到地道小馆应有尽有。同时，上海"
            "还是文化与创新的交汇点，艺术展览、科技展会和国际活动频繁。如果你喜欢快节奏的生活和多元"
            "的氛围，上海会是个很吸引人的地方。你想了解哪方面的具体信息呢？")


class FakeModel:
    """(audio, sr, timing) tuples like the reference's fakes (T/test_qwen3_tts_handler_backend.py:756-762)."""

    def __init__(self, chunks):
        import types
        self.chunks, self.calls = chunks, []
        self.model = types.SimpleNamespace(model=types.SimpleNamespace(tts_model_type="custom_voice"))

    def get_supported_speakers(self):
        return ["aiden"]

    def warmup(self, prefill_len=100):
        self.calls.append(("warmup", prefill_len))

    def generate_custom_voice_streaming(self, **kw):
        self.calls.append(("gen", kw))
        for c in self.chunks:
            yield (c, 24000, {})

    def close(self):
        pass


def _handler_module(use_reference: bool):
    """Import handlers.qwen3_tts_handler against the reference base or the mirror base."""
    for m in [k for k in sys.modules if k.startswith("speech_to_speech_b200.handlers.qwen3_tts_handler")]:
        del sys.modules[m]
    if use_reference and not HAVE_UPSTREAM:
        pytest.skip("the upstream speech_to_speech package is not available")
    # the mirror base is only chosen when `speech_to_speech` cannot be imported: block it (a None entry in sys.modules) for
    # the duration of the import and PUT the already-imported modules BACK, so that other test modules keep seeing the class
    # objects they imported
    hidden = {}
    if not use_reference:
        for m in [k for k in sys.modules if k == "speech_to_speech" or k.startswith("speech_to_speech.")]:
            hidden[m] = sys.modules.pop(m)
        sys.modules["speech_to_speech"] = None
    try:
        mod = importlib.import_module("speech_to_speech_b200.handlers.qwen3_tts_handler")
    finally:
        if not use_reference:
            del sys.modules["speech_to_speech"]
        for m in [k for k in sys.modules if (k == "speech_to_speech" or k.startswith("speech_to_speech.")) and k in hidden]:
            del sys.modules[m]
        sys.modules.update(hidden)
    want = "speech_to_speech.TTS.qwen3_tts_handler" if use_reference else "speech_to_speech_b200.host.mirror_tts"
    if mod._Base.__module__ != want:
        pytest.skip(f"base class resolved to {mod._Base.__module__}")
    return mod


def _make(mod, fake, monkeypatch, **kw):
    monkeypatch.setattr(mod, "acquire_shared", lambda key, build, closer: fake)
    monkeypatch.setattr(mod, "release_shared", lambda key: None)
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    if hasattr(sys.modules[mod._Base.__module__], "console"):
        monkeypatch.setattr(sys.modules[mod._Base.__module__].console, "print", lambda *a, **k: None)
    return mod.B200Qwen3TTSHandler(Event(), queue_in=Queue(), queue_out=Queue(), setup_args=(Event(),),
                                   setup_kwargs=dict(model_name="random:micro", device="cuda", **kw))


def _tts_input(mod, text):
    try:
        from speech_to_speech.pipeline.messages import TTSInput
        if mod._Base.__module__.startswith("speech_to_speech."):
            return TTSInput(text=text)
    except Exception:
        pass
    from speech_to_speech_b200.host.mirror import TTSInput
    return TTSInput(text=text)


@pytest.mark.parametrize("use_reference", [True, False])
def test_process_yields_int16_blocks_and_passes_the_reference_kwargs(monkeypatch, use_reference):
    mod = _handler_module(use_reference)
    t = np.arange(24000, dtype=np.float32) / 24000
    chunks = [0.3 * np.sin(2 * np.pi * 220 * t[i:i + 4800]).astype(np.float32) for i in range(0, 24000, 4800)]
    fake = FakeModel(chunks)
    h = _make(mod, fake, monkeypatch, speaker="Aiden", blocksize=512, max_sessions=3)
    assert ("warmup", 100) in fake.calls                              # setup() warmed the model up like the reference (:555-572)
    fake.calls.clear()
    out = list(h.process(_tts_input(mod, "Hello there.")))
    assert out and all(isinstance(b, np.ndarray) and b.dtype == np.int16 and b.shape == (512,) for b in out)
    # 1 s of 24 kHz audio -> 16000 samples @ 16 kHz minus the trimmed ramp-up, in 512-sample blocks (tail zero-padded)
    assert 15000 // 512 <= len(out) <= 16000 // 512 + 1
    (kind, kw), = [c for c in fake.calls if c[0] == "gen"]
    assert kw["text"] == "Hello there." and kw["speaker"] == "Aiden" and kw["chunk_size"] == 8
    assert kw["max_new_tokens"] == 360 and kw["non_streaming_mode"] is True and kw["language"] == "auto"
    # bit-identical to the reference's own post-processing of the same chunks (scipy resample_poly + int16)
    from oracle import tts_post_ref as T
    ref = np.concatenate([T.postproc(c) for c in chunks])
    got = np.concatenate(out)
    start = max(0, int(np.argmax(np.abs(ref) > 327)) - 640)
    assert np.array_equal(got[: len(ref) - start], ref[start:])
    h.cleanup()


@pytest.mark.parametrize("use_reference", [True, False])
def test_end_of_response_yields_audio_response_done(monkeypatch, use_reference):
    mod = _handler_module(use_reference)
    h = _make(mod, FakeModel([np.full(512, 0.1, np.float32)]), monkeypatch)
    if mod._Base.__module__.startswith("speech_to_speech."):
        from speech_to_speech.pipeline.messages import AUDIO_RESPONSE_DONE, EndOfResponse
    else:
        from speech_to_speech_b200.host.mirror import AUDIO_RESPONSE_DONE, EndOfResponse
    assert list(h.process(EndOfResponse())) == [AUDIO_RESPONSE_DONE]


@pytest.mark.parametrize("use_reference", [True, False])
def test_token_budget_goldens_of_the_reference(monkeypatch, use_reference):
    """The reference's pinned values (T/test_qwen3_tts_handler_backend.py:915-964): 360, 360 (CJK short), 576 (CJK long), cap."""
    mod = _handler_module(use_reference)
    h = object.__new__(mod.B200Qwen3TTSHandler)
    h.streaming_chunk_size, h.max_new_tokens = 8, 1536
    assert h._estimate_max_new_tokens("Hello there.") == 360
    assert h._estimate_max_new_tokens(CJK_SHORT) == 360
    assert h._estimate_max_new_tokens(CJK_LONG) == 576
    b = h._estimate_max_new_tokens(LONG)
    assert b > 360 and b % 8 == 0 and b <= 1536
    h.max_new_tokens = 400
    assert h._estimate_max_new_tokens(LONG) == 400
    h.max_new_tokens = 2400
    assert h._estimate_max_new_tokens(" ".join([LONG] * 3)) > 1536
    assert h._estimate_max_new_tokens("") == 360


def test_mirror_budget_equals_the_reference_function_on_random_text(golden_dir):
    """The mirror's `_estimate_max_new_tokens` against the budgets the reference's Qwen3TTSHandler gave for the same seeded
    random texts (tests/golden/make_golden.py tts_handler)."""
    from speech_to_speech_b200.host.mirror_tts import MirrorQwen3TTSHandler
    gold = np.load(os.path.join(golden_dir, "tts_handler_reference.npz"))
    b = object.__new__(MirrorQwen3TTSHandler)
    rng = np.random.default_rng(0)
    alphabet = list("abcdefghij klmnop, qrst. uvw! xyz? 上海是一座城市，。") + [" "] * 6
    for (chunk, cap), crcs, budgets in zip(gold["budget_cases"].tolist(), gold["budget_text_crc32"], gold["budgets"]):
        b.streaming_chunk_size, b.max_new_tokens = chunk, cap
        for crc, budget in zip(crcs.tolist(), budgets.tolist()):
            text = "".join(rng.choice(alphabet, int(rng.integers(0, 900))))
            assert zlib.crc32(text.encode()) == crc            # the same text the reference was given
            assert b._estimate_max_new_tokens(text) == budget, text


@pytest.mark.parametrize("use_reference", [True, False])
def test_cpu_device_is_rejected_and_errors_do_not_kill_the_stage(monkeypatch, use_reference):
    mod = _handler_module(use_reference)
    monkeypatch.setattr(mod, "acquire_shared", lambda key, build, closer: FakeModel([]))
    with pytest.raises(ValueError):
        mod.B200Qwen3TTSHandler(Event(), queue_in=Queue(), queue_out=Queue(), setup_args=(Event(),),
                                setup_kwargs=dict(model_name="random:micro", device="cpu"))

    class Boom(FakeModel):
        def generate_custom_voice_streaming(self, **kw):
            raise RuntimeError("device fell over")
            yield  # pragma: no cover
    h = _make(mod, Boom([]), monkeypatch)
    assert list(h.process(_tts_input(mod, "Hi."))) == []      # logged and swallowed like the reference (:864-865)


def test_device_audio_satisfies_the_numpy_tuple_contract():
    import torch
    from speech_to_speech_b200.tts_model import DeviceAudio, byte_tokenizer
    x = torch.linspace(-1, 1, 100)
    d = DeviceAudio(x)
    a = np.asarray(d, dtype=np.float32)
    assert a.dtype == np.float32 and a.shape == (100,) and d.size == 100 and np.allclose(a, x.numpy())
    tok = byte_tokenizer(512)
    ids = tok("Hello, wörld")
    assert ids and all(0 <= i < 496 for i in ids)


@pytest.mark.parametrize("use_reference", [True, False])
def test_concurrent_handlers_on_the_real_model_object_with_a_fake_engine(monkeypatch, use_reference):
    """The handler slot on top of tts_model.B200Qwen3TTS itself (session batcher, prefetched chunk requests, DeviceAudio) with a
    fake engine and a fake device post-processor: 4 handler threads speak at once, every one of them receives its own audio in
    order, and the engine saw merged launches."""
    import threading
    import time
    import types
    import torch
    mod = _handler_module(use_reference)
    from speech_to_speech_b200.tts_model import B200Qwen3TTS

    class Eng:
        device, codec_eos = 0, -1
        cfg = types.SimpleNamespace(max_positions=4096, max_text=128)

        def __init__(self):
            self.n, self.launches = {}, []

        def max_batch(self):
            return 16

        def prefill(self, slot, ids, spk):
            self.n[slot] = 0

        def frames(self, s):
            return self.n[s]

        def set_frames(self, s, n):
            self.n[s] = n

        def decode_frames(self, slots, n):
            self.launches.append(len(slots))
            time.sleep(0.01)
            for s in slots:
                self.n[s] += n
            return torch.zeros((len(slots), n, 16), dtype=torch.int32)

        def history_context(self, s, valid, left):
            return min(left, self.n[s] - valid)

        def decode_audio_batch(self, slots, valid, left):   # 1920 samples per frame; the value names the slot
            return [torch.full((valid * 1920,), 0.1 * (s + 1)) for s in slots]

        def close(self):
            pass

    eng = Eng()
    model = B200Qwen3TTS(eng, lambda text: [1, 2, 3], {"aiden": 0}, max_sessions=4, batch_wait_s=0.05, batch_gap_s=0.004)
    monkeypatch.setattr(mod.B200Qwen3TTSHandler, "_b200_post",
                        types.SimpleNamespace(from_device=lambda t: (t.numpy()[::3].repeat(2)[: (2 * t.numel() + 2) // 3] * 32767).astype(np.int16)))
    hs = [_make(mod, model, monkeypatch, speaker="Aiden", blocksize=512, max_sessions=4) for _ in range(4)]
    eng.launches.clear()
    outs = {}

    def speak(i):
        hs[i].max_new_tokens = 40                     # 5 chunks of 8 frames
        outs[i] = list(hs[i].process(_tts_input(mod, "Hello there.")))
    ths = [threading.Thread(target=speak, args=(i,)) for i in range(4)]
    [t.start() for t in ths]
    [t.join(60) for t in ths]
    assert sorted(model._free) == [0, 1, 2, 3]                     # every slot came back
    levels = set()
    for i in range(4):
        blocks = outs[i]
        assert blocks and all(b.dtype == np.int16 and b.shape == (512,) for b in blocks)
        vals = {int(v) for v in np.unique(np.concatenate(blocks)) if v != 0}
        assert len(vals) == 1, vals                                # one session's audio only, never another slot's
        levels |= vals
        assert 40 * 1280 // 512 - 2 <= len(blocks) <= 40 * 1280 // 512 + 1
    assert len(levels) == 4
    assert max(eng.launches) >= 2 and len(eng.launches) < 4 * 5   # chunk requests of concurrent sessions shared launches
    model.close()
