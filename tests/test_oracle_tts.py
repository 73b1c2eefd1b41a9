"""CPU: the TTS post-processing oracle (oracle/tts_post_ref.py) against scipy and against what the reference handler's own
helper methods (`Qwen3TTSHandler._resample_to_pipeline_sr`, `_to_int16`, TTS/qwen3_tts_handler.py:612-613, 674-680)
returned, stored in tests/golden/tts_handler_reference.npz.  Bit-exact: the CUDA kernel is then held to the same vectors
on the GPU."""
import os

import numpy as np
import pytest

from oracle import tts_post_ref as T


@pytest.mark.parametrize("n", [1, 2, 3, 7, 61, 100, 333, 1919, 1920])
def test_direct_restatement_is_bit_identical_to_scipy(n):
    x = (0.3 * np.random.default_rng(n).standard_normal(n)).astype(np.float32)
    ref = T.resample_to_16k(x, 24000)
    got = T.resample_direct(x)
    assert got.dtype == np.float32 and got.shape == ref.shape
    assert np.array_equal(got, ref.astype(np.float32))


def test_int16_conversion_clips_and_truncates_like_numpy():
    x = np.array([0.0, 0.5, -0.5, 0.99999, 1.0, 1.5, -1.0, -1.5, 1e-6, -1e-6], np.float32)
    assert T.to_int16(x).tolist() == [0, 16384, -16384, 32767, 32767, 32767, -32768, -32768, 0, 0]


def test_stream_blocks_trims_leading_silence_and_pads_the_tail():
    sil = np.zeros(2400, np.float32)
    tone = (0.2 * np.sin(2 * np.pi * 440 * np.arange(4800) / 24000)).astype(np.float32)
    blocks = T.stream_blocks([sil, sil, tone, tone], blocksize=512)
    assert all(b.dtype == np.int16 and b.shape == (512,) for b in blocks)
    flat = np.concatenate(blocks)
    # 2 x 4800 samples @24k -> 6400 @16k; the two silent chunks are dropped entirely; zero-padded to a block multiple
    assert len(flat) == 13 * 512 and np.abs(flat[:6400]).max() > 3000 and not flat[6400:].any()


@pytest.fixture(scope="module")
def upstream(golden_dir):
    """What the upstream handler's own helpers returned (tests/golden/make_golden.py tts_handler)."""
    return np.load(os.path.join(golden_dir, "tts_handler_reference.npz"))


def _handler_base():
    """The class the TTS handler slot builds on: the upstream Qwen3TTSHandler when installed, the mirror otherwise."""
    from speech_to_speech_b200.handlers.qwen3_tts_handler import _base_class
    return _base_class()


def test_oracle_equals_the_reference_handler_helpers(upstream):
    base = _handler_base()
    h = object.__new__(base)
    rng = np.random.default_rng(7)
    for n in (1, 480, 1920, 15360, 48001):
        x = (0.4 * rng.standard_normal(n)).astype(np.float32)
        ref16k, ref_int16 = upstream[f"resampled_{n}"], upstream[f"int16_{n}"]
        assert np.array_equal(T.resample_to_16k(x, 24000), ref16k)
        assert np.array_equal(T.to_int16(ref16k), ref_int16)
        assert np.array_equal(T.postproc(x), ref_int16)
        assert np.array_equal(base._resample_to_pipeline_sr(h, x, 24000), ref16k)
        assert np.array_equal(base._to_int16(h, ref16k), ref_int16)
    same = rng.standard_normal(100).astype(np.float32)
    assert base._resample_to_pipeline_sr(h, same, 16000) is same  # pipeline rate passes through untouched


def test_patched_tts_handler_keeps_the_reference_pinned_token_budgets(upstream):
    """The only golden values the reference's tests hold on this path are `_estimate_max_new_tokens` = 360 / 576 / cap
    (tests/test_qwen3_tts_handler_backend.py:915-964).  The handler class with the GPU post-processing patched in must
    still produce them (the estimator stays the base class's own Python) and must leave non-24 kHz audio on the scipy path."""
    from speech_to_speech_b200.handlers.qwen3_tts_postproc import patch_handler_class

    base = _handler_base()
    cls = patch_handler_class(base)
    assert issubclass(cls, base)
    h = object.__new__(cls)
    h.streaming_chunk_size, h.max_new_tokens = 8, 1536
    long_text = " ".join(["This is a deliberately long sentence for the Qwen3 TTS budget estimator."] * 12)
    assert h._estimate_max_new_tokens("Hello there.") == 360
    assert h._estimate_max_new_tokens("我懂，心情不好时会让人特别疲惫。") == 360
    cjk_long = ("上海是一座充满活力的现代化大都市，既有繁华的金融中心和摩天大楼，也有老城厢的弄堂风情"
                "和江南水乡的韵味。这里交通便利，餐饮选择丰富，从精致西餐到地道小馆应有尽有。同时，上海"
                "还是文化与创新的交汇点，艺术展览、科技展会和国际活动频繁。如果你喜欢快节奏的生活和多元"
                "的氛围，上海会是个很吸引人的地方。你想了解哪方面的具体信息呢？")
    assert h._estimate_max_new_tokens(cjk_long) == 576
    budget = h._estimate_max_new_tokens(long_text)
    assert budget > 360 and budget % 8 == 0 and budget <= 1536
    h.max_new_tokens = 400
    assert h._estimate_max_new_tokens(long_text) == 400
    # audio that is not 24 kHz never touches the GPU path: identical to the reference's scipy result
    x = (0.2 * np.random.default_rng(0).standard_normal(4410)).astype(np.float32)
    assert np.array_equal(h._resample_to_pipeline_sr(x, 44100), upstream["resampled_44100"])
    assert np.array_equal(h._to_int16(upstream["resampled_44100"]), upstream["int16_44100"])
