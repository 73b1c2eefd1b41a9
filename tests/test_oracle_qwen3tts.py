"""The numpy talker / code-predictor oracle (oracle/qwen3tts_ref.py) against the golden vectors generated from the
transformers cousin (tests/golden/make_golden.py qwen3tts): codes bit-exact, logits within 2e-4.
Parity with the real Qwen3-TTS (faster-qwen3-tts, absent) stays unpinned."""
import os

import numpy as np
import pytest

from oracle import qwen3tts_ref as R


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "qwen3tts_micro.npz"))


@pytest.fixture(scope="module")
def model():
    g = R.GEOMETRIES["micro"]
    return g, R.make_weights(g, 0)


def test_prompt_layout_matches_the_cousin(gold, model):
    g, w = model
    embeds, trailing, pad = R.build_prompt(w, g, gold["text_ids"].tolist(), int(gold["speaker"]))
    assert embeds.shape == gold["prompt_embeds"].shape == (9, g.talker.d_model)
    np.testing.assert_allclose(embeds, gold["prompt_embeds"], atol=2e-5)
    np.testing.assert_allclose(trailing, gold["trailing"], atol=2e-5)


def test_codes_bit_exact_and_logits_close(gold, model):
    g, w = model
    F = int(gold["max_frames"])
    codes, t_logits, p_logits = R.generate(w, g, gold["text_ids"].tolist(), int(gold["speaker"]), F, return_logits=True)
    ref = gold["codes"]
    # the cousin returns the residual codes of every frame but the last generated one (they are computed when the NEXT
    # talker step is prepared): F - 1 full frames, F first codes
    assert ref.shape == (F - 1, g.n_groups)
    assert np.array_equal(codes[: F - 1], ref)
    assert codes[:, 0].tolist() == gold["code0_all"].tolist()
    fin = np.isfinite(gold["talker_logits"])
    assert np.array_equal(fin, np.isfinite(t_logits))           # the same ids are suppressed
    assert np.abs(t_logits[fin] - gold["talker_logits"][fin]).max() < 2e-4
    # the golden keeps each row's top logits and a seeded half of the rest (NaN elsewhere, make_golden.sample_logits)
    kept = ~np.isnan(gold["predictor_logits"])
    assert kept.mean() > 0.5 and np.isfinite(p_logits[: F - 1]).all()
    assert np.abs(p_logits[: F - 1][kept] - gold["predictor_logits"][kept]).max() < 2e-4


def test_suppress_list_is_the_cousins(model):
    g, _ = model
    s = R.suppress_ids(g)
    assert len(s) == 1023 and g.codec_eos not in s and min(s) == g.talker.vocab - 1024


def test_eos_stops_generation(model):
    g, w = model
    w2 = dict(w)
    head = w["codec_head.weight"].copy()
    head[g.codec_eos] = 50.0 * np.sign(head.sum() + 1.0)  # make eos dominate whenever the hidden state has a positive sum
    w2["codec_head.weight"] = head
    codes = R.generate(w2, g, [5, 6, 7], 2301, 6)
    assert codes.shape[0] <= 6 and codes.shape[1] == g.n_groups
