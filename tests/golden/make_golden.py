"""Generate golden vectors from `transformers` (the package the reference delegates to).

Run in the builder container (transformers 5.5.0, CPU):
    python tests/golden/make_golden.py [whisper|llama|code2wav|qwen3tts|all]
    PYTHONPATH=<speech-to-speech checkout>/src python tests/golden/make_golden.py tts_handler

The reference holds no golden mel/logits/ids for this path (SURVEY.md section 4), so the
pin is the upstream model code itself: WhisperFeatureExtractor + WhisperForConditionalGeneration
(what S/STT/whisper_stt_handler.py:71-87,243 calls) and LlamaForCausalLM
(S/LLM/language_model.py:811-817) at seeded random-init weights from oracle/weights.py.
Fixtures are subsampled to stay small; the sampling indices are stored with them.
"""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.dirname(os.path.abspath(__file__))

from oracle import weights as W  # noqa: E402

# Decoder prompt / suppress lists used for every random-init Whisper case.  Real checkpoints
# take these from generation_config.json; random-init configs have none (SURVEY.md 8c), so
# we drive generate() with an explicit 4-token prefix and explicit suppress lists.
WHISPER_CASES = {
    "micro": dict(prefix=[4000, 4001, 4002, 4003], eos=4095, suppress=[1, 2, 7, 8, 9, 10, 14, 25, 4000, 4001],
                  begin_suppress=[220, 4095], max_new=24, audio_seed=0, n_samples=160000),
    "tiny": dict(prefix=[50258, 50259, 50359, 50363], eos=50257,
                 suppress=[1, 2, 7, 8, 9, 10, 14, 25, 26, 27, 28, 29, 31, 58, 59, 60, 61, 62, 63, 90, 91, 92, 93,
                           359, 503, 522, 542, 873, 893, 902, 918, 922, 931, 1350, 1853, 1982, 2460, 2627, 3246,
                           3253, 3268, 3536, 3846, 3961, 4183, 4667, 6585, 6647, 7273, 9061, 9383, 10428, 10929,
                           11938, 12033, 12331, 12562, 13793, 14157, 14635, 15265, 15618, 16553, 16604, 18362,
                           18956, 20075, 21675, 22520, 26130, 26161, 26435, 28279, 29464, 31650, 32302, 32470,
                           36865, 42863, 47425, 49870, 50254, 50258, 50358, 50359, 50360, 50361, 50362],
                 begin_suppress=[220, 50257], max_new=32, audio_seed=1, n_samples=160000),
}


def build_hf_whisper(geom: W.WhisperGeometry, weights):
    import torch
    from transformers import WhisperConfig, WhisperForConditionalGeneration

    cfg = WhisperConfig(
        vocab_size=geom.vocab, num_mel_bins=geom.n_mels, d_model=geom.d_model,
        encoder_layers=geom.enc_layers, decoder_layers=geom.dec_layers,
        encoder_attention_heads=geom.heads, decoder_attention_heads=geom.heads,
        encoder_ffn_dim=geom.ffn, decoder_ffn_dim=geom.ffn,
        max_source_positions=geom.max_source_positions, max_target_positions=geom.max_target_positions,
        pad_token_id=0, bos_token_id=0, eos_token_id=0, decoder_start_token_id=0,
        suppress_tokens=None, begin_suppress_tokens=None,
    )
    cfg._attn_implementation = "eager"
    model = WhisperForConditionalGeneration(cfg).eval()
    sd = {k: torch.from_numpy(v.copy()) for k, v in weights.items()}
    sd["proj_out.weight"] = sd["model.decoder.embed_tokens.weight"]
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all("proj_out" in m for m in missing), missing
    return model


def whisper_golden(name: str):
    import torch
    from transformers import WhisperFeatureExtractor

    case = WHISPER_CASES[name]
    geom = W.WHISPER_GEOMETRIES[name]
    weights = W.make_whisper_weights(geom, seed=0)
    model = build_hf_whisper(geom, weights)
    audio = W.synthetic_audio(case["audio_seed"], case["n_samples"])

    fe = WhisperFeatureExtractor(feature_size=geom.n_mels)
    feats = fe(audio, sampling_rate=16000, return_tensors="pt").input_features  # [1, n_mels, 3000]
    with torch.no_grad():
        enc = model.get_encoder()(feats, output_hidden_states=True)
        enc_out = enc.last_hidden_state[0].numpy()
        hs = [h[0].numpy() for h in enc.hidden_states]  # conv+pos, then after each layer
        # teacher-free greedy through the public generate() exactly as the handler calls it
        eos = case["eos"]
        model.generation_config.eos_token_id = eos
        model.generation_config.pad_token_id = eos
        model.generation_config.decoder_start_token_id = case["prefix"][0]
        out = model.generate(
            feats,
            decoder_input_ids=torch.tensor([case["prefix"]]),
            max_new_tokens=case["max_new"], num_beams=1, do_sample=False,
            suppress_tokens=case["suppress"], begin_suppress_tokens=case["begin_suppress"],
            return_timestamps=False, output_scores=True, return_dict_in_generate=True,
        )
        seq = out.sequences[0].tolist()
        scores = torch.stack([s[0] for s in out.scores]).numpy()  # processed logits [steps, V]
    n_pref = len(case["prefix"])
    gen_ids = seq[n_pref:] if seq[:n_pref] == case["prefix"] else seq
    gen_ids = gen_ids[: scores.shape[0]]

    mel = feats[0].numpy()
    frame_idx = np.arange(0, 3000, 7)
    row_idx = np.arange(0, 1500, 25)
    top_idx = np.argsort(-scores, axis=1)[:, :8]
    top_val = np.take_along_axis(scores, top_idx, axis=1)
    col_idx = np.arange(0, geom.vocab, 16)
    np.savez_compressed(
        os.path.join(OUT, f"whisper_{name}.npz"),
        mel_frames=mel[:, frame_idx], frame_idx=frame_idx, mel_max=mel.max(), mel_mean=mel.mean(),
        enc_rows=enc_out[row_idx], row_idx=row_idx,
        conv_rows=hs[0][row_idx], layer0_rows=hs[1][row_idx],
        enc_abs_mean=np.abs(enc_out).mean(),
        gen_ids=np.asarray(gen_ids, np.int32),
        top_idx=top_idx.astype(np.int32), top_val=top_val.astype(np.float32),
        step0_cols=scores[0][col_idx], col_idx=col_idx,
        prefix=np.asarray(case["prefix"], np.int32), eos=eos,
        suppress=np.asarray(case["suppress"], np.int32),
        begin_suppress=np.asarray(case["begin_suppress"], np.int32),
        max_new=case["max_new"], audio_seed=case["audio_seed"], n_samples=case["n_samples"],
    )
    print(f"whisper_{name}: ids={gen_ids[:12]}... n={len(gen_ids)} mel[{mel.min():.3f},{mel.max():.3f}]")


def whisper_langdetect_golden(name: str = "micro"):
    """`WhisperGenerationMixin.detect_language` (TF generation_whisper.py:1610-1674) -- the call the reference's
    `_detect_language` makes (S/STT/whisper_stt_handler.py:166-197) -- on the seeded random-init model, with `lang_to_id` set
    on its generation_config (a random-init config has none).  Pins oracle.whisper_ref.detect_language."""
    import torch
    from transformers import WhisperFeatureExtractor

    geom = W.WHISPER_GEOMETRIES[name]
    weights = W.make_whisper_weights(geom, seed=0)
    model = build_hf_whisper(geom, weights)
    sot = geom.vocab - 96
    codes = ["en", "zh", "de", "es", "fr", "ja", "ko", "ru"]
    lang_to_id = {f"<|{c}|>": sot + 1 + i for i, c in enumerate(codes)}
    model.generation_config.lang_to_id = lang_to_id
    model.generation_config.decoder_start_token_id = sot
    model.config.decoder_start_token_id = sot
    fe = WhisperFeatureExtractor(feature_size=geom.n_mels)
    seeds, lens, got, logits = [0, 21, 22, 23, 24, 25], [160000, 48000, 480000, 16000, 96000, 240000], [], []
    for seed, n in zip(seeds, lens):
        audio = W.synthetic_audio(seed, n)
        feats = fe(audio, sampling_rate=16000, return_tensors="pt").input_features
        with torch.no_grad():
            enc = model.get_encoder()(feats)
            lang = model.detect_language(encoder_outputs=enc, generation_config=model.generation_config)
            dec = model(encoder_outputs=enc, decoder_input_ids=torch.tensor([[sot]])).logits[0, -1].numpy()
        got.append(int(lang[0]))
        logits.append(dec[list(lang_to_id.values())])
    path = os.path.join(OUT, f"whisper_langdetect_{name}.npz")
    np.savez_compressed(path, audio_seeds=np.asarray(seeds), n_samples=np.asarray(lens), sot=sot,
                        lang_ids=np.asarray(list(lang_to_id.values()), np.int32), detected=np.asarray(got, np.int32),
                        lang_logits=np.stack(logits).astype(np.float32))
    print("wrote", path, got)


def build_hf_llama(geom: W.LlamaGeometry, weights):
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM

    if geom.qk_norm:  # Qwen3 family: same decoder with RMSNorm on q / k heads
        from transformers import Qwen3Config, Qwen3ForCausalLM
        cfg = Qwen3Config(
            vocab_size=geom.vocab, hidden_size=geom.d_model, intermediate_size=geom.ffn, num_hidden_layers=geom.layers,
            num_attention_heads=geom.heads, num_key_value_heads=geom.kv_heads, head_dim=geom.head_dim,
            max_position_embeddings=geom.max_positions, rms_norm_eps=geom.rms_eps, rope_theta=geom.rope_theta,
            tie_word_embeddings=False, attention_bias=False, use_sliding_window=False,
        )
        cfg._attn_implementation = "eager"
        model = Qwen3ForCausalLM(cfg).eval()
        model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in weights.items()}, strict=True)
        return model
    cfg = LlamaConfig(
        vocab_size=geom.vocab, hidden_size=geom.d_model, intermediate_size=geom.ffn,
        num_hidden_layers=geom.layers, num_attention_heads=geom.heads, num_key_value_heads=geom.kv_heads,
        head_dim=geom.head_dim, max_position_embeddings=geom.max_positions, rms_norm_eps=geom.rms_eps,
        rope_theta=geom.rope_theta, tie_word_embeddings=False, attention_bias=False, mlp_bias=False,
    )
    cfg._attn_implementation = "eager"
    model = LlamaForCausalLM(cfg).eval()
    sd = {k: torch.from_numpy(v.copy()) for k, v in weights.items()}
    model.load_state_dict(sd, strict=True)
    return model


LLAMA_CASES = {
    "micro": dict(prompt_len=24, max_new=16, seed=3),
    "mini": dict(prompt_len=64, max_new=24, seed=4),
    "qwen3-micro": dict(prompt_len=24, max_new=16, seed=5),
}


def llama_prompt(geom: W.LlamaGeometry, n: int, seed: int) -> np.ndarray:
    return np.random.default_rng(seed).integers(0, geom.vocab, size=n).astype(np.int32)


def llama_golden(name: str):
    import torch

    case = LLAMA_CASES[name]
    geom = W.LLAMA_GEOMETRIES[name]
    weights = W.make_llama_weights(geom, seed=0)
    model = build_hf_llama(geom, weights)
    prompt = llama_prompt(geom, case["prompt_len"], case["seed"])
    ids = torch.from_numpy(prompt.astype(np.int64))[None]
    with torch.no_grad():
        full = model(ids, output_hidden_states=True)
        prefill_logits = full.logits[0].numpy()  # [P, V]
        h_last = full.hidden_states[-1][0].numpy()
        h1 = full.hidden_states[1][0].numpy()
        out = model.generate(
            ids, max_new_tokens=case["max_new"], min_new_tokens=case["max_new"], do_sample=False,
            output_scores=True, return_dict_in_generate=True, pad_token_id=0,
        )
        gen = out.sequences[0, ids.shape[1]:].numpy().astype(np.int32)
        scores = torch.stack([s[0] for s in out.scores]).numpy()
    top_idx = np.argsort(-scores, axis=1)[:, :8]
    top_val = np.take_along_axis(scores, top_idx, axis=1)
    col_idx = np.arange(0, geom.vocab, 8)
    np.savez_compressed(
        os.path.join(OUT, f"llama_{name}.npz"),
        prompt=prompt, gen_ids=gen, top_idx=top_idx.astype(np.int32), top_val=top_val.astype(np.float32),
        prefill_last_cols=prefill_logits[-1][col_idx], prefill_mid_cols=prefill_logits[len(prompt) // 2][col_idx],
        col_idx=col_idx, h1_last=h1[-1], hN_last=h_last[-1], max_new=case["max_new"],
    )
    print(f"llama_{name}: gen={gen[:10]}...")


def code2wav_golden(name: str = "micro"):
    """Qwen3OmniMoeCode2Wav (the published cousin of the Qwen3-TTS 12 Hz codec decoder; oracle/code2wav_ref.py) at seeded
    weights: codes [Q, T] -> waveform, plus the pre-transformer output."""
    import torch
    from transformers.models.qwen3_omni_moe.configuration_qwen3_omni_moe import Qwen3OmniMoeCode2WavConfig
    from transformers.models.qwen3_omni_moe.modeling_qwen3_omni_moe import Qwen3OmniMoeCode2Wav
    from oracle import code2wav_ref as C

    g = C.GEOMETRIES[name]
    w = C.make_weights(g, 0)
    cfg = Qwen3OmniMoeCode2WavConfig(codebook_size=g.codebook_size, hidden_size=g.hidden, num_attention_heads=g.heads,
                                     num_key_value_heads=g.kv_heads, intermediate_size=g.inter, num_hidden_layers=g.layers,
                                     num_quantizers=g.quantizers, upsample_rates=g.upsample_rates,
                                     upsampling_ratios=g.upsampling_ratios, decoder_dim=g.decoder_dim,
                                     sliding_window=g.sliding_window, max_position_embeddings=g.max_positions, rms_norm_eps=g.rms_eps)
    m = Qwen3OmniMoeCode2Wav(cfg).eval()
    assert set(m.state_dict().keys()) == set(w.keys())
    m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    codes = np.random.default_rng(1).integers(0, g.codebook_size, (g.quantizers, 20)).astype(np.int64)
    with torch.no_grad():
        t = torch.from_numpy(codes)[None]
        hidden = m.pre_transformer(inputs_embeds=m.code_embedding(t + m.code_offset).mean(1)).last_hidden_state[0].numpy()
        wav = m(t)[0, 0].numpy()
        chunked = m.chunked_decode(t, chunk_size=8, left_context_size=6)[0, 0].numpy()
    path = os.path.join(OUT, f"code2wav_{name}.npz")
    np.savez_compressed(path, codes=codes, hidden=hidden.astype(np.float32), wav=wav.astype(np.float32),
                        chunked=chunked.astype(np.float32), chunk_size=8, left_context=6, transformers_version=__import__("transformers").__version__)
    print("wrote", path, wav.shape, float(np.abs(wav).max()))


def sample_logits(logits: np.ndarray, keep: float = 0.5, top: int = 8, seed: int = 5) -> np.ndarray:
    """Keep the file under 1 MB: every row keeps its `top` largest logits (the top-1 / top-2 margins stay exact) and a seeded
    `keep` share of the other entries; the rest become NaN."""
    kept = np.random.default_rng(seed).random(logits.shape) < keep
    np.put_along_axis(kept, np.argsort(logits, axis=-1)[..., -top:], True, axis=-1)
    return np.where(kept, logits, np.float32(np.nan)).astype(np.float32)


def qwen3tts_golden(name: str = "micro", text_len: int = 6, max_frames: int = 10):
    """Talker + code predictor of the published cousin (`Qwen3OmniMoeTalkerForConditionalGeneration`, transformers) at
    seeded weights, driven exactly like `Qwen3OmniMoeForConditionalGeneration.generate` step 2 drives it, with the two
    substitutions oracle/qwen3tts_ref.py states: the talker's MoE block is replaced by the dense
    `Qwen3OmniMoeTalkerTextMLP` (the real Qwen3-TTS talker is dense), and both `generate` calls run greedily
    (do_sample=False, no repetition penalty).  Records the codes of every frame and the talker / predictor logits."""
    import torch
    from transformers.models.qwen3_omni_moe.configuration_qwen3_omni_moe import Qwen3OmniMoeTalkerConfig
    from transformers.models.qwen3_omni_moe import modeling_qwen3_omni_moe as M
    from oracle import qwen3tts_ref as R

    g = R.GEOMETRIES[name]
    w = R.make_weights(g, 0)
    t, c = g.talker, g.predictor
    rope = {"rope_type": "default", "rope_theta": t.rope_theta}
    tc = dict(vocab_size=t.vocab, hidden_size=t.d_model, intermediate_size=t.ffn, num_hidden_layers=t.layers,
              num_attention_heads=t.heads, num_key_value_heads=t.kv_heads, head_dim=t.head_dim, rms_norm_eps=t.rms_eps,
              num_experts=2, num_experts_per_tok=1, moe_intermediate_size=64, shared_expert_intermediate_size=64,
              rope_parameters=dict(rope, mrope_section=[t.head_dim // 8, t.head_dim // 8 + t.head_dim // 16, t.head_dim // 4 - t.head_dim // 8 - t.head_dim // 16 + t.head_dim // 8],
                                   mrope_interleaved=True))
    # three sections that add up to head_dim / 2 (the split is irrelevant here: all three carry the same text position)
    sec = tc["rope_parameters"]["mrope_section"]
    sec[2] = t.head_dim // 2 - sec[0] - sec[1]
    cp = dict(vocab_size=c.vocab, hidden_size=c.d_model, intermediate_size=c.ffn, num_hidden_layers=c.layers,
              num_attention_heads=c.heads, num_key_value_heads=c.kv_heads, head_dim=c.head_dim, rms_norm_eps=c.rms_eps,
              num_code_groups=g.n_groups, rope_parameters={"rope_type": "default", "rope_theta": c.rope_theta})
    speaker = 2301
    cfg = Qwen3OmniMoeTalkerConfig(text_config=tc, code_predictor_config=cp, num_code_groups=g.n_groups,
                                   thinker_hidden_size=g.text_hidden, codec_eos_token_id=g.codec_eos,
                                   codec_nothink_id=g.codec_nothink, codec_think_bos_id=g.codec_think_bos,
                                   codec_think_eos_id=g.codec_think_eos, codec_pad_id=g.codec_pad, codec_bos_id=g.codec_bos,
                                   speaker_id={"aiden": speaker}, spatial_merge_size=2)
    m = M.Qwen3OmniMoeTalkerForConditionalGeneration(cfg).eval()
    for layer in m.model.layers:   # substitution 1: dense MLP
        layer.mlp = M.Qwen3OmniMoeTalkerTextMLP(cfg.text_config, intermediate_size=t.ffn)
    sd = m.state_dict()
    own = {}
    for k in sd:
        if k.startswith("hidden_projection."):
            own[k] = sd[k]          # multimodal path of the cousin: unused by a text-only TTS turn
        else:
            assert k in w, k
            own[k] = torch.from_numpy(w[k])
    assert set(w) - set(sd) == {"text_embedding.weight"}, set(w) - set(sd)
    m.load_state_dict(own)
    emb = torch.from_numpy(w["text_embedding.weight"])
    text_ids = np.random.default_rng(11).integers(0, g.tts_bos - 8, text_len).tolist()
    ids = torch.tensor([[g.im_start, g.assistant, g.newline] + text_ids])

    # ---- Qwen3OmniMoeForConditionalGeneration.generate, "2. Prepare talker input" (TF:4019-4075), text-only turn
    class Host:   # the attributes _get_talker_assistant_parts reads from the top-level model
        pass
    host = Host()
    host.talker = m
    host.config = type("C", (), {"talker_config": cfg, "tts_pad_token_id": g.tts_pad})()
    with torch.no_grad():
        special = torch.tensor([[g.tts_bos, g.tts_eos, g.tts_pad]])
        bos_e, eos_e, pad_e = m.text_projection(emb[special]).chunk(3, dim=1)
        embeds, in_ids, trailing = M.Qwen3OmniMoeForConditionalGeneration._get_talker_assistant_parts(
            host, 0, ids.shape[1], speaker, emb[ids], pad_e, bos_e, eos_e)
        orig = m.code_predictor.generate

        pred_scores = []

        def greedy_predictor(**kw):   # substitution 2: greedy code predictor
            kw.update(do_sample=False, top_k=None, top_p=None, output_scores=True)
            out = orig(**kw)
            pred_scores.append(torch.stack([s[0] for s in out.scores]).numpy())
            return out
        m.code_predictor.generate = greedy_predictor
        suppress = [i for i in range(t.vocab - 1024, t.vocab) if i != g.codec_eos]
        res = m.generate(inputs_embeds=embeds, trailing_text_hidden=trailing, tts_pad_embed=pad_e, talker_input_ids=in_ids,
                         max_new_tokens=max_frames, do_sample=False, eos_token_id=g.codec_eos, suppress_tokens=suppress,
                         output_hidden_states=True, return_dict_in_generate=True, output_scores=True, pad_token_id=g.codec_pad,
                         attention_mask=torch.ones_like(in_ids))
        codes = torch.stack([h[-1] for h in res.hidden_states if h[-1] is not None], dim=1)[0].numpy()   # [F, 16]
        t_scores = torch.stack([s[0] for s in res.scores]).numpy()
    path = os.path.join(OUT, f"qwen3tts_{name}.npz")
    np.savez_compressed(path, text_ids=np.asarray(text_ids, np.int32), speaker=speaker, codes=codes.astype(np.int32),
                        code0_all=res.sequences[0].numpy().astype(np.int32), talker_logits=t_scores.astype(np.float32),
                        predictor_logits=sample_logits(np.stack(pred_scores).astype(np.float32)),
                        prompt_embeds=embeds[0].numpy().astype(np.float32),
                        trailing=trailing[0].numpy().astype(np.float32), max_frames=max_frames,
                        transformers_version=__import__("transformers").__version__)
    print("wrote", path, codes.shape, codes[:2].tolist(), "code0", res.sequences[0].tolist())


TTS_HANDLER_SIZES = (1, 480, 1920, 15360, 48001)
BUDGET_ALPHABET = list("abcdefghij klmnop, qrst. uvw! xyz? 上海是一座城市，。") + [" "] * 6
BUDGET_CASES = ((8, 1536), (4, 700), (1, 5000))


def tts_handler_golden():
    """What the upstream Qwen3TTSHandler (huggingface/speech-to-speech, TTS/qwen3_tts_handler.py) returns from
    `_resample_to_pipeline_sr` / `_to_int16` on seeded audio and from `_estimate_max_new_tokens` on seeded random text.
    Needs the upstream sources importable, e.g. PYTHONPATH=<speech-to-speech checkout>/src (not part of `all`)."""
    from speech_to_speech.TTS.qwen3_tts_handler import Qwen3TTSHandler

    h = object.__new__(Qwen3TTSHandler)
    out = {}
    rng = np.random.default_rng(7)       # the inputs are regenerated from these seeds by tests/test_oracle_tts.py
    for n in TTS_HANDLER_SIZES:
        x = (0.4 * rng.standard_normal(n)).astype(np.float32)
        y = h._resample_to_pipeline_sr(x, 24000)
        out[f"resampled_{n}"], out[f"int16_{n}"] = y, h._to_int16(y)
    x = (0.2 * np.random.default_rng(0).standard_normal(4410)).astype(np.float32)
    y = h._resample_to_pipeline_sr(x, 44100)
    out["resampled_44100"], out["int16_44100"] = y, h._to_int16(y)
    rng = np.random.default_rng(0)       # the texts too (tests/test_tts_handler.py); their CRC-32s are stored to check that
    crcs, budgets = [], []
    for chunk, cap in BUDGET_CASES:
        h.streaming_chunk_size, h.max_new_tokens = chunk, cap
        for _ in range(200):
            text = "".join(rng.choice(BUDGET_ALPHABET, int(rng.integers(0, 900))))
            crcs.append(zlib.crc32(text.encode()))
            budgets.append(h._estimate_max_new_tokens(text))
    path = os.path.join(OUT, "tts_handler_reference.npz")
    np.savez_compressed(path, budget_cases=np.asarray(BUDGET_CASES, np.int32),
                        budget_text_crc32=np.asarray(crcs, np.uint32).reshape(len(BUDGET_CASES), -1),
                        budgets=np.asarray(budgets, np.int32).reshape(len(BUDGET_CASES), -1), **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what == "tts_handler":
        tts_handler_golden()
    if what in ("whisper", "all"):
        for n in WHISPER_CASES:
            whisper_golden(n)
    if what in ("langdetect", "all"):
        whisper_langdetect_golden("micro")
    if what in ("llama", "all"):
        for n in LLAMA_CASES:
            llama_golden(n)
    if what in ("code2wav", "all"):
        code2wav_golden("micro")
    if what in ("qwen3tts", "all"):
        qwen3tts_golden("micro")
