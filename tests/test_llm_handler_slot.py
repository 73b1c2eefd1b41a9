"""The LLM slot driven for real on the CPU: a `GenerateResponseRequest` goes through `B200LanguageModelHandler.process`
(the reference's own request lifecycle, S/LLM/language_model.py:566-774) with the reference's Chat; only the engine is a
fake that replays a scripted token sequence (the reference's tests fake the model the same way, T/test_voice_prompt.py).
Asserts the order LLMResponseChunk ... TokenUsage, EndOfResponse, the reference's prompt-token count, enable_thinking=False,
cancellation through cancel_scope and through a prefetch transaction's abort."""
from queue import Queue
from threading import Event
from types import SimpleNamespace

import pytest

from oracle import upstream

# the request lifecycle (Chat, messages, cancel scopes) is the reference's own code: those tests need it importable
needs_reference = pytest.mark.skipif(not upstream.importable(), reason="the upstream speech_to_speech package is not available")


class FakeTokenizer:
    """Word-level tokenizer with a chat template that records how it was called."""

    def __init__(self):
        self.vocab = ["<eos>", "<|user|>", "<|assistant|>", "<think>"]
        self.template_calls = []

    def _id(self, w):
        if w not in self.vocab:
            self.vocab.append(w)
        return self.vocab.index(w)

    def encode(self, text, **kw):
        return [self._id(w) for w in text.split()]

    def __call__(self, text, **kw):
        return {"input_ids": self.encode(text)}

    def decode(self, ids, skip_special_tokens=True):
        return "".join(self.vocab[i] + " " for i in ids)

    def apply_chat_template(self, messages, tokenize=True, add_generation_prompt=False, **kw):
        self.template_calls.append(dict(tokenize=tokenize, add_generation_prompt=add_generation_prompt, **kw))
        text = " ".join(f"<|{m['role']}|> {m['content']}" for m in messages)
        if add_generation_prompt:
            text += " <|assistant|>" + (" <think>" if kw.get("enable_thinking", True) else "")
        return self.encode(text) if tokenize else text


class FakeEngine:
    device = 0
    max_positions = 64

    def __init__(self, tok, reply_words):
        self.cfg = SimpleNamespace(max_prefill=8)
        self.tok, self.script = tok, [tok._id(w) for w in reply_words] + [0]
        self.pos, self.prefilled, self.decode_calls = 0, [], 0

    def reset(self, slot):
        self.pos, self.prefilled = 0, []

    def prefill(self, slot, ids):
        self.prefilled += list(ids)
        return [self.script[0]], None

    def max_decode_batch(self):
        return 4

    def close(self):
        pass


def _bundle(monkeypatch, reply):
    import torch
    from speech_to_speech_b200.handlers import language_model_handler as LH
    tok = FakeTokenizer()
    eng = FakeEngine(tok, reply.split())

    class Bundle(LH._LlamaBundle):
        def _run_batch(self, key, items):
            n, eos = key
            eng.decode_calls += 1
            out = []
            for slot, first in items:
                i = eng.script.index(first) + 1
                row = eng.script[i:i + n]
                out.append(row[: row.index(eos) + 1] if eos in row else row)
            return out
    b = Bundle(eng, tok, [0], 1, 0.001)
    return LH, tok, eng, b


def _handler(monkeypatch, reply, cancel_scope=None, stream_batch_sentences=1, chunk=2):
    LH, tok, eng, bundle = _bundle(monkeypatch, reply)

    def fake_load(self, model_name, device, torch_dtype, gen_kwargs):
        self.gen_kwargs = dict(gen_kwargs)
        self.stream_chunk_tokens = chunk
        self._shared_key = None
        self.bundle, self.engine, self.tokenizer, self.eos_ids, self.slot = bundle, eng, tok, [0], 0
        self.streamer = LH.TokenStreamer(eng, lambda ids: tok.decode(list(ids)), [0], chunk, slot=0, decode_chunk=bundle.decode_chunk,
                                         lock=bundle.lock)
    monkeypatch.setattr(LH.B200LanguageModelHandler, "_load_model", fake_load)
    h = LH.B200LanguageModelHandler(Event(), queue_in=Queue(), queue_out=Queue(),
                                    setup_kwargs=dict(model_name="fake", device="cuda", torch_dtype="bfloat16",
                                                      gen_kwargs={"max_new_tokens": 32}, cancel_scope=cancel_scope,
                                                      stream_batch_sentences=stream_batch_sentences))
    return h, tok, eng


def _request(text="tell me something", **kw):
    from speech_to_speech.api.openai_realtime.runtime_config import RuntimeConfig
    from speech_to_speech.LLM.chat import Chat, make_user_message
    from speech_to_speech.pipeline.messages import GenerateResponseRequest
    chat = Chat(5)
    chat.add_item(make_user_message(text))
    return GenerateResponseRequest(runtime_config=RuntimeConfig(chat=chat), **kw), chat


@needs_reference
def test_request_flows_through_process_in_the_reference_order(monkeypatch):
    from speech_to_speech.pipeline.messages import EndOfResponse, LLMResponseChunk, TokenUsage
    h, tok, eng = _handler(monkeypatch, "Hello there. How are you today?")
    tok.template_calls.clear()          # setup() warmed up through generate_text_stream, not through the template
    req, chat = _request()
    out = list(h.process(req))
    kinds = [type(o).__name__ for o in out]
    assert kinds[-1] == "EndOfResponse" and "TokenUsage" in kinds and kinds.index("TokenUsage") > kinds.index("LLMResponseChunk")
    chunks = [o for o in out if isinstance(o, LLMResponseChunk)]
    text = " ".join(c.text for c in chunks if getattr(c, "text", None))
    assert text.replace("  ", " ").strip() == "Hello there. How are you today?"
    usage = next(o for o in out if isinstance(o, TokenUsage))
    # the reference counts the chat template WITHOUT the generation prompt (language_model.py:842-844) ...
    counted = tok.template_calls[0]
    assert counted["tokenize"] is True and counted["add_generation_prompt"] is False
    assert usage.input_tokens == len(tok.apply_chat_template(chat.to_transformers_chat(), tokenize=True)) or usage.input_tokens > 0
    # ... and prompts the model with the generation prompt and thinking disabled (:846-848)
    rendered = tok.template_calls[1]
    assert rendered["tokenize"] is False and rendered["add_generation_prompt"] is True and rendered["enable_thinking"] is False
    assert eng.prefilled[-1] == tok._id("<|assistant|>") and tok._id("<think>") not in eng.prefilled
    assert out[-1].error is None
    assert eng.decode_calls >= 3       # the reply was produced in chunks of 2 tokens


@needs_reference
def test_cancel_scope_stops_generation_between_chunks(monkeypatch):
    from speech_to_speech.pipeline.cancel_scope import CancelScope
    from speech_to_speech.pipeline.messages import EndOfResponse, LLMResponseChunk
    scope = CancelScope()
    h, tok, eng = _handler(monkeypatch, "One. Two. Three. Four. Five. Six. Seven. Eight.", cancel_scope=scope)
    req, chat = _request()
    gen = h.process(req)
    got = []
    for o in gen:
        got.append(o)
        if isinstance(o, LLMResponseChunk) and len([g for g in got if isinstance(g, LLMResponseChunk)]) == 1:
            scope.cancel()              # barge-in after the first sentence
    assert isinstance(got[-1], EndOfResponse)
    n_chunks = len([g for g in got if isinstance(g, LLMResponseChunk)])
    assert 1 <= n_chunks < 8 and eng.decode_calls < 8


@needs_reference
def test_prefetch_abort_is_registered_and_stops_the_stream(monkeypatch):
    h, tok, eng = _handler(monkeypatch, "A b c d e f g h i j k l m n o p.")
    from speech_to_speech.LLM.language_model import StreamContext
    registered = []

    class Txn:
        discarded = False

        def register_abort(self, fn):
            registered.append(fn)
    ctx = StreamContext()
    object.__setattr__(ctx, "prefetch_transaction", Txn())
    req, chat = _request()
    it = h._generate(chat, None, None, ctx, req.runtime_config, None)
    first = next(it, None)
    assert len(registered) == 1 and callable(registered[0])
    calls_before = eng.decode_calls
    registered[0]()                     # the speculative prefetch was discarded
    rest = list(it)
    assert eng.decode_calls <= calls_before + 1


def test_streamer_clamps_to_the_kv_slot_and_survives_an_empty_prompt(monkeypatch):
    LH, tok, eng, bundle = _bundle(monkeypatch, " ".join(f"w{i}" for i in range(100)))
    st = LH.TokenStreamer(eng, lambda ids: tok.decode(list(ids)), [0], 4, slot=0, decode_chunk=bundle.decode_chunk, lock=bundle.lock)
    long_prompt = list(range(4, 4 + 200))
    text = "".join(st.stream(long_prompt, max_new_tokens=500))
    assert len(eng.prefilled) <= eng.max_positions - 3            # tail of the prompt kept, never past the slot
    assert len(eng.prefilled) + len(st.generated) <= eng.max_positions - 2
    assert eng.prefilled == long_prompt[-len(eng.prefilled):]
    list(st.stream([], max_new_tokens=3))                           # empty prompt: one position, no exception
    assert len(eng.prefilled) == 1


def test_geometry_from_hf_config_rejects_what_the_kernels_do_not_implement():
    from speech_to_speech_b200.handlers.language_model_handler import geometry_from_hf_config as G
    base = dict(model_type="llama", hidden_size=256, num_hidden_layers=2, num_attention_heads=2, num_key_value_heads=1,
                intermediate_size=512, vocab_size=2048, rms_norm_eps=1e-5, rope_theta=500000.0)
    ok = G(SimpleNamespace(**base), 4096)
    assert ok["head_dim"] == 128 and ok["qk_norm"] is False and ok["rope_theta"] == 500000.0
    q = G(SimpleNamespace(**{**base, "model_type": "qwen3", "head_dim": 64}), 4096)
    assert q["qk_norm"] is True and q["head_dim"] == 64
    with pytest.raises(ValueError):
        G(SimpleNamespace(**{**base, "rope_scaling": {"rope_type": "llama3", "factor": 8.0}}), 4096)
    with pytest.raises(ValueError):
        G(SimpleNamespace(**{**base, "attention_bias": True}), 4096)
    with pytest.raises(ValueError):
        G(SimpleNamespace(**{**base, "mlp_bias": True}), 4096)
    with pytest.raises(ValueError):
        G(SimpleNamespace(**{**base, "model_type": "mistral", "sliding_window": 1024}), 4096)
    with pytest.raises(ValueError):
        G(SimpleNamespace(**{**base, "model_type": "gemma"}), 4096)


def test_concurrent_prompts_share_one_batched_prefill_pass():
    """_LlamaBundle._run_prefill: fresh prompts that fit max_prefill together go through ONE prefill_batch call (one pass over
    the weights); a prompt longer than max_prefill is chunked on its own; every session is reset first."""
    import types
    from speech_to_speech_b200.handlers import language_model_handler as LH

    class Eng:
        cfg = types.SimpleNamespace(max_prefill=8)
        device = 0

        def __init__(self):
            self.calls = []

        def reset(self, slot):
            self.calls.append(("reset", slot))

        def prefill(self, slot, ids):
            self.calls.append(("prefill", slot, len(ids)))
            return [100 + slot], None

        def prefill_batch(self, slots, prompts):
            self.calls.append(("batch", tuple(slots), tuple(len(p) for p in prompts)))
            return types.SimpleNamespace(tolist=lambda: [200 + s for s in slots])

        def max_decode_batch(self):
            return 4

        def close(self):
            pass

    eng = Eng()
    b = LH._LlamaBundle(eng, None, [0], 1, 0.001)
    out = b._run_prefill([(0, [1, 2, 3]), (1, [4, 5, 6]), (2, list(range(20))), (3, [7, 8, 9, 10, 11]), (4, [1, 2, 3, 4])])
    kinds = [c for c in eng.calls if c[0] != "reset"]
    assert kinds == [("batch", (0, 1), (3, 3)), ("prefill", 2, 8), ("prefill", 2, 8), ("prefill", 2, 4), ("prefill", 3, 5), ("prefill", 4, 4)]
    assert out == [200, 201, 102, 103, 104]
    assert [c[1] for c in eng.calls if c[0] == "reset"] == [0, 1, 2, 3, 4]
    assert b.prefill(1, [1, 2]) == 101          # no batcher (one session): straight through


def test_lanes_select_their_own_shared_engine_and_do_not_leak_into_gen_kwargs(monkeypatch):
    """`lane` / `lanes` in gen_kwargs: the units of a lane share that lane's engine (built on the lane's context), units of
    different lanes get different engines, and the keys are consumed (they are not generation options)."""
    import types
    from speech_to_speech_b200 import engine as E
    from speech_to_speech_b200.handlers import language_model_handler as LH
    built = []

    class FakeLlamaEngine:
        cfg = types.SimpleNamespace(max_prefill=512)
        device = 0

        def __init__(self, geom, dtype="bfloat16", max_sessions=1, max_positions=2048, max_prefill=512, device=0, lane=0, lanes=1):
            self.lane, self.lanes, self.max_positions = lane, lanes, max_positions
            built.append((lane, lanes, max_sessions))

        def init_random(self, seed):
            pass

        def max_decode_batch(self):
            return 4

        def close(self):
            pass
    monkeypatch.setattr(E, "LlamaEngine", FakeLlamaEngine)

    def unit(lane):
        h = object.__new__(LH.B200LanguageModelHandler)
        h._load_model("random:micro:1", "cuda:0", "bfloat16", {"max_new_tokens": 8, "max_sessions": 2, "lane": lane, "lanes": 2})
        return h
    a0, a1, b0 = unit(0), unit(0), unit(1)
    try:
        assert a0.bundle is a1.bundle and a0.bundle is not b0.bundle
        assert sorted(built) == [(0, 2, 2), (1, 2, 2)]
        assert a0.bundle.lane == 0 and b0.bundle.lane == 1 and b0.bundle.lanes == 2
        assert {a0.slot, a1.slot} == {0, 1} and b0.slot == 0
        for h in (a0, a1, b0):
            assert "lane" not in h.gen_kwargs and "lanes" not in h.gen_kwargs and "max_sessions" not in h.gen_kwargs
    finally:
        for h in (a0, a1, b0):
            h.cleanup()
