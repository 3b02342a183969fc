"""Host-side logic on CPU (no GPU): hook lifecycle, n_kept arithmetic, pipeline plumbing, DecodingPress
scheduling — the reference's own tests (tests/test_press_call.py, tests/presses/test_presses.py:143-162,
tests/test_pipeline.py, tests/test_decoding_compression.py) re-hosted on random-init models.
The CUDA library is replaced by the oracle-backed stand-in of tests/cpu_backend.py (monkeypatch)."""
import logging

import pytest
import torch
from transformers import DynamicCache

import kvpress_b200
from kvpress_b200 import (DecodingPress, ExpectedAttentionPress, KnormPress, KVPressTextGenerationPipeline,
                          ScorerPress, SnapKVPress, StreamingLLMPress, native)
from kvpress_b200.presses.decoding_press import find_target_compression_ratio
from kvpress_b200.presses.scorer_press import kept_count
from oracle import press_oracle as O
from tests import cpu_backend
from tests.tiny_models import tiny_llama, tiny_qwen3, word_tokenizer, words


@pytest.fixture
def backend(monkeypatch):
    cpu_backend.install(monkeypatch)


@pytest.fixture(scope="module")
def model():
    return tiny_llama()


@pytest.fixture(scope="module")
def pipe():
    # device pinned: with a GPU present, transformers' Pipeline would move the CPU model to cuda:0
    return KVPressTextGenerationPipeline(model=tiny_llama(), tokenizer=word_tokenizer(), device="cpu")


def test_product_refuses_cpu_tensors_without_backend():
    k = torch.randn(1, 2, 64, 16)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        native.knorm_compress(k, k, 32)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        KnormPress(0.5).compress(None, None, k, k, None, {})


def test_context_manager_adds_and_removes_hooks(model):
    press = KnormPress(compression_ratio=0.2)
    with press(model):
        for layer in model.model.layers:
            assert len(layer.self_attn._forward_hooks) == 1
    for layer in model.model.layers:
        assert len(layer.self_attn._forward_hooks) == 0


def test_hooks_removed_when_forward_raises(model):
    press = KnormPress(compression_ratio=0.2)  # no backend installed: compress raises on CPU
    with pytest.raises(RuntimeError):
        with press(model):
            model(torch.randint(0, 200, (1, 32)), past_key_values=DynamicCache())
    for layer in model.model.layers:
        assert len(layer.self_attn._forward_hooks) == 0


@pytest.mark.parametrize("press_cls", [KnormPress, StreamingLLMPress, SnapKVPress, ExpectedAttentionPress])
@pytest.mark.parametrize("ratio", [0.0, 0.2, 0.5, 0.7])
def test_compression_applies_only_inside_context(backend, model, press_cls, ratio):
    press = press_cls(compression_ratio=ratio)
    ids = torch.randint(0, 200, (2, 130))
    with press(model):
        cache = model(ids, past_key_values=DynamicCache()).past_key_values
    want = kept_count(130, ratio)
    for layer in cache.layers:
        assert layer.keys.shape[2] == want == cache.get_seq_length()
        assert layer.values.shape[2] == want
    cache = model(ids, past_key_values=DynamicCache()).past_key_values
    for layer in cache.layers:
        assert layer.keys.shape[2] == 130


def test_no_compression_while_decoding(backend, model):
    press = KnormPress(compression_ratio=0.5)
    ids = torch.randint(0, 200, (1, 64))
    with press(model):
        cache = model(ids, past_key_values=DynamicCache()).past_key_values
        assert cache.get_seq_length() == 32
        model(torch.randint(0, 200, (1, 1)), past_key_values=cache)  # decoding step: untouched
        assert cache.get_seq_length() == 33
        model(torch.randint(0, 200, (1, 7)), past_key_values=cache)  # multi-token continuation
        assert cache.get_seq_length() == 40


class StoreKnormPress(KnormPress):
    """Overrides score(): compress() must then go through score() + the generic select path."""

    def __post_init__(self):
        super().__post_init__()
        self.scores = []

    def score(self, module, hidden_states, keys, values, attentions, kwargs):
        s = -keys.norm(dim=-1)
        self.scores.append(s)
        return s


def test_kept_keys_are_the_highest_scoring(backend, model):
    """Reference tests/presses/test_presses.py:143-162."""
    for ratio in [0.0, 0.2, 0.4, 0.6, 0.8]:
        press = StoreKnormPress(compression_ratio=ratio)
        with press(model):
            cache = model(torch.randint(0, 200, (5, 256)), past_key_values=DynamicCache()).past_key_values
        if ratio == 0:
            assert press.scores == []  # early-out before scoring (scorer_press.py:86-87)
            continue
        assert len(press.scores) == len(cache.layers)
        for scores, layer in zip(press.scores, cache.layers):
            kept = -layer.keys.norm(dim=-1)
            n = kept.shape[-1]
            assert torch.allclose(scores.sort(-1).values[..., -n:], kept.sort(-1).values)


def test_score_is_a_public_standalone_method(backend, model):
    attn = model.model.layers[0].self_attn
    attn.rotary_emb = model.model.rotary_emb
    hidden = torch.randn(1, 100, model.config.hidden_size)
    k = torch.randn(1, 2, 100, 16)
    v = torch.randn(1, 2, 100, 16)
    pe = model.model.rotary_emb(hidden, torch.arange(100)[None])
    for press in (KnormPress(0.5), StreamingLLMPress(0.5), SnapKVPress(0.5, window_size=16),
                  ExpectedAttentionPress(0.5)):
        s = press.score(attn, hidden, k, v, None, {"position_embeddings": pe})
        assert s.shape == (1, 2, 100)
    press = KnormPress(0.3)
    press.compression_ratio = 0.6  # wrappers mutate it in place
    k2, v2 = press.compress(attn, hidden, k, v, None, {})
    assert k2.shape[2] == kept_count(100, 0.6)


def test_qwen3_prologue_uses_q_norm(backend):
    qwen = tiny_qwen3()
    ids = torch.randint(0, 200, (1, 150))
    for press in (SnapKVPress(0.5, window_size=16), ExpectedAttentionPress(0.5)):
        with press(qwen):
            cache = qwen(ids, past_key_values=DynamicCache()).past_key_values
        assert cache.get_seq_length() == 75
    attn = qwen.model.layers[0].self_attn
    hidden = torch.randn(1, 9, qwen.config.hidden_size)
    from kvpress_b200.utils import get_prerope_query_states
    got = get_prerope_query_states(attn, hidden)
    want = O.prerope_queries(hidden, attn.q_proj.weight, 4, 16, q_norm_weight=attn.q_norm.weight,
                             eps=attn.q_norm.variance_epsilon)
    assert torch.allclose(got, want, atol=1e-6)


# ---------------------------------------------------------------------------------------------------
# pipeline
# ---------------------------------------------------------------------------------------------------
def test_pipeline_lengths_and_logs(backend, pipe, caplog):
    context = words(23, seed=1)
    with caplog.at_level(logging.DEBUG):
        out = pipe(context, question=words(3, seed=2), press=ExpectedAttentionPress(compression_ratio=0.4),
                   max_new_tokens=5)
    assert isinstance(out["answer"], str)
    messages = [r.message for r in caplog.records]
    n_ctx = 24  # bos + 23 words
    assert f"Context Length: {n_ctx}" in messages
    assert f"Compressed Context Length: {kept_count(n_ctx, 0.4)}" in messages


def test_pipeline_questions_and_cache_invariance(backend, pipe):
    context = words(200, seed=3)
    cache = DynamicCache()
    out = pipe(context, questions=[words(4, seed=4), words(5, seed=5)], press=KnormPress(0.5), cache=cache,
               max_new_tokens=4)
    assert len(out["answers"]) == 2
    assert cache.get_seq_length() == kept_count(201, 0.5)  # answers were stripped from the cache again
    keys_before = [layer.keys.clone() for layer in cache.layers]
    pipe.generate_answer(torch.randint(0, 200, (1, 6)), cache, context_length=201, max_new_tokens=3)
    pipe._remove_answer_from_cache(cache, [kept_count(201, 0.5)] * len(cache.layers))
    for before, layer in zip(keys_before, cache.layers):
        assert torch.equal(before, layer.keys)
    with pytest.raises(AssertionError):
        pipe(context, question="w3", questions=["w4"])


def test_pipeline_matches_manual_prefill_and_greedy_decode(backend, pipe):
    """Reference tests/test_generate.py: the pipeline answer equals a hand-rolled prefill + greedy loop."""
    context, question = words(120, seed=6), words(4, seed=7)
    press = KnormPress(0.5)
    answer = pipe(context, question=question, press=press, max_new_tokens=6)["answer"]
    tok, model = pipe.tokenizer, pipe.model
    ctx_ids = tok.encode(tok.bos_token + context, return_tensors="pt", add_special_tokens=False)
    q_ids = tok.encode(question + "\n", return_tensors="pt", add_special_tokens=False)
    cache = DynamicCache()
    with press(model):
        model.model(input_ids=ctx_ids, past_key_values=cache)
    pos = torch.arange(ctx_ids.shape[1], ctx_ids.shape[1] + q_ids.shape[1])[None]
    out = model(input_ids=q_ids, past_key_values=cache, position_ids=pos)
    ids = [out.logits[0, -1].argmax()]
    for i in range(5):
        out = model(input_ids=ids[-1].view(1, 1), past_key_values=cache, position_ids=pos[:, -1:] + 1 + i)
        ids.append(out.logits[0, -1].argmax())
        if ids[-1].item() == model.generation_config.eos_token_id:
            break
    assert answer == tok.decode(torch.stack(ids), skip_special_tokens=True)


# ---------------------------------------------------------------------------------------------------
# DecodingPress
# ---------------------------------------------------------------------------------------------------
def test_decoding_ratio_arithmetic():
    """Reference tests/test_decoding_compression.py:236-271."""
    assert kept_count(108, 0.5) == 54
    r = find_target_compression_ratio(58, 54)
    assert abs(r - (1 - 54 / 58)) < 1e-3 and kept_count(58, r) == 54
    assert find_target_compression_ratio(40, 54) == 0.0
    for q_len, target in [(2560, 2048), (4607, 2048), (131072, 39321), (2049, 2048), (3000, 1), (7, 3)]:
        assert find_target_compression_ratio(q_len, target) == O.find_target_compression_ratio(q_len, target)


@pytest.mark.parametrize("base", [KnormPress, StreamingLLMPress, SnapKVPress, ExpectedAttentionPress])
def test_decoding_press_size_bounds(backend, pipe, base):
    """target <= len <= target + interval - 1 after enough steps (reference :50-183)."""
    kw = {"window_size": 4} if base is SnapKVPress else {}
    press = DecodingPress(base_press=base(**kw), compression_interval=8, target_size=48)
    cache = DynamicCache()
    pipe(words(100, seed=8), question=words(3, seed=9), press=press, cache=cache, max_new_tokens=30)
    # answers are stripped: inspect during generation instead
    sizes = []
    orig = press.forward_hook

    def spy(module, inp, kwargs, output):
        out = orig(module, inp, kwargs, output)
        if module.layer_idx == 0:
            sizes.append(kwargs["past_key_values"].get_seq_length(0))
        return out

    press.forward_hook = spy
    pipe(words(100, seed=8), question=words(3, seed=9), press=press, cache=DynamicCache(), max_new_tokens=30)
    assert min(sizes[8:]) >= 48 and max(sizes[8:]) <= 48 + 8 - 1
    assert 48 in sizes
    assert press.layer_step_counts == {} and press.hidden_states_buffer == {}  # reset() on exit


def test_decoding_press_buffers_only_when_needed(backend, pipe):
    cheap = DecodingPress(base_press=KnormPress(), compression_interval=4, target_size=32)
    costly = DecodingPress(base_press=SnapKVPress(window_size=4), compression_interval=6, target_size=32)
    seen = {}
    for name, press in (("cheap", cheap), ("costly", costly)):
        orig = press.forward_hook

        def spy(module, inp, kwargs, output, press=press, orig=orig, name=name):
            out = orig(module, inp, kwargs, output)
            seen[name] = max(seen.get(name, 0), len(press.hidden_states_buffer[module.layer_idx]))
            return out

        press.forward_hook = spy
        pipe(words(60, seed=10), question=words(2, seed=11), press=press, max_new_tokens=10)
    assert seen["cheap"] == 0 and seen["costly"] > 0


def test_decoding_press_rejects_multiple_questions(backend, pipe):
    press = DecodingPress(base_press=KnormPress(), compression_interval=4, target_size=32)
    with pytest.raises(ValueError):
        pipe(words(50), questions=["w3", "w4"], press=press)
    with pytest.raises(AssertionError):
        DecodingPress(base_press=object())


def test_public_surface():
    for name in ["BasePress", "ScorerPress", "KnormPress", "SnapKVPress", "ExpectedAttentionPress",
                 "StreamingLLMPress", "DecodingPress", "KVPressTextGenerationPipeline"]:
        assert hasattr(kvpress_b200, name)
    import dataclasses
    defaults = {f.name: f.default for f in dataclasses.fields(SnapKVPress)}
    assert defaults == {"compression_ratio": 0.0, "window_size": 64, "kernel_size": 5}
    defaults = {f.name: f.default for f in dataclasses.fields(ExpectedAttentionPress)}
    assert defaults == {"compression_ratio": 0.0, "n_future_positions": 512, "n_sink": 4, "use_covariance": True,
                        "use_vnorm": True, "epsilon": 0.0}
    assert {f.name: f.default for f in dataclasses.fields(StreamingLLMPress)} == {"compression_ratio": 0.0, "n_sink": 4}
    d = {f.name: f.default for f in dataclasses.fields(DecodingPress) if f.name != "base_press"}
    assert d == {"compression_interval": 512, "target_size": 2048, "hidden_states_buffer_size": 256}
    from transformers.pipelines import PIPELINE_REGISTRY
    assert "kv-press-text-generation" in PIPELINE_REGISTRY.get_supported_tasks()
    with pytest.raises(AssertionError):
        ScorerPress(compression_ratio=1.0)


def test_host_staging_has_no_cpu_path():
    """compress_host needs pinned host buffers and a CUDA device; on a CPU-only box it must refuse, not fall back."""
    from kvpress_b200 import host_staging

    K = torch.randn(1, 2, 64, 64).to(torch.bfloat16)
    with pytest.raises(RuntimeError, match="pinned"):
        host_staging.compress_host("knorm", K, K, 32)


def test_prefill_decoding_press_runs_both_phases(backend, pipe):
    """prefill_decoding_press.py:18-103: the prefill press shortens the prompt cache once, the decoding press then
    keeps the cache inside [target, target + interval) while tokens are generated; decoding state is reset on exit."""
    from kvpress_b200 import PrefillDecodingPress

    decoding = DecodingPress(base_press=KnormPress(), compression_interval=6, target_size=40)
    press = PrefillDecodingPress(prefilling_press=KnormPress(0.5), decoding_press=decoding)
    sizes = []
    orig = press.forward_hook

    def spy(module, inp, kwargs, output):
        out = orig(module, inp, kwargs, output)
        if module.layer_idx == 0:
            sizes.append(kwargs["past_key_values"].get_seq_length(0))
        return out

    press.forward_hook = spy
    context = words(100, seed=20)
    pipe(context, question=words(3, seed=21), press=press, cache=DynamicCache(), max_new_tokens=24)
    n_ctx = len(pipe.tokenizer(context)["input_ids"]) if hasattr(pipe.tokenizer(context), "__getitem__") else 100
    assert sizes[0] == kept_count(n_ctx, 0.5)                  # prefill phase: prefilling_press only
    assert min(sizes[8:]) >= 40 and max(sizes[8:]) <= 40 + 6 - 1 and 40 in sizes
    assert decoding.layer_step_counts == {}
    # either side may be missing
    only_prefill = PrefillDecodingPress(prefilling_press=KnormPress(0.5))
    cache = DynamicCache()
    pipe(context, question=words(3, seed=21), press=only_prefill, cache=cache, max_new_tokens=4)
    assert cache.get_seq_length() == kept_count(n_ctx, 0.5)


def test_compression_ratio_decoding_press_target_follows_tokens_seen(backend, model):
    """compression_ratio_decoding_press.py:13-50: target = int(tokens_seen * (1 - r)) from position_ids."""
    from kvpress_b200 import CompressionRatioDecodingPress

    press = CompressionRatioDecodingPress(base_press=KnormPress(), compression_interval=4, target_compression_ratio=0.75)
    assert press._resolve_target_size({"position_ids": torch.tensor([[198, 199]])}) == 50
    assert press._resolve_target_size({"position_ids": torch.tensor([[0]])}) == 1
    with pytest.raises(NotImplementedError):
        press._resolve_target_size({})
    with pytest.raises(AssertionError):
        CompressionRatioDecodingPress(base_press=KnormPress(), target_compression_ratio=1.0)
    # through the hooks: 60-token prompt, then single-token steps with explicit position_ids
    ids = torch.randint(2, 250, (1, 60))
    cache = DynamicCache()
    with press(model):
        model.model(input_ids=ids, past_key_values=cache)
        assert cache.get_seq_length() == 60               # prefill untouched
        for step in range(8):
            pos = torch.tensor([[60 + step]])
            model.model(input_ids=torch.randint(2, 250, (1, 1)), past_key_values=cache, position_ids=pos)
        # two compactions happened (steps 4 and 8); the last one saw 68 tokens -> int(68 * 0.25) = 17
        assert cache.get_seq_length() == 17


@torch.no_grad()
def test_adakv_fake_keys_equal_an_explicit_per_head_mask(backend, model):
    """attention_patch.py: overwriting the pruned keys of a head with the hyperplane fake key must give the same
    decoding step as masking those (head, position) pairs with -inf. Also checks the AdaKV budget arithmetic."""
    import copy

    from kvpress_b200 import AdaKVPress

    ids = torch.randint(2, 250, (2, 90))
    S, H, G = 90, model.config.num_key_value_heads, model.config.num_attention_heads // model.config.num_key_value_heads
    press = AdaKVPress(KnormPress(0.6), alpha_safeguard=0.25)
    cache = DynamicCache()
    attns = [layer.self_attn for layer in model.model.layers]
    with press(model):
        model.model(input_ids=ids, past_key_values=cache)
        masks = [a.masked_key_indices for a in attns]
        n_kept = kept_count(S, 0.6)
        for b, h, s in masks:
            assert b.numel() == 2 * H * (S - n_kept)
            pruned_per_head = torch.zeros(2, H, dtype=torch.long).index_put_((b, h), torch.ones_like(b), accumulate=True)
            assert (S - pruned_per_head >= int(n_kept * 0.25)).all()        # safeguard: every head keeps n_safe
            assert pruned_per_head.sum(1).eq(H * (S - n_kept)).all()         # same total budget per batch element
        patched_cache = copy.deepcopy(cache)
        y_patch = model.model(input_ids=ids[:, :1], past_key_values=patched_cache).last_hidden_state
    for a in attns:
        a.masked_key_indices = None

    # the same step with an explicit additive mask per layer (q-heads of a kv-head share its mask)
    layer_masks = []
    for b, h, s in masks:
        m = torch.zeros(2, H, 1, S + 1)
        m[b, h, 0, s] = float("-inf")
        layer_masks.append(m.repeat_interleave(G, dim=1))
    handles = []
    for a, m in zip(attns, layer_masks):
        def pre(module, args, kwargs, m=m):
            kwargs["attention_mask"] = m
            return args, kwargs
        handles.append(a.register_forward_pre_hook(pre, with_kwargs=True))
    try:
        y_mask = model.model(input_ids=ids[:, :1], past_key_values=copy.deepcopy(cache)).last_hidden_state
    finally:
        for hd in handles:
            hd.remove()
    y_plain = model.model(input_ids=ids[:, :1], past_key_values=copy.deepcopy(cache)).last_hidden_state
    assert torch.allclose(y_patch, y_mask, atol=1e-5)
    assert not torch.allclose(y_patch, y_plain, atol=1e-4)


# ---- shapes outside the tcgen05 instantiations: cuBLAS score stage (kvpress_b200/wide_head_scores.py) ----------------
def test_wide_head_shape_predicates():
    from kvpress_b200 import wide_head_scores as W

    assert W.snapkv_on_tensor_cores(128, 4, 64) and W.snapkv_on_tensor_cores(64, 8, 64)
    assert not W.snapkv_on_tensor_cores(96, 1, 64) and not W.snapkv_on_tensor_cores(256, 2, 64)
    assert not W.snapkv_on_tensor_cores(128, 16, 64)                      # 1024 window-query rows per kv head
    assert W.expected_attention_on_tensor_cores(96, 3, False)             # the covariance-free scan takes any head_dim
    assert not W.expected_attention_on_tensor_cores(96, 1, True) and not W.expected_attention_on_tensor_cores(128, 16, False)


def test_wide_head_scores_refuse_cpu_tensors():
    from kvpress_b200 import wide_head_scores as W

    k = torch.randn(1, 1, 40, 96).to(torch.bfloat16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        W.snapkv_scores(k, k[:, :, -8:], 8, 5)


@pytest.mark.parametrize("D,G,dtype", [(96, 1, torch.bfloat16), (256, 2, torch.bfloat16), (96, 3, torch.float16)])
def test_wide_head_score_math_is_the_fp32_formula_rounded_once(monkeypatch, D, G, dtype):
    """The arithmetic of the cuBLAS score stage (device check lifted for the CPU box) against the oracle's fp32
    evaluation of the reference formulas: <= 1 ulp of the 16-bit score, forced positions carry max + 1."""
    from kvpress_b200 import wide_head_scores as W
    from oracle import press_oracle as O
    from tests.conftest import ulp16_diff

    monkeypatch.setattr(W, "_require_cuda", lambda t: None)
    torch.manual_seed(D + G)
    B, Hkv, S, w = 2, 2, 300, 16
    k = torch.randn(B, Hkv, S, D).to(dtype)
    v = torch.randn(B, Hkv, S, D).to(dtype)
    q = (torch.randn(B, Hkv * G, w, D) * 0.5).to(dtype)
    got = W.snapkv_scores(k, q, w, 5, chunk=128)
    want = O.snapkv_scores_fp32(q, k, w, 5).to(dtype)
    assert ulp16_diff(got[..., :-w], want[..., :-w]).max().item() <= 1
    assert (got[..., -w:] == (got[..., :-w].float().max() + 1).to(dtype)).all()
    mu = (torch.randn(B, Hkv * G, D) * 0.3).to(dtype)
    a = torch.randn(B, Hkv * G, D, D) / D ** 0.5
    cov = (a @ a.transpose(-1, -2) * 0.5).to(dtype)
    for c, eps, vn in ((cov, 0.0, True), (None, 0.0, False), (cov, 1e-2, True)):
        got = W.expected_attention_scores(k, v, mu, c, eps, 4, vn, chunk=64)
        want = O.expected_attention_scores_fp32(k, v, mu, c, eps, 4, vn).to(dtype)
        assert ulp16_diff(got[..., 4:], want[..., 4:]).max().item() <= 1
        assert (got[..., :4] == (got[..., 4:].float().max() + 1).to(dtype)).all()
