"""Differential test against the UNMODIFIED reference: the re-written presses, driven through the same hooks on the
same random-init model, must retain the same rows as the reference presses. What the reference retained on these exact
inputs is stored in tests/golden/differential.npz (written by tests/golden/make_differential.py from a checkout of the
original package), so the comparison runs on any host.

Retained rows are identified by their position in the uncompressed prefill cache, which is exact on any host. Float
results of the reference (kept key norms, re-rotated keys, a decoding step's output) are compared within the spread
the tiny model's own CPU forward has between hosts: its GEMMs round differently under different instruction sets."""
import json

import numpy as np
import pytest
import torch
from transformers import DynamicCache

from kvpress_b200 import ExpectedAttentionPress, KeyDiffPress, KnormPress, SnapKVPress, StreamingLLMPress
from tests import cpu_backend
from tests.conftest import GOLDEN_DIR
from tests.tiny_models import tiny_llama, tiny_qwen3

# float results of the reference: a float32 forward on another instruction set differs in the last bits only
FLOAT_TOL = dict(rtol=1e-5, atol=1e-5)


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN_DIR / "differential.npz")


def row_signature(x):
    """One float64 per row of x [..., n, D]: its dot product with a fixed random vector."""
    g = torch.Generator().manual_seed(0)
    w = torch.randn(x.shape[-1], generator=g, dtype=torch.float64)
    return x.double() @ w


def _rows_signature(keys, values):
    """Order-independent signature of the retained (K, V) rows of every head."""
    return (row_signature(keys) + 3.0 * row_signature(values)).sort(-1).values


def full_cache(model, ids):
    cache = DynamicCache()
    with torch.no_grad():
        model.model(input_ids=ids, past_key_values=cache)
    return cache


def kept_positions(cache, full):
    """Per layer, [B, H, n] positions in the uncompressed prefill cache `full` of the rows `cache` retains, in cache
    order. No press modifies values and every row's value vector is distinct, so a row is found by its values."""
    out = []
    for lc, lf in zip(cache.layers, full.layers):
        eq = (lc.values[:, :, :, None, :] == lf.values[:, :, None, :, :]).all(-1)        # [B, H, n, S]
        assert (eq.sum(-1) == 1).all(), "a retained row is not a row of the uncompressed cache"
        out.append(eq.int().argmax(-1))
    return out


def masked_triples(attns):
    """AdaKV: per layer, the set of masked (batch, head, position) triples as a sorted [N, 3] tensor."""
    return [torch.unique(torch.stack(a.masked_key_indices, dim=-1).long(), dim=0) for a in attns]


def _assert_same_rows(cache, key, ref, model, ids, ordered=False):
    """`cache` retains, layer by layer, the rows the reference retained (stored under `key`); `ordered`: in the same
    row order too, i.e. the caches are equal row by row."""
    assert [la.keys.shape[2] for la in cache.layers] == ref[f"{key}/len"].tolist()
    for i, pos in enumerate(kept_positions(cache, full_cache(model, ids))):
        want = torch.from_numpy(ref[f"{key}/pos{i}"]).long()
        assert torch.equal(pos if ordered else pos.sort(-1).values, want if ordered else want.sort(-1).values), (key, i)


CASES = [
    ("knorm", lambda m: m.KnormPress, KnormPress, {}),
    ("streaming", lambda m: m.StreamingLLMPress, StreamingLLMPress, {"n_sink": 4}),
    ("snapkv", lambda m: m.SnapKVPress, SnapKVPress, {"window_size": 16, "kernel_size": 5}),
    ("expected_attention", lambda m: m.ExpectedAttentionPress, ExpectedAttentionPress, {"n_sink": 4}),
    ("keydiff", lambda m: m.KeyDiffPress, KeyDiffPress, {}),
    ("tova", lambda m: m.TOVAPress, __import__("kvpress_b200").TOVAPress, {}),
]
SAME_ROWS_RATIOS = [0.25, 0.5, 0.7]
FAMILIES = ["llama", "qwen3"]


def _model(family, **kw):
    return tiny_llama(**kw) if family == "llama" else tiny_qwen3(**kw)


def same_rows_ids():
    # distinct tokens per sequence: a repeated token gives layer-0 keys of exactly equal norm (RoPE keeps
    # norms), i.e. exact score ties that torch.topk and the kernels may legitimately break differently
    return _distinct_ids(5)


@pytest.mark.parametrize("name,ref_cls,our_cls,kw", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("ratio", SAME_ROWS_RATIOS)
@pytest.mark.parametrize("family", FAMILIES)
def test_same_rows_as_reference(monkeypatch, ref, name, ref_cls, our_cls, kw, ratio, family):
    cpu_backend.install(monkeypatch)
    model = _model(family)
    ids = same_rows_ids()
    S = ids.shape[1]
    key = f"same_rows/{name}/{ratio}/{family}"

    ours = DynamicCache()
    with our_cls(compression_ratio=ratio, **kw)(model):
        model.model(input_ids=ids, past_key_values=ours)

    assert ours.get_seq_length() == int(ref[f"{key}/len"][0]) == int(S * (1 - ratio))
    if name == "knorm":
        # Qwen3's k_norm makes every key norm (nearly) equal: exact ties, broken differently by
        # torch.topk and by the lowest-position rule. The multiset of kept scores must still agree.
        for i, lo in enumerate(ours.layers):
            want = torch.from_numpy(ref[f"{key}/norms{i}"])
            assert lo.keys.shape[2] == want.shape[-1]
            assert torch.allclose(lo.keys.norm(dim=-1).sort(-1).values, want)
    else:
        _assert_same_rows(ours, key, ref, model, ids)


@pytest.mark.parametrize("inner", ["streaming", "snapkv"])
@pytest.mark.parametrize("family", FAMILIES)
def test_key_rerotation_same_cache_as_reference(monkeypatch, ref, inner, family):
    """KeyRerotationPress (key_rerotation_press.py:133-152): the reference sorts the kept indices, so the
    compacted cache must agree ROW BY ROW, re-rotated keys included."""
    from kvpress_b200 import KeyRerotationPress

    cpu_backend.install(monkeypatch)
    model = _model(family)
    ids = _distinct_ids(7)
    S, ratio = ids.shape[1], 0.4
    _, _, our_cls, kw = next(c for c in CASES if c[0] == inner)
    key = f"rerotation/{inner}/{family}"

    ours = DynamicCache()
    press = KeyRerotationPress(our_cls(compression_ratio=ratio, **kw))
    assert press.compression_ratio == ratio
    with press(model):
        model.model(input_ids=ids, past_key_values=ours)

    assert ours.get_seq_length() == int(S * (1 - ratio))
    _assert_same_rows(ours, key, ref, model, ids, ordered=True)
    for i, lo in enumerate(ours.layers):
        assert torch.allclose(row_signature(lo.keys), torch.from_numpy(ref[f"{key}/ksig{i}"]), **FLOAT_TOL)


def _distinct_ids(seed, n=160, batch=2):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randperm(250, generator=g)[:n] + 2 for _ in range(batch)])


def _prefill(press, model, ids):
    cache = DynamicCache()
    with press(model):
        model.model(input_ids=ids, past_key_values=cache)
    return cache


PYRAMID_CASES = [(0.3, 20), (0.6, 4), (0.5, 1), (0.9, 20)]
PYRAMID_GRID = [(q_len, r, b, layer) for q_len in (100, 777, 4096, 131072) for r in (0.1, 0.5, 0.75, 0.95)
                for b in (1, 5, 20) for layer in (0, 7, 31)]


@pytest.mark.parametrize("ratio,beta", PYRAMID_CASES)
def test_pyramidkv_same_rows_and_budgets_as_reference(monkeypatch, ref, ratio, beta):
    """pyramidkv_press.py:47-112: per-layer budgets (incl. the fallback branch) and the kept rows."""
    from kvpress_b200 import PyramidKVPress
    from kvpress_b200.presses.pyramidkv_press import pyramid_layer_budget

    cpu_backend.install(monkeypatch)
    model = tiny_llama(layers=4)
    ids = _distinct_ids(11)
    ours = _prefill(PyramidKVPress(compression_ratio=ratio, window_size=16, kernel_size=5, beta=beta), model, ids)
    lens = [layer.keys.shape[2] for layer in ours.layers]
    n_layers = model.config.num_hidden_layers
    assert lens == [pyramid_layer_budget(160, ratio, 16, beta, n_layers, i) for i in range(n_layers)]
    _assert_same_rows(ours, f"pyramid/{ratio}/{beta}", ref, model, ids)
    # the budget formula alone, over a grid, against the reference method (window 64, 32 layers)
    got = [pyramid_layer_budget(q_len, r, 64, b, 32, layer) for q_len, r, b, layer in PYRAMID_GRID]
    assert got == ref["pyramid_budget_grid"].tolist()


CHUNK_CASES = [(160, 40), (150, 64), (100, 256)]


def _inner(inner, ratio):
    """(our press, its kwargs) of the inner scorers the wrapper tests use."""
    _, _, our_cls, kw = next(c for c in CASES if c[0] == inner)
    if inner == "snapkv":
        kw = {"window_size": 8, "kernel_size": 3}
    return our_cls(compression_ratio=ratio, **kw)


@pytest.mark.parametrize("inner", ["knorm", "snapkv"])
@pytest.mark.parametrize("n_tokens,chunk", CHUNK_CASES)
def test_chunk_press_same_rows_as_reference(monkeypatch, ref, inner, n_tokens, chunk):
    from kvpress_b200 import ChunkPress

    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    ids = _distinct_ids(12, n=n_tokens)
    ours = _prefill(ChunkPress(_inner(inner, 0.5), chunk_length=chunk), model, ids)
    _assert_same_rows(ours, f"chunk/{inner}/{n_tokens}/{chunk}", ref, model, ids)


def per_layer_ratios(model):
    return [0.2, 0.6][: model.config.num_hidden_layers] + [0.5] * max(0, model.config.num_hidden_layers - 2)


def test_composed_and_per_layer_wrappers_same_rows_as_reference(monkeypatch, ref):
    from kvpress_b200 import ComposedPress, PerLayerCompressionPress

    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    ids = _distinct_ids(13)
    # second press = Knorm: its scores do not depend on the ROW ORDER the first press leaves behind (the reference
    # emits top-k order, this package ascending positions; index-based scorers such as SnapKV's window or
    # StreamingLLM's sinks would read a different "last w rows" from the reference's permuted cache)
    op = ComposedPress([SnapKVPress(0.25, window_size=16), KnormPress(0.4)])
    ours = _prefill(op, model, ids)
    assert op.compression_ratio == pytest.approx(float(ref["composed/ratio"]))
    _assert_same_rows(ours, "composed", ref, model, ids)

    op = PerLayerCompressionPress(SnapKVPress(window_size=16), per_layer_ratios(model))
    ours = _prefill(op, model, ids)
    assert op.compression_ratio == pytest.approx(float(ref["per_layer/ratio"]))
    with pytest.raises(AttributeError):
        op.compression_ratio = 0.1
    _assert_same_rows(ours, "per_layer", ref, model, ids)


def test_random_press_same_rows_as_reference_on_cpu(monkeypatch, ref):
    from kvpress_b200 import RandomPress

    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    ids = _distinct_ids(14)
    _assert_same_rows(_prefill(RandomPress(0.5, seed=3), model, ids), "random", ref, model, ids)


def adakv_run(press, model, ids, with_cache_position):
    """Prefill under `press`, then one decoding step: (cache, masked triples per layer, the step's hidden states)."""
    S = ids.shape[1]
    attns = [layer.self_attn for layer in model.model.layers]
    cache = DynamicCache()
    with press(model):
        extra = {"cache_position": torch.arange(S)} if with_cache_position else {}
        model.model(input_ids=ids, past_key_values=cache, **extra)
        m = masked_triples(attns)
        extra = {"cache_position": torch.tensor([S])} if with_cache_position else {}
        step = model.model(input_ids=ids[:, :1], past_key_values=cache, **extra).last_hidden_state
    for a in attns:
        a.masked_key_indices = None
    return cache, m, step


@pytest.mark.parametrize("inner", ["expected_attention", "snapkv"])
@pytest.mark.parametrize("alpha", [0.2, 0.0, 1.0])
def test_adakv_masks_the_same_keys_as_reference(monkeypatch, ref, inner, alpha):
    """adakv_press.py:53-78: per-head safeguard + bottom-k across heads; the pruned (batch, head, position)
    triples must be the reference's, and one decoding step through attention_patch must give the same output."""
    from kvpress_b200 import AdaKVPress

    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    ids = _distinct_ids(21)
    S = ids.shape[1]
    _, _, our_cls, kw = next(c for c in CASES if c[0] == inner)
    key = f"adakv/{inner}/{alpha}"

    c_our, m_our, y_our = adakv_run(AdaKVPress(our_cls(compression_ratio=0.5, **kw), alpha_safeguard=alpha), model, ids,
                                    False)
    H = model.config.num_key_value_heads
    for i, a in enumerate(m_our):
        assert a.shape[0] == ids.shape[0] * H * (S - int(S * 0.5))
        assert torch.equal(a, torch.from_numpy(ref[f"{key}/masked{i}"]).long())
    assert c_our.get_seq_length() == S + 1      # AdaKV never shrinks the cache
    assert torch.allclose(y_our, torch.from_numpy(ref[f"{key}/step"]), atol=1e-5)


CHUNKKV_CASES = [(160, 20), (150, 20), (150, 32), (15, 20)]


@pytest.mark.parametrize("inner", ["knorm", "snapkv", "expected_attention"])
@pytest.mark.parametrize("n_tokens,chunk", CHUNKKV_CASES)
def test_chunkkv_press_same_rows_as_reference(monkeypatch, ref, inner, n_tokens, chunk):
    """chunkkv_press.py:52-117: whole chunks kept, ranked by head-summed mean score; ragged tail; S < chunk."""
    from kvpress_b200 import ChunkKVPress

    if inner != "knorm" and n_tokens < 32:
        pytest.skip("window scorers need more tokens than their window")
    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    ids = _distinct_ids(31, n=n_tokens)
    ours = _prefill(ChunkKVPress(_inner(inner, 0.4), chunk_length=chunk), model, ids)
    # S < chunk: plain press.compress, same rows (the reference in top-k order); otherwise both emit position order:
    # the caches are equal row by row
    _assert_same_rows(ours, f"chunkkv/{inner}/{n_tokens}/{chunk}", ref, model, ids, ordered=n_tokens >= chunk)
    if n_tokens >= chunk:
        full = full_cache(model, ids)
        for pos, lo, lf in zip(kept_positions(ours, full), ours.layers, full.layers):
            assert torch.equal(lo.keys, lf.keys.gather(2, pos[..., None].expand_as(lo.keys)))


@pytest.mark.parametrize("inner", ["knorm", "keydiff"])
@pytest.mark.parametrize("block_size", [16, 50, 400])
def test_block_press_same_rows_as_reference(monkeypatch, ref, inner, block_size):
    """block_press.py:49-98 incl. the reference's own invariant (tests/presses/test_block_press.py:30-63):
    a block at least as long as the context is the plain press."""
    from kvpress_b200 import BlockPress

    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    ids = _distinct_ids(32)
    _, _, our_cls, kw = next(c for c in CASES if c[0] == inner)
    ours = _prefill(BlockPress(our_cls(compression_ratio=0.5, **kw), block_size=block_size), model, ids)
    _assert_same_rows(ours, f"block/{inner}/{block_size}", ref, model, ids)
    if block_size >= ids.shape[1]:
        plain = _prefill(our_cls(compression_ratio=0.5, **kw), model, ids)
        for lo, lp in zip(ours.layers, plain.layers):
            assert torch.allclose(_rows_signature(lo.keys, lo.values), _rows_signature(lp.keys, lp.values), atol=1e-9)


def stats_batches():
    return [_distinct_ids(40 + i, n=120, batch=1) for i in range(3)]


def write_reference_stats(ref, folder):
    """The statistics folder the reference's ExpectedAttentionStats.save_pretrained wrote, byte for byte."""
    folder.mkdir(parents=True, exist_ok=True)
    for name in ("config.json", "model.safetensors"):
        (folder / name).write_bytes(ref[f"ea_stats/file/{name}"].tobytes())
    return folder


def test_expected_attention_stats_press_same_rows_and_folder_layout_as_reference(monkeypatch, ref, tmp_path):
    """expected_attention_with_stats.py:21-110: stored (mu, Sigma) per layer instead of the per-prompt prologue;
    statistics folders are interchangeable with the reference's PyTorchModelHubMixin layout; the offline collector
    reproduces the reference formula (mean, unbiased covariance of the pre-RoPE queries beyond n_sink)."""
    from safetensors import safe_open

    from kvpress_b200 import ExpectedAttentionStatsPress
    from kvpress_b200.presses.expected_attention_with_stats import ExpectedAttentionStats, collect_query_statistics

    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    cfg = model.config
    L, Hq, D = cfg.num_hidden_layers, cfg.num_attention_heads, cfg.head_dim
    batches = stats_batches()
    stats = collect_query_statistics(model, batches, n_sink=4)
    # independent restatement of the reference's collect_queries arithmetic
    from kvpress_b200.utils import get_prerope_query_states
    qs = [[] for _ in range(L)]
    hooks = [layer.self_attn.register_forward_pre_hook(
        lambda m, a, kw, i=i: qs[i].append(get_prerope_query_states(m, kw["hidden_states"])[:, :, 4:]), with_kwargs=True)
        for i, layer in enumerate(model.model.layers)]
    with torch.no_grad():
        for ids in batches:
            model.model(input_ids=ids)
    for h in hooks:
        h.remove()
    for i in range(L):
        q = torch.cat(qs[i], dim=-2)[0]                                     # [Hq, N, D]
        mean = q.mean(dim=-2)
        c = q - mean.unsqueeze(-2)
        assert torch.allclose(stats.query_mean[i], mean, atol=1e-5)
        assert torch.allclose(stats.query_cov[i], c.transpose(-2, -1) @ c / (q.shape[-2] - 1), atol=1e-5)

    # folder layout: ours has the reference's files, config and tensors; the reference's folder -> our loader
    stats.save_pretrained(str(tmp_path / "ours"))
    theirs = write_reference_stats(ref, tmp_path / "theirs")
    assert sorted(p.name for p in (tmp_path / "ours").iterdir()) == sorted(p.name for p in theirs.iterdir())
    assert json.loads((tmp_path / "ours" / "config.json").read_text()) == json.loads((theirs / "config.json").read_text())
    with safe_open(str(tmp_path / "ours" / "model.safetensors"), "pt") as o, \
            safe_open(str(theirs / "model.safetensors"), "pt") as t:
        assert sorted(o.keys()) == sorted(t.keys())
        for k in t.keys():
            assert o.get_tensor(k).dtype == t.get_tensor(k).dtype and o.get_tensor(k).shape == t.get_tensor(k).shape
        assert torch.equal(o.get_tensor("query_mean"), stats.query_mean.data)
        assert torch.equal(o.get_tensor("query_cov"), stats.query_cov.data)
        ref_cov = t.get_tensor("query_cov")
        assert torch.allclose(ref_cov, stats.query_cov.data, atol=1e-5)     # the reference saved what we collected
    back = ExpectedAttentionStats.from_pretrained(str(theirs))
    assert torch.equal(back.query_cov.data, ref_cov) and back.meta["n_sink"] == 4

    # the presses: same rows, with and without covariance; hidden states are not needed
    ids = _distinct_ids(50)
    for use_cov in (True, False):
        op = ExpectedAttentionStatsPress(compression_ratio=0.5, use_covariance=use_cov, stats_folder=str(theirs))
        o_cache = _prefill(op, model, ids)
        assert op.mu.shape == (L, Hq, D)
        assert torch.allclose(op.mu, torch.from_numpy(ref[f"ea_stats/mu/{use_cov}"]), **FLOAT_TOL)
        _assert_same_rows(o_cache, f"ea_stats/press/{use_cov}", ref, model, ids)
    assert ExpectedAttentionStatsPress.needs_hidden_states is False
    with pytest.raises(ValueError, match="No statistics given"):
        ExpectedAttentionStatsPress(0.5).post_init_from_model(model)


# ---------------------------------------------------------------------------------------------------------------------
# pipeline-level differentials: the reference pipeline was driven on the same model (make_differential.py restores the
# `cache_position` kwarg transformers >= 5.3 no longer hands to attention modules, SURVEY F7)
# ---------------------------------------------------------------------------------------------------------------------
def pipeline_inputs():
    from tests.tiny_models import words

    return words(150, seed=3), [words(4, seed=4), words(6, seed=5)]


def position_spy(model, seen):
    def pre(module, args, kwargs):
        if kwargs.get("position_ids") is not None:
            seen.append(kwargs["position_ids"].flatten().tolist())
    return model.model.register_forward_pre_hook(pre, with_kwargs=True)


@pytest.mark.parametrize("family", FAMILIES)
def test_pipeline_with_key_rerotation_matches_reference(monkeypatch, ref, family):
    """pipeline.py:231-232 of the reference: after KeyRerotationPress the question / answer positions continue from
    the COMPRESSED length. Same answers, and the positions the model sees are the reference's."""
    from kvpress_b200 import KeyRerotationPress, KVPressTextGenerationPipeline
    from tests.tiny_models import word_tokenizer

    cpu_backend.install(monkeypatch)
    model = _model(family)
    our_pipe = KVPressTextGenerationPipeline(model=model, tokenizer=word_tokenizer(), device="cpu")
    context, questions = pipeline_inputs()
    seen = []
    h = position_spy(model, seen)
    try:
        ours = our_pipe(context, questions=questions, max_new_tokens=6,
                        press=KeyRerotationPress(StreamingLLMPress(compression_ratio=0.4, n_sink=4)))
    finally:
        h.remove()
    key = f"pipeline_rerotation/{family}"
    assert ours["answers"] == ref[f"{key}/answers"].tolist()
    assert seen == [ref[f"{key}/seen{j}"].tolist() for j in range(int(ref[f"{key}/n_seen"]))] and len(seen) > 2
    n_kept = int(151 * (1 - 0.4))
    assert seen[0][0] == n_kept          # the first question token sits right after the compacted cache


DECODING_KW = dict(compression_interval=7, target_size=40, hidden_states_buffer_size=256)


def decoding_inputs():
    from tests.tiny_models import words

    return words(60, seed=8), words(5, seed=9)


def test_decoding_press_with_stats_press_matches_reference(monkeypatch, ref, tmp_path):
    """DecodingPress(ExpectedAttentionStatsPress): the stats press reads only the LENGTH of the buffered hidden states
    (future RoPE positions); the zero-copy length-only buffer must reproduce the reference's concatenated buffer."""
    from kvpress_b200 import DecodingPress, ExpectedAttentionStatsPress, KVPressTextGenerationPipeline
    from tests.tiny_models import word_tokenizer

    cpu_backend.install(monkeypatch)
    model = tiny_llama()
    our_pipe = KVPressTextGenerationPipeline(model=model, tokenizer=word_tokenizer(), device="cpu")
    context, question = decoding_inputs()
    # few future positions: the average RoPE rotation then depends visibly on where they start (q_len)
    skw = dict(stats_folder=str(write_reference_stats(ref, tmp_path / "stats")), n_future_positions=3)
    op = DecodingPress(base_press=ExpectedAttentionStatsPress(**skw), **DECODING_KW)
    ours_cache = DynamicCache()
    ours = our_pipe(context, question=question, max_new_tokens=24, press=op, cache=ours_cache)
    assert ours["answer"] == str(ref["decoding/answer"])
    assert [la.keys.shape[2] for la in ours_cache.layers] == ref["decoding/len"].tolist()
    # rows appended while decoding have no position in a prefill cache: the row signatures are compared instead
    for i, lo in enumerate(ours_cache.layers):
        assert torch.allclose(_rows_signature(lo.keys, lo.values), torch.from_numpy(ref[f"decoding/sig{i}"]), **FLOAT_TOL)
    assert not op.hidden_states_buffer and not op.hidden_states_lens     # reset on exit, nothing was cloned
