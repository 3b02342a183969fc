"""Generates tests/golden/differential.npz for tests/test_reference_differential.py by driving the UNMODIFIED original
kvpress presses through the same hooks, on the same random-init tiny models and tokens the tests use. Run from the
repository root with the directory that holds the original `kvpress` package:

    python tests/golden/make_differential.py <checkout-of-the-original-kvpress>

Stored per case: the positions (in the uncompressed prefill cache) of the rows every layer retains; where a test
needs them, the reference's float results (kept key norms, re-rotated key signatures, a decoding step's output, row
signatures of a decoded cache), pipeline answers and the positions the model saw, and one statistics folder as the
reference's ExpectedAttentionStats.save_pretrained wrote it (bytes of config.json and model.safetensors).
Harness shims: a stub `fire` module (kvpress imports it at package import for an unrelated CLI) and, as transformers
>= 5.3 no longer hands `cache_position` to attention, that kwarg passed or restored for the reference's hooks.
"""
import sys
import tempfile
import types
from pathlib import Path

import numpy as np
import pytest
import torch
from transformers import DynamicCache

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from tests import test_reference_differential as T  # noqa: E402
from tests.tiny_models import tiny_llama, word_tokenizer  # noqa: E402

OUT = Path(__file__).resolve().parent / "differential.npz"


def import_reference(path):
    sys.modules.setdefault("fire", types.ModuleType("fire"))
    sys.path.insert(0, str(path))
    import kvpress  # noqa

    return kvpress


def ref_prefill(press, model, ids):
    cache = DynamicCache()
    with press(model):
        model.model(input_ids=ids, past_key_values=cache, cache_position=torch.arange(ids.shape[1]))
    return cache


def restore_cache_position(model):
    def pre(module, args, kwargs):
        if kwargs.get("cache_position") is None:
            past = kwargs["past_key_values"].get_seq_length(module.layer_idx)
            kwargs["cache_position"] = torch.arange(past, past + kwargs["hidden_states"].shape[1])
        return args, kwargs

    return [layer.self_attn.register_forward_pre_hook(pre, with_kwargs=True) for layer in model.model.layers]


def put_rows(z, key, cache, model, ids):
    z[f"{key}/len"] = np.array([la.keys.shape[2] for la in cache.layers], dtype=np.int32)
    for i, p in enumerate(T.kept_positions(cache, T.full_cache(model, ids))):
        z[f"{key}/pos{i}"] = p.numpy().astype(np.int16)


@torch.no_grad()
def main(ref_path):
    ref = import_reference(ref_path)
    z = {}
    mp = pytest.MonkeyPatch()
    from tests import cpu_backend

    cpu_backend.install(mp)          # this package's presses (statistics collection) on the CPU oracle

    for name, ref_cls, _, kw in T.CASES:
        for ratio in T.SAME_ROWS_RATIOS:
            for family in T.FAMILIES:
                model, ids = T._model(family), T.same_rows_ids()
                key = f"same_rows/{name}/{ratio}/{family}"
                cache = ref_prefill(ref_cls(ref)(compression_ratio=ratio, **kw), model, ids)
                put_rows(z, key, cache, model, ids)
                if name == "knorm":
                    for i, la in enumerate(cache.layers):
                        z[f"{key}/norms{i}"] = la.keys.norm(dim=-1).sort(-1).values.numpy()

    for inner in ("streaming", "snapkv"):
        for family in T.FAMILIES:
            model, ids = T._model(family), T._distinct_ids(7)
            _, ref_cls, _, kw = next(c for c in T.CASES if c[0] == inner)
            key = f"rerotation/{inner}/{family}"
            cache = ref_prefill(ref.KeyRerotationPress(ref_cls(ref)(compression_ratio=0.4, **kw)), model, ids)
            put_rows(z, key, cache, model, ids)
            for i, la in enumerate(cache.layers):
                z[f"{key}/ksig{i}"] = T.row_signature(la.keys).numpy()

    from types import SimpleNamespace

    for ratio, beta in T.PYRAMID_CASES:
        model, ids = tiny_llama(layers=4), T._distinct_ids(11)
        press = ref.PyramidKVPress(compression_ratio=ratio, window_size=16, kernel_size=5, beta=beta)
        put_rows(z, f"pyramid/{ratio}/{beta}", ref_prefill(press, model, ids), model, ids)
    z["pyramid_budget_grid"] = np.array([
        ref.PyramidKVPress(compression_ratio=r, window_size=64, beta=b).get_layer_budget(
            SimpleNamespace(config=SimpleNamespace(num_hidden_layers=32), layer_idx=layer), q_len)
        for q_len, r, b, layer in T.PYRAMID_GRID], dtype=np.int64)

    def inner_press(inner, ratio):
        _, ref_cls, _, kw = next(c for c in T.CASES if c[0] == inner)
        if inner == "snapkv":
            kw = {"window_size": 8, "kernel_size": 3}
        return ref_cls(ref)(compression_ratio=ratio, **kw)

    for inner in ("knorm", "snapkv"):
        for n_tokens, chunk in T.CHUNK_CASES:
            model, ids = tiny_llama(), T._distinct_ids(12, n=n_tokens)
            press = ref.ChunkPress(inner_press(inner, 0.5), chunk_length=chunk)
            put_rows(z, f"chunk/{inner}/{n_tokens}/{chunk}", ref_prefill(press, model, ids), model, ids)

    model, ids = tiny_llama(), T._distinct_ids(13)
    rp = ref.ComposedPress([ref.SnapKVPress(0.25, window_size=16), ref.KnormPress(0.4)])
    put_rows(z, "composed", ref_prefill(rp, model, ids), model, ids)
    z["composed/ratio"] = np.array(rp.compression_ratio, dtype=np.float64)
    rp = ref.PerLayerCompressionPress(ref.SnapKVPress(window_size=16), T.per_layer_ratios(model))
    put_rows(z, "per_layer", ref_prefill(rp, model, ids), model, ids)
    z["per_layer/ratio"] = np.array(rp.compression_ratio, dtype=np.float64)

    model, ids = tiny_llama(), T._distinct_ids(14)
    put_rows(z, "random", ref_prefill(ref.RandomPress(0.5, seed=3), model, ids), model, ids)

    for inner in ("expected_attention", "snapkv"):
        for alpha in (0.2, 0.0, 1.0):
            model, ids = tiny_llama(), T._distinct_ids(21)
            _, ref_cls, _, kw = next(c for c in T.CASES if c[0] == inner)
            press = ref.AdaKVPress(ref_cls(ref)(compression_ratio=0.5, **kw), alpha_safeguard=alpha)
            _, masked, step = T.adakv_run(press, model, ids, True)
            key = f"adakv/{inner}/{alpha}"
            for i, m in enumerate(masked):
                z[f"{key}/masked{i}"] = m.numpy().astype(np.int16)
            z[f"{key}/step"] = step.detach().numpy()

    for inner in ("knorm", "snapkv", "expected_attention"):
        for n_tokens, chunk in T.CHUNKKV_CASES:
            if inner != "knorm" and n_tokens < 32:
                continue
            model, ids = tiny_llama(), T._distinct_ids(31, n=n_tokens)
            press = ref.ChunkKVPress(inner_press(inner, 0.4), chunk_length=chunk)
            put_rows(z, f"chunkkv/{inner}/{n_tokens}/{chunk}", ref_prefill(press, model, ids), model, ids)

    for inner in ("knorm", "keydiff"):
        for block_size in (16, 50, 400):
            model, ids = tiny_llama(), T._distinct_ids(32)
            _, ref_cls, _, kw = next(c for c in T.CASES if c[0] == inner)
            press = ref.BlockPress(ref_cls(ref)(compression_ratio=0.5, **kw), block_size=block_size)
            put_rows(z, f"block/{inner}/{block_size}", ref_prefill(press, model, ids), model, ids)

    # statistics: collected by this package, saved, loaded by the reference, saved again by the reference
    from kvpress.presses.expected_attention_with_stats import ExpectedAttentionStats as RefStats

    from kvpress_b200.presses.expected_attention_with_stats import collect_query_statistics

    tmp = Path(tempfile.mkdtemp())
    model = tiny_llama()
    collect_query_statistics(model, T.stats_batches(), n_sink=4).save_pretrained(str(tmp / "ours"))
    RefStats.from_pretrained(str(tmp / "ours")).save_pretrained(str(tmp / "theirs"))
    for name in ("config.json", "model.safetensors"):
        z[f"ea_stats/file/{name}"] = np.frombuffer((tmp / "theirs" / name).read_bytes(), dtype=np.uint8)
    ids = T._distinct_ids(50)
    for use_cov in (True, False):
        rp = ref.ExpectedAttentionStatsPress(compression_ratio=0.5, use_covariance=use_cov, stats_folder=str(tmp / "ours"))
        put_rows(z, f"ea_stats/press/{use_cov}", ref_prefill(rp, model, ids), model, ids)
        z[f"ea_stats/mu/{use_cov}"] = rp.mu.detach().numpy()

    for family in T.FAMILIES:
        model = T._model(family)
        pipe = ref.KVPressTextGenerationPipeline(model=model, tokenizer=word_tokenizer(), device="cpu")
        context, questions = T.pipeline_inputs()
        seen = []
        handles = restore_cache_position(model) + [T.position_spy(model, seen)]
        try:
            out = pipe(context, questions=questions, max_new_tokens=6,
                       press=ref.KeyRerotationPress(ref.StreamingLLMPress(compression_ratio=0.4, n_sink=4)))
        finally:
            for h in handles:
                h.remove()
        key = f"pipeline_rerotation/{family}"
        z[f"{key}/answers"] = np.array(out["answers"])
        z[f"{key}/n_seen"] = np.array(len(seen))
        for j, s in enumerate(seen):
            z[f"{key}/seen{j}"] = np.array(s, dtype=np.int32)

    model = tiny_llama()
    pipe = ref.KVPressTextGenerationPipeline(model=model, tokenizer=word_tokenizer(), device="cpu")
    context, question = T.decoding_inputs()
    skw = dict(stats_folder=str(tmp / "theirs"), n_future_positions=3)
    cache = DynamicCache()
    handles = restore_cache_position(model)
    try:
        out = pipe(context, question=question, max_new_tokens=24,
                   press=ref.DecodingPress(base_press=ref.ExpectedAttentionStatsPress(**skw), **T.DECODING_KW), cache=cache)
    finally:
        for h in handles:
            h.remove()
    z["decoding/answer"] = np.array(out["answer"])
    z["decoding/len"] = np.array([la.keys.shape[2] for la in cache.layers], dtype=np.int32)
    for i, la in enumerate(cache.layers):
        z[f"decoding/sig{i}"] = T._rows_signature(la.keys, la.values).numpy()

    mp.undo()
    np.savez_compressed(OUT, **z)
    print(OUT, len(z), "arrays,", OUT.stat().st_size, "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
