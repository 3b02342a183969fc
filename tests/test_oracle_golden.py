"""The CPU oracle (oracle/press_oracle.py) against the golden vectors produced by the imported
reference (tests/golden/make_golden.py). This is what pins the oracle; the GPU parity tests then
compare the CUDA path against the oracle and against the same golden files."""
import os

import numpy as np
import pytest
import torch

from oracle import press_oracle as O
from tests.conftest import GOLDEN_DIR, REFERENCE_DIR, assert_gemm_prologue, ulp16_diff


def test_knorm_scores_match_reference(golden):
    got = O.knorm_scores(golden.t("keys"))
    assert torch.equal(got, golden.t("knorm_scores"))


def test_streaming_scores_and_kept_sets(golden):
    keys = golden.t("keys")
    for i, r in enumerate(golden.ratios):
        assert torch.equal(O.streaming_scores(keys, r, 4), golden.t(f"streaming_scores_{i}"))
        n_kept = O.kept_count(golden.S, r)
        ref_kept = golden.t(f"streaming_kept_{i}")
        want = O.streaming_kept(golden.S, n_kept, 4).to(torch.int32)
        assert torch.equal(ref_kept, want.expand_as(ref_kept))


def test_snapkv_prologue_and_scores(golden_or_live):
    golden = golden_or_live
    w, ksz = (int(x) for x in golden.z["snap_window"])
    q = O.snapkv_window_queries(golden.t("hidden_states"), golden.t("q_weight"), golden.Hq, golden.D,
                                golden.t("cos"), golden.t("sin"), w)
    # the q_proj GEMM: bit-exact against the live reference, host-GEMM spread against a stored file
    assert_gemm_prologue(q, golden.t("snap_q_window"), golden.live, "snap_q_window")
    # the path proper, from the reference's own window queries: bit-exact on any host
    assert torch.equal(O.snapkv_scores(golden.t("snap_q_window"), golden.t("keys"), w, ksz), golden.t("snap_scores"))
    if golden.live:
        assert torch.equal(O.snapkv_scores(q, golden.t("keys"), w, ksz), golden.t("snap_scores"))


def test_snapkv_fp32_restatement_is_close_to_reference(golden):
    w, ksz = (int(x) for x in golden.z["snap_window"])
    hi = O.snapkv_scores_fp32(golden.t("snap_q_window"), golden.t("keys"), w, ksz)[..., :-w]
    ref = golden.t("snap_scores")[..., :-w].float()
    # the reference rounds to 16 bit at ~7 points; its scores sit within a few 16-bit ulps of fp32 math
    rel = ((hi - ref).abs() / hi.abs().clamp_min(1e-30))
    assert rel.max() < 3e-2 and rel.mean() < 4e-3


def test_expected_attention_stats_and_scores(golden_or_live):
    golden = golden_or_live
    mu, cov = O.expected_attention_stats(golden.t("hidden_states"), golden.t("q_weight"), golden.Hq, golden.D,
                                         golden.t("ea_cos_future"), golden.t("ea_sin_future"), 4)
    assert_gemm_prologue(mu, golden.t("ea_mu"), golden.live, "ea_mu")
    assert_gemm_prologue(cov, golden.t("ea_cov"), golden.live, "ea_cov")
    mu, cov = golden.t("ea_mu"), golden.t("ea_cov")     # the scan, from the reference's own statistics
    k, v = golden.t("keys"), golden.t("values")
    assert torch.equal(O.expected_attention_scores(k, v, mu, cov, 0.0, 4, True), golden.t("ea_scores"))
    assert torch.equal(O.expected_attention_scores(k, v, mu, None, 0.0, 4, False),
                       golden.t("ea_scores_nocov_novnorm"))
    assert torch.equal(O.expected_attention_scores(k, v, mu, cov, 1e-2, 4, True), golden.t("ea_scores_eps"))


def test_kept_sets_match_reference_topk(golden):
    """oracle top-k + gather == the reference's compress() output sets, and the kernels' canonical
    lowest-position tie rule is a VALID answer w.r.t. the reference scores."""
    k, v = golden.t("keys"), golden.t("values")
    score_of = {
        "knorm": golden.t("knorm_scores"),
        "snap": golden.t("snap_scores"),
        "ea": golden.t("ea_scores"),
    }
    for i, r in enumerate(golden.ratios):
        n_kept = O.kept_count(golden.S, r)
        for tag, sc in score_of.items():
            k2, v2, idx = O.compress_with_scores(sc, k, v, n_kept)
            ref = golden.t(f"{tag}_kept_{i}")
            assert torch.equal(idx.sort(-1).values.to(torch.int32), ref), (tag, r)
            assert torch.equal(k2, O.gather_rows(k, idx)) and torch.equal(v2, O.gather_rows(v, idx))
            canon = O.select_lowest_index_ties(sc, n_kept)
            assert O.check_selection(sc, canon, n_kept)["ok"], (tag, r)
            # and the reference's own set passes the same tie-aware check
            assert O.check_selection(sc, ref.long(), n_kept)["ok"]


def test_check_selection_rejects_wrong_sets(golden):
    sc = golden.t("knorm_scores")
    n_kept = golden.S // 2
    canon = O.select_lowest_index_ties(sc, n_kept)
    bad = canon.clone()
    worst = sc.float().argmin(-1)
    bad[..., 0] = worst  # swap in the worst-scoring position
    assert not O.check_selection(sc, bad, n_kept)["ok"]


def test_decoding_ratio_table():
    table = np.load(GOLDEN_DIR / "decoding_ratio.npz")["table"]
    for q_len, target, ratio, kept in table:
        got = O.find_target_compression_ratio(int(q_len), int(target))
        assert got == ratio
        assert O.kept_count(int(q_len), got) == int(kept)


def test_kept_count_float64_arithmetic():
    assert O.kept_count(131072, 0.7) == 39321  # 1 - 0.7 = 0.30000000000000004
    assert O.kept_count(23, 0.4) == 13
    assert O.kept_count(108, 0.5) == 54


def test_ulp_helper():
    a = torch.tensor([1.0, -1.0, 0.0], dtype=torch.bfloat16)
    b = torch.tensor([1.0078125, -1.0078125, -0.0], dtype=torch.bfloat16)
    assert ulp16_diff(a, b).tolist() == [1, 1, 0]


# ---- KeyRerotationPress (SURVEY §8f row 1) ------------------------------------------------------------
def _rerotation_cases():
    z = np.load(GOLDEN_DIR / "rerotation.npz")
    for tag, (B, H, S, D, is_half) in zip("abc", z["cases"]):
        dtype = torch.float16 if is_half else torch.bfloat16
        get = lambda k, tag=tag, dtype=dtype: (  # noqa: E731
            torch.from_numpy(z[f"{tag}_{k}"].copy()).view(dtype) if z[f"{tag}_{k}"].dtype == np.uint16
            else torch.from_numpy(z[f"{tag}_{k}"].copy()))
        yield tag, int(S), [float(r) for r in z["ratios"]], get


def test_rerotation_matches_reference_bit_exact():
    """The oracle's rerotate_keys / key_rerotation_compress against KeyRerotationPress.compress outputs."""
    for tag, S, ratios, get in _rerotation_cases():
        keys, values, inv_freq, scores = get("keys"), get("values"), get("inv_freq"), get("scores")
        for i, r in enumerate(ratios):
            n_kept = O.kept_count(S, r)
            k2, v2, idx = O.key_rerotation_compress(scores, keys, values, n_kept, inv_freq)
            assert torch.equal(k2.view(torch.int16), get(f"perm_k_{i}").view(torch.int16)), (tag, r)
            if i == 0:
                assert torch.equal(v2, get("perm_v_0"))
            # canonical (lowest-index ties) selection coincides when scores are distinct
            assert torch.equal(O.select_lowest_index_ties(scores, n_kept), idx)
            kn_idx = get(f"knorm_idx_{i}").long()
            k3 = O.rerotate_keys(keys, kn_idx, inv_freq)
            assert torch.equal(k3.view(torch.int16), get(f"knorm_k_{i}").view(torch.int16)), (tag, r)


# ---- KeyDiffPress (SURVEY §8f row 3) --------------------------------------------------------------------
def _keydiff_cases():
    z = np.load(GOLDEN_DIR / "keydiff.npz")
    for tag, (B, H, S, D, is_half) in zip("abc", z["cases"]):
        dtype = torch.float16 if is_half else torch.bfloat16
        yield (tag, torch.from_numpy(z[f"{tag}_keys"].copy()).view(dtype),
               torch.from_numpy(z[f"{tag}_scores"].copy()).view(dtype))


def test_keydiff_oracle_matches_reference_and_its_fp32_form():
    for tag, keys, ref_scores in _keydiff_cases():
        got = O.keydiff_scores(keys)
        assert torch.equal(got.view(torch.int16), ref_scores.view(torch.int16)), tag
        # the fp32 evaluation (what the kernel rounds once) stays within a few 16-bit ulps of the reference,
        # which rounds after each of its ~6 ATen ops
        hi = O.keydiff_scores_fp32(keys).to(keys.dtype)
        d = ulp16_diff(hi, ref_scores)
        near_zero = ref_scores.float().abs() < 2.0 ** -6      # ulps are meaningless around a sign change
        assert d[~near_zero].max().item() <= 8 and (d[~near_zero] <= 2).float().mean().item() > 0.97, tag
        if near_zero.any():
            assert (hi.float() - ref_scores.float()).abs()[near_zero].max().item() < 2.0 ** -8


@pytest.mark.parametrize("live", [False, True], ids=["stored", "live"])
def test_large32k_oracle_matches_reference(live):
    """S = 32768 (tests/golden/large32k.npz; inputs regenerated from the seed): the oracle restatements of Knorm, the
    SnapKV / TOVA window attention, the ExpectedAttention prologue and scan are bit-exact at a long context too.
    `live` regenerates the arrays with the imported reference on this host (build container only): everything is
    bit-exact there. Against the STORED file the stages downstream of a q_proj GEMM recomputed on this host may carry
    another host's GEMM rounding (q is not stored at this size): bit-exact or <= 1 ulp on >= 99 % equal elements."""
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding

    from tests.golden.make_golden import build_large, large_inputs, tensor_checksum

    if live:
        if not os.path.isdir(REFERENCE_DIR):
            pytest.skip("no /root/reference here: live pinning runs in the build container only")
        z = build_large()
    else:
        z = np.load(GOLDEN_DIR / "large32k.npz")

    def after_q_proj(got, want, what):
        if torch.equal(got, want):
            return
        assert not live, f"{what}: differs from the reference run live on this host"
        d = ulp16_diff(got, want)
        assert d.max().item() <= 1 and (d == 0).float().mean().item() >= 0.99, what
    B, Hq, Hkv, D, hidden, S, seed = (int(x) for x in z["meta"])
    h, k, v = large_inputs(seed, B, Hkv, S, D, hidden)
    assert (tensor_checksum(h, k, v) == z["checksum"]).all(), "torch CPU RNG no longer reproduces the seeded inputs"

    def t(name):
        return torch.from_numpy(z[name].copy()).view(torch.bfloat16)

    cfg = LlamaConfig(hidden_size=hidden, num_attention_heads=Hq, num_key_value_heads=Hkv, head_dim=D,
                      max_position_embeddings=65536, rope_theta=500000.0)
    rot = LlamaRotaryEmbedding(cfg)
    cos, sin = rot(h, torch.arange(S)[None])
    qw = t("q_weight")
    assert torch.equal(O.knorm_scores(k), t("knorm_scores"))
    q_last = O.snapkv_window_queries(h, qw, Hq, D, cos, sin, 1)[:, :, 0]
    after_q_proj(O.tova_scores(q_last, k), t("tova_scores"), "tova_scores")
    q_win = O.snapkv_window_queries(h, qw, Hq, D, cos, sin, 64)
    after_q_proj(O.snapkv_scores(q_win, k, 64, 5), t("snap_scores"), "snap_scores")
    cf, sf = rot(h, torch.arange(S, S + 512)[None])
    mu, cov = O.expected_attention_stats(h, qw, Hq, D, cf[0], sf[0], 4)
    assert_gemm_prologue(mu, t("ea_mu"), live, "ea_mu")
    assert_gemm_prologue(cov, t("ea_cov"), live, "ea_cov")
    assert torch.equal(O.expected_attention_scores(k, v, t("ea_mu"), t("ea_cov"), 0.0, 4, True), t("ea_scores"))
    for i, r in enumerate(z["ratios"]):
        n_kept = O.kept_count(S, float(r))
        for tag in ("knorm", "snap", "ea", "tova"):
            kept = torch.from_numpy(z[f"{tag}_kept_{i}"].copy())
            assert O.check_selection(t(f"{tag}_scores"), kept, n_kept)["ok"]
