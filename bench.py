#!/usr/bin/env python
"""bench.py — throughput of the fused score -> top-k -> gather path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--no-extras]
                    [--dump-outputs DIR]

A "step" is one ScorerPress.compress call on one layer's synthetic cache [B, Hkv, S, D] (bf16).
Prints ONE JSON line on rank 0:
  value        tokens scored+compacted per second, whole job (all ranks), inputs resident in HBM. The step is the
               C-ABI call (kvp_*_compress) captured once into a CUDA graph per input set and replayed
               (kvpress_b200.native.GraphedCall): the same kernels, one host launch per step, so the number is
               GPU-bound on any host. `eager` reports the same call issued directly (no graph) beside it, and
               `host_us_per_call` the host time either way costs.
  e2e          the same metric through the package's public host-buffer API
               (kvpress_b200.host_staging.compress_host): pinned HOST K/V copied in, compacted K'/V' copied back,
               copies inside the timed region
  roofline     algorithmic bytes of one compress call / its CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline the reference's own ScorerPress.compress (oracle/_ref, unmodified) — or, when that copy was not
               built, the oracle port of its ATen sequence — on the host cores
  extras       (same process, after the headline; device-timed the same way) the other BASELINE.json configs:
               configs[1] snapkv_32k, configs[3] the DecodingPress loop, configs[4] the 80-layer Llama-3.1-70B SnapKV
               prefill with layers pipeline-split over the ranks, the EA call including its prologue, knorm_128k.
Multi-GPU: the path has no exchange step; ranks process independent batch shards (weak scaling) — or, for
configs[4], disjoint layer ranges — and NCCL is used only for the barrier and the max-over-ranks of the timings.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

L2_BYTES = 126 * 1024 * 1024

# name -> workload description. `config_index` refers to BASELINE.json "configs".
WORKLOADS = {
    # BASELINE.json configs[2]: the 128k single-GPU configuration the metric is quoted on
    "ea_128k": dict(scorer="expected_attention", B=1, Hkv=8, Hq=32, S=131072, D=128, ratio=0.7, config_index=2,
                    label="ExpectedAttentionPress r=0.7, Llama-3.1-8B layer shape, 128k ctx"),
    # BASELINE.json configs[1]
    "snapkv_32k": dict(scorer="snapkv", B=1, Hkv=8, Hq=32, S=32768, D=128, ratio=0.5, config_index=1,
                       label="SnapKVPress r=0.5, Llama-3.1-8B layer shape, 32k ctx"),
    # per-layer shape of configs[4] (70B: Hq=64)
    "snapkv_128k_70b": dict(scorer="snapkv", B=1, Hkv=8, Hq=64, S=131072, D=128, ratio=0.5, config_index=4,
                            label="SnapKVPress r=0.5, Llama-3.1-70B layer shape, 128k ctx"),
    "knorm_128k": dict(scorer="knorm", B=1, Hkv=8, Hq=8, S=131072, D=128, ratio=0.5, config_index=None,
                       label="KnormPress r=0.5, Llama-3.1-8B layer shape, 128k ctx"),
    # SURVEY §8f row 1: KeyRerotationPress(KnormPress): score + select + compaction with re-rotated keys
    "rerotate_knorm_128k": dict(scorer="knorm_rerotate", B=1, Hkv=8, Hq=8, S=131072, D=128, ratio=0.5,
                                config_index=None, label="KeyRerotationPress(KnormPress) r=0.5, 128k ctx"),
    # SURVEY §8f row 2: AdaKVPress(ExpectedAttentionPress): EA scores, then the two head-wise selections (no compaction)
    "adakv_ea_128k": dict(scorer="adakv_ea", B=1, Hkv=8, Hq=32, S=131072, D=128, ratio=0.7, config_index=None,
                          label="AdaKVPress(ExpectedAttentionPress) r=0.7 head-wise selection, 128k ctx"),
    # SURVEY §8f row 3: KeyDiffPress (two streaming passes over K, then select + compact)
    "keydiff_128k": dict(scorer="keydiff", B=1, Hkv=8, Hq=8, S=131072, D=128, ratio=0.5, config_index=None,
                         label="KeyDiffPress r=0.5, Llama-3.1-8B layer shape, 128k ctx"),
    "streaming_128k": dict(scorer="streaming", B=1, Hkv=8, Hq=8, S=131072, D=128, ratio=0.5, config_index=None,
                           label="StreamingLLMPress r=0.5, 128k ctx"),
    # steady state of configs[3]: DecodingPress(Knorm, 512, 2048) compaction 2560 -> 2048
    "decoding_knorm": dict(scorer="knorm", B=1, Hkv=8, Hq=8, S=2560, D=128, ratio=None, n_kept=2048,
                           config_index=3, label="DecodingPress(Knorm) steady-state compaction 2560->2048"),
}
DEFAULT_WORKLOAD = "ea_128k"


def kept_count(S: int, ratio: float) -> int:
    return int(S * (1 - ratio))


def algorithmic_bytes(w: dict, n_kept: int) -> int:
    """SURVEY §8(d): every input byte read once + every output byte written once, per (b, kv-head)."""
    row = w["D"] * 2
    S = w["S"]
    per_head = {
        "knorm": row * (S + 3 * n_kept),
        "knorm_rerotate": row * (S + 3 * n_kept),
        "keydiff": row * (2 * S + 3 * n_kept),  # the anchor needs all of K before any score: K is read twice
        "adakv_ea": row * 2 * S,  # read all K and all V once; the output is index triples only
        "snapkv": row * (S + 3 * n_kept),
        "expected_attention": row * (2 * S + 2 * n_kept),
        "streaming": row * 4 * n_kept,
    }[w["scorer"]]
    return per_head * w["B"] * w["Hkv"]


def algorithmic_flops(w: dict) -> float:
    """SURVEY §8(d): dense FLOPs of the tensor-core score stage (0 for the streaming scorers)."""
    B, Hq, S, D = w["B"], w["Hq"], w["S"], w["D"]
    if w["scorer"] == "expected_attention":
        return float(B * Hq * S * (2 * D * D + 4 * D))
    if w["scorer"] == "snapkv":
        return float(2 * 2 * 64 * B * Hq * S * D)  # two exact-softmax passes of 2*w*Hq*S*D
    return 0.0


def mufu_bound_us(w: dict) -> float:
    """SnapKV's exact softmax costs two exponentials per (window query, key): pass 1 for the normalisers, pass 2 for the
    normalised column sums. MUFU.EX2 issues 16 per clock per SM; packed f16x2 / bf16x2 forms compile to two MUFU ops on
    sm_100a, so this is a hard floor of the exact two-pass algorithm: 2 * w * Hq * S exps / (16 * 148 SMs * 1.965 GHz)."""
    if w["scorer"] != "snapkv":
        return 0.0
    return 2.0 * 64 * w["B"] * w["Hq"] * w["S"] / (16.0 * 148 * 1.965e9) * 1e6


def load_traffic(workload: str):
    """DRAM bytes one compress call moves (sum over its kernels, dram__bytes_read + write per launch) from the
    committed ncu launch list of the same command: profiles/traffic.json, written by tools/ncu_launches.py."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        return json.loads(p.read_text()).get(workload)
    return None


def load_peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d.get("bf16_tflops", 1590.0)),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", 1400.0)),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


# --------------------------------------------------------------------------------------------------
# synthetic inputs
# --------------------------------------------------------------------------------------------------
def make_inputs(w: dict, device, seed: int, pinned_host: bool = False):
    """K, V ~ N(0,1) bf16 [B,Hkv,S,D] (+ scorer-specific small operands), seeded per rank."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    B, H, Hq, S, D = w["B"], w["Hkv"], w["Hq"], w["S"], w["D"]
    if device != "cpu" and not pinned_host:
        gd = torch.Generator(device=device).manual_seed(seed)
        K = torch.randn((B, H, S, D), generator=gd, device=device, dtype=torch.float32).to(torch.bfloat16)
        V = torch.randn((B, H, S, D), generator=gd, device=device, dtype=torch.float32).to(torch.bfloat16)
    else:
        K = torch.randn((B, H, S, D), generator=g, dtype=torch.float32).to(torch.bfloat16)
        V = torch.randn((B, H, S, D), generator=g, dtype=torch.float32).to(torch.bfloat16)
        if pinned_host:
            K, V = K.pin_memory(), V.pin_memory()
    extra = {}
    if w["scorer"] == "knorm_rerotate":
        extra["inv_freq"] = 1.0 / (500000.0 ** (torch.arange(0, D, 2).float() / D))  # Llama-3 rope_theta
    if w["scorer"] == "snapkv":
        extra["q_window"] = torch.randn((B, Hq, 64, D), generator=g, dtype=torch.float32).to(torch.bfloat16)
    if w["scorer"] in ("expected_attention", "adakv_ea"):
        extra["mu"] = (0.5 * torch.randn((B, Hq, D), generator=g)).to(torch.bfloat16)
        a = torch.randn((B, Hq, D, D), generator=g) / D ** 0.5
        extra["cov"] = (a @ a.transpose(-1, -2)).to(torch.bfloat16)  # PSD like a real covariance
    if device != "cpu":
        extra = {k: v.to(device) for k, v in extra.items()}
    return K, V, extra


def run_native(w: dict, K, V, extra, n_kept: int):
    from kvpress_b200 import native

    s = w["scorer"]
    if s == "knorm":
        return native.knorm_compress(K, V, n_kept)[:2]
    if s == "keydiff":
        return native.keydiff_compress(K, V, n_kept)[:2]
    if s == "knorm_rerotate":
        return native.scores_compress_rerotate(native.knorm_score(K), K, V, n_kept, extra["inv_freq"])[:2]
    if s == "adakv_ea":
        sc = native.expected_attention_score(K, V, extra["mu"], extra["cov"], 1e-2, 4, True)
        n_safe = int(n_kept * 0.2)
        sc = sc.scatter(-1, native.scores_select(sc, n_safe).long(), torch.finfo(sc.dtype).max)
        H, S = sc.shape[1], sc.shape[2]
        return native.scores_select((-sc).reshape(sc.shape[0], 1, H * S), H * (S - n_kept)), None
    if s == "streaming":
        return native.streaming_compress(K, V, n_kept, 4)[:2]
    if s == "snapkv":
        return native.snapkv_compress(K, V, extra["q_window"], 64, 5, n_kept)[:2]
    if s == "expected_attention":
        return native.expected_attention_compress(K, V, extra["mu"], extra["cov"], 0.0, 4, True, n_kept)[:2]
    raise ValueError(s)


def run_oracle(w: dict, K, V, extra, ratio: float):
    from oracle import press_oracle as O

    s = w["scorer"]
    if s == "knorm":
        return O.knorm_compress(K, V, ratio)
    if s == "keydiff":
        n_kept = O.kept_count(K.shape[2], ratio)
        idx = O.topk_indices(O.keydiff_scores(K), n_kept)
        return O.gather_rows(K, idx), O.gather_rows(V, idx)
    if s == "knorm_rerotate":
        n_kept = O.kept_count(K.shape[2], ratio)
        return O.key_rerotation_compress(O.knorm_scores(K), K, V, n_kept, extra["inv_freq"])[:2]
    if s == "adakv_ea":
        sc = O.expected_attention_scores(K, V, extra["mu"], extra["cov"], 1e-2, 4, True)
        n_kept = O.kept_count(K.shape[2], ratio)
        sc = sc.scatter(-1, sc.topk(int(n_kept * 0.2), dim=-1).indices, torch.finfo(sc.dtype).max)
        H, S = sc.shape[1], sc.shape[2]
        return torch.topk(-sc.reshape(sc.shape[0], -1), H * (S - n_kept), dim=1).indices, None
    if s == "streaming":
        return O.streaming_compress(K, V, ratio, 4)
    if s == "snapkv":
        return O.snapkv_compress(extra["q_window"], K, V, ratio, 64, 5)
    if s == "expected_attention":
        return O.expected_attention_compress(K, V, extra["mu"], extra["cov"], ratio)
    raise ValueError(s)


def effective_ratio(w: dict) -> float:
    if w.get("ratio") is not None:
        return w["ratio"]
    from oracle import press_oracle as O

    return O.find_target_compression_ratio(w["S"], w["n_kept"])


# --------------------------------------------------------------------------------------------------
# the UNMODIFIED reference on the host cores (oracle/_ref, built by oracle/build_ref.py)
# --------------------------------------------------------------------------------------------------
def make_reference_runner(w: dict):
    """Returns run(K, V, extra, ratio) that calls the reference's own `press.compress(...)` — ScorerPress.compress
    (scorer_press.py:76-102) with the scorer's own score() — on CPU tensors, or None if oracle/_ref was not built
    or this workload has no single reference press. The workload's config hands the scorer its small operands
    ((mu, Sigma) for ExpectedAttention, RoPE'd window queries for SnapKV) instead of hidden states, exactly like
    the B200 arm; the reference classes are only told where to take them from:
      * ExpectedAttention: a subclass overrides get_query_statistics (the prologue, :62-124) to return them;
      * SnapKV: the window queries travel as `hidden_states[:, -w:]` through an identity q_proj and identity RoPE
        (cos = 1, sin = 0), so compute_window_attention (:41-69) runs unmodified on them."""
    from oracle.build_ref import import_ref

    ref = import_ref()
    if ref is None:
        return None
    from types import SimpleNamespace

    s, D, Hq, Hkv = w["scorer"], w["D"], w["Hq"], w["Hkv"]
    module = SimpleNamespace(head_dim=D, layer_idx=0,
                             config=SimpleNamespace(num_attention_heads=Hq, num_key_value_heads=Hkv))
    if s == "knorm":
        def run(K, V, extra, ratio):
            return ref.KnormPress(compression_ratio=ratio).compress(module, None, K, V, None, {})
    elif s == "streaming":
        def run(K, V, extra, ratio):
            return ref.StreamingLLMPress(compression_ratio=ratio, n_sink=4).compress(module, None, K, V, None, {})
    elif s == "keydiff":
        def run(K, V, extra, ratio):
            return ref.KeyDiffPress(compression_ratio=ratio).compress(module, None, K, V, None, {})
    elif s == "expected_attention":
        class GivenStats(ref.ExpectedAttentionPress):
            stats = None

            def get_query_statistics(self, module, hidden_states):
                return self.stats

        def run(K, V, extra, ratio):
            press = GivenStats(compression_ratio=ratio, n_sink=4, use_covariance=True, use_vnorm=True, epsilon=0.0)
            press.stats = (extra["mu"], extra["cov"])
            return press.compress(module, K[:, 0, :, :1], K, V, None, {})
    elif s == "snapkv":
        module.q_proj = torch.nn.Identity()
        built = {}

        def run(K, V, extra, ratio):
            q = extra["q_window"]                                   # [B, Hq, w, D] -> rows [S-w, S) of [B, S, Hq*D]
            B, _, wlen, _ = q.shape
            S = K.shape[2]
            if built.get("key") != (q.data_ptr(), S):               # built once, outside the steady-state steps
                hidden = torch.zeros((B, S, Hq * D), dtype=q.dtype)
                hidden[:, S - wlen:] = q.transpose(1, 2).reshape(B, wlen, Hq * D)
                built.update(key=(q.data_ptr(), S), hidden=hidden,
                             pe=(torch.ones((1, S, D), dtype=q.dtype), torch.zeros((1, S, D), dtype=q.dtype)))
            press = ref.SnapKVPress(compression_ratio=ratio, window_size=wlen, kernel_size=5)
            return press.compress(module, built["hidden"], K, V, None, {"position_embeddings": built["pe"]})
    else:
        return None
    return run


# --------------------------------------------------------------------------------------------------
# clocks sampler (pynvml; nvidia-smi columns of B200_PROFILING.md)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {
        0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
        0x80: "hw_power_brake_slowdown",
    }

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:  # no NVML: report nulls rather than fail the bench
            self._nv = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def __enter__(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self) -> dict:
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# --------------------------------------------------------------------------------------------------
# CPU arm
# --------------------------------------------------------------------------------------------------
def cpu_sample_size(w: dict, per_step_budget_s: float) -> int:
    """S of the bounded sample: shrunk (power of two) until one CPU call is expected to fit the per-step budget.
    Rough cost model: ms per 1k tokens on a many-core host, from round-1 measurements of both arms."""
    per_k = {"knorm": 1.2, "keydiff": 3.0, "knorm_rerotate": 3.0, "adakv_ea": 25.0, "streaming": 1.2, "snapkv": 8.0,
             "expected_attention": 25.0}[w["scorer"]]
    S = w["S"]
    while S > 4096 and per_k * S / 1000 / 1000 > per_step_budget_s:
        S //= 2
    return S


def cpu_arm(w: dict, warmup: int, steps: int, per_step_budget_s: float):
    """Times the CPU implementation of the path on a bounded sample of the workload: `warmup` untimed + exactly
    `steps` timed calls, each on the same [B, Hkv, S_sample, D] cache. Returns a dict for the JSON line."""
    torch.set_num_threads(os.cpu_count() or 1)
    ratio = effective_ratio(w)
    S = cpu_sample_size(w, per_step_budget_s)
    ws = dict(w, S=S)
    K, V, extra = make_inputs(ws, "cpu", 1234)
    runner = make_reference_runner(w)
    kind = "reference" if runner is not None else "port"
    if runner is None:
        def runner(K, V, extra, ratio):
            return run_oracle(ws, K, V, extra, ratio)
    with torch.no_grad():
        for _ in range(max(warmup, 1)):
            runner(K, V, extra, ratio)
        t0 = time.perf_counter()
        for _ in range(steps):
            runner(K, V, extra, ratio)
        secs = (time.perf_counter() - t0) / steps
    what = ("the reference's own ScorerPress.compress (oracle/_ref, unmodified)" if kind == "reference"
            else "oracle port of the reference's ATen sequence")
    sample = (f"{what}: {w['scorer']} compress on [B={ws['B']},Hkv={ws['Hkv']},S={S},D={ws['D']}] bf16 "
              f"(workload S={w['S']}), mean of {steps} calls after {max(warmup, 1)} warm-up")
    return {"value": ws["B"] * S / secs, "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": sample, "seconds_per_call": secs, "steps": steps}


# --------------------------------------------------------------------------------------------------
# multi-rank bookkeeping (no data-path collective: ranks own disjoint batch shards)
# --------------------------------------------------------------------------------------------------
def rank_seed(rank: int, i: int = 0) -> int:
    """Every rank synthesises its own shard; seeds never collide across ranks / input sets."""
    return 1234 + 1000 * rank + i


def max_over_ranks(ms_local: float, dist, device) -> float:
    """The step time of the job is the slowest rank's device time."""
    t = torch.tensor([ms_local], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def whole_job_tokens_per_s(tokens_per_rank_step: int, world: int, ms_per_step: float) -> float:
    """Weak scaling: every rank processes tokens_per_rank_step per step; value is the job aggregate."""
    return tokens_per_rank_step * world / (ms_per_step * 1e-3)


def layer_range(n_layers: int, world: int, rank: int) -> range:
    """configs[4]: contiguous layer ownership the way device_map="auto" places a pipeline-split model."""
    per = -(-n_layers // world)
    return range(min(rank * per, n_layers), min((rank + 1) * per, n_layers))


def bind_to_gpu_numa(local_rank: int):
    """Pin this rank (and therefore its pinned-host allocations, first touch) to the CPUs NVML reports as local to
    its GPU. Without it half of the ranks of an 8-GPU box stage their 700 MB/step through the far socket."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * i + b for i, word in enumerate(mask) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": len(cpus), "first": min(cpus)}
    except Exception as ex:  # binding is an optimisation, never a requirement
        return {"error": repr(ex)[:120]}
    return None


def timed_loop(calls, steps: int):
    """`steps` back-to-back calls (calls[i % len]) bracketed by CUDA events on the current stream. Returns
    (device ms per step, host us per call spent enqueueing, what the last call returned)."""
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = len(calls)
    last = None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    start.record()
    for i in range(steps):
        last = calls[i % n]()
    stop.record()
    host_us = (time.perf_counter() - t0) / steps * 1e6
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / steps, host_us, last


DUMP_BUDGET_BYTES = 60 << 20      # under 64 MB in all, .npy headers included


def dump_outputs(out_dir: str, w: dict, outputs) -> dict:
    """Writes what one timed call returned as <out_dir>/<name>.npy: the compacted keys / values as float32, or (AdaKV)
    the pruned flat indices as float64, which holds them exactly. An array above its share of DUMP_BUDGET_BYTES is cut
    to a fixed sample of its rows (last axis kept whole): the first rows of a seeded permutation, in ascending order,
    so that two builds given the same arguments write the same rows. Returns {name: what was written}."""
    import numpy as np

    names = ("pruned_indices",) if w["scorer"] == "adakv_ea" else ("keys", "values")
    arrays = {n: t for n, t in zip(names, outputs) if t is not None}
    budget = DUMP_BUDGET_BYTES // len(arrays)
    os.makedirs(out_dir, exist_ok=True)
    written = {}
    for name, t in arrays.items():
        t = t.detach().to("cpu", torch.float64 if name == "pruned_indices" else torch.float32)
        rows = t.reshape(-1, t.shape[-1])
        n_rows = max(1, budget // (rows.shape[1] * rows.element_size()))
        sampled = n_rows < rows.shape[0]
        if sampled:
            pick = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:n_rows].sort().values
            t = rows[pick]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy())
        written[name] = {"shape": list(t.shape), "dtype": str(t.dtype).replace("torch.", ""),
                         "sampled_rows_of": list(rows.shape) if sampled else None}
    return written


# --------------------------------------------------------------------------------------------------
# extras: the other BASELINE.json configs, device-timed in the same process
# --------------------------------------------------------------------------------------------------
def extra_workload(name: str, device, rank: int, steps: int, peaks: dict) -> dict:
    from kvpress_b200 import native

    w = WORKLOADS[name]
    ratio = effective_ratio(w)
    n_kept = w.get("n_kept") or kept_count(w["S"], ratio)
    bytes_per_set = 2 * w["B"] * w["Hkv"] * w["S"] * w["D"] * 2
    n_sets = max(1, min(8, -(-4 * L2_BYTES // bytes_per_set)))
    sets = [make_inputs(w, device, rank_seed(rank, 50 + i)) for i in range(n_sets)]
    graphs = [native.capture(lambda s=s: run_native(w, s[0], s[1], s[2], n_kept)) for s in sets]
    calls = [g.replay for g in graphs]
    timed_loop(calls, 3)
    ms, host_us, _ = timed_loop(calls, steps)
    eager = [lambda s=s: run_native(w, s[0], s[1], s[2], n_kept) for s in sets]
    timed_loop(eager, 3)
    ms_e, host_e, _ = timed_loop(eager, steps)
    abytes = algorithmic_bytes(w, n_kept)
    out = {"workload": name, "baseline_config_index": w["config_index"], "description": w["label"],
           "us_per_step": ms * 1e3, "tokens_per_s": w["B"] * w["S"] / (ms * 1e-3), "steps": steps,
           "host_us_per_call": host_us, "eager_us_per_step": ms_e * 1e3, "eager_host_us_per_call": host_e,
           "algorithmic_bytes": abytes, "achieved_gbs": abytes / (ms * 1e-3) / 1e9,
           "frac_of_hbm_peak": abytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "n_input_sets": n_sets}
    flops = algorithmic_flops(w)
    if flops:
        out["tensor_bound_us"] = flops / (peaks["bf16_tflops_sustained"] * 1e12) * 1e6
        out["hbm_bound_us"] = abytes / (peaks["hbm_gbs"] * 1e9) * 1e6
    if mufu_bound_us(w):
        out["mufu_bound_us"] = mufu_bound_us(w)
        out["frac_of_binding_roof"] = max(out.get("hbm_bound_us", 0.0), out.get("tensor_bound_us", 0.0),
                                          out["mufu_bound_us"]) / (ms * 1e3)
    del graphs, sets
    torch.cuda.empty_cache()
    return out


def extra_layer_split(device, rank: int, world: int, dist, steps: int, n_layers: int, peaks: dict) -> dict:
    """BASELINE.json configs[4]: SnapKVPress r=0.5 on Llama-3.1-70B (80 layers, Hq 64, Hkv 8, D 128) at 128k, layers
    pipeline-split over the ranks like device_map="auto" (README.md:213-220, evaluate.py:393-394): rank r owns a
    contiguous range and compresses each of its layers' caches where they live; nothing crosses NVLink. One step =
    one prefill's worth of compress calls (every layer once). Strong scaling: the 80 layers are fixed."""
    from kvpress_b200 import native

    w = WORKLOADS["snapkv_128k_70b"]
    n_kept = kept_count(w["S"], w["ratio"])
    mine = layer_range(n_layers, world, rank)
    layers = [make_inputs(w, device, rank_seed(rank, 100 + i)) for i in mine]   # every layer has its own cache

    def prefill_pass():
        for K, V, extra in layers:
            run_native(w, K, V, extra, n_kept)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    g = native.capture(prefill_pass) if layers else None
    call = g.replay if g is not None else (lambda: None)
    for _ in range(2):
        call()
    barrier()
    ms, host_us, _ = timed_loop([call], steps)
    barrier()
    ms = max_over_ranks(ms, dist, device)
    abytes = algorithmic_bytes(w, n_kept) * len(mine)
    out = {"workload": "snapkv_128k_70b_layer_split", "baseline_config_index": 4,
           "description": f"SnapKVPress r=0.5, Llama-3.1-70B, 128k ctx, {n_layers} layers pipeline-split over {world} rank(s)",
           "n_layers": n_layers, "layers_per_rank": len(layer_range(n_layers, world, 0)), "steps": steps,
           "ms_per_prefill_pass": ms, "us_per_layer": ms * 1e3 / max(1, len(layer_range(n_layers, world, 0))),
           "tokens_per_s": w["S"] * n_layers / (ms * 1e-3), "scaling": "strong (fixed 80 layers)",
           "host_us_per_pass": host_us,
           "frac_of_hbm_peak_rank0": (abytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if abytes else None,
           "collective": "none in the data path (barrier + MAX all-reduce of the timings)"}
    del g, layers
    torch.cuda.empty_cache()
    return out


def extra_ea_with_prologue(device, rank: int, steps: int) -> dict:
    """SURVEY H4: ExpectedAttentionPress.compress end to end INCLUDING its prologue (expected_attention_press.py:
    62-124): q_proj over the whole 128k prompt (4.4 TFLOP), query mean / covariance (137 GFLOP), average RoPE —
    torch / cuBLAS on the host side of the boundary — then the fused scan. Llama-3.1-8B layer, random-init q_proj."""
    from types import SimpleNamespace

    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding

    from kvpress_b200 import ExpectedAttentionPress

    w = WORKLOADS["ea_128k"]
    S, D, Hq, Hkv, hidden = w["S"], w["D"], w["Hq"], w["Hkv"], 4096
    K, V, _ = make_inputs(w, device, rank_seed(rank, 70))
    gd = torch.Generator(device=device).manual_seed(7)
    h = torch.randn((1, S, hidden), generator=gd, device=device, dtype=torch.float32).to(torch.bfloat16)
    cfg = LlamaConfig(hidden_size=hidden, num_attention_heads=Hq, num_key_value_heads=Hkv, head_dim=D,
                      max_position_embeddings=S + 1024, rope_theta=500000.0)
    q_proj = torch.nn.Linear(hidden, Hq * D, bias=False, device=device, dtype=torch.bfloat16)
    torch.nn.init.normal_(q_proj.weight, std=0.02, generator=gd)
    module = SimpleNamespace(head_dim=D, layer_idx=0, config=cfg, q_proj=q_proj,
                             rotary_emb=LlamaRotaryEmbedding(cfg).to(device))
    press = ExpectedAttentionPress(compression_ratio=w["ratio"])
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    with torch.no_grad():
        for _ in range(2):
            press.compress(module, h, K, V, None, {})
        torch.cuda.synchronize()
        t_stats = t_total = 0.0
        for _ in range(steps):
            ev[0].record()
            press.get_query_statistics(module, h)
            ev[1].record()
            press.compress(module, h, K, V, None, {})
            ev[2].record()
            torch.cuda.synchronize()
            t_stats += ev[0].elapsed_time(ev[1])
            t_total += ev[1].elapsed_time(ev[2])
    ms_total, ms_stats = t_total / steps, t_stats / steps
    flops = 2.0 * (S - 4) * hidden * Hq * D + 2.0 * Hq * (S - 4) * D * D
    del h, K, V
    torch.cuda.empty_cache()
    return {"workload": "ea_128k_with_prologue", "baseline_config_index": 2,
            "description": "ExpectedAttentionPress.compress(module, hidden_states, K, V) incl. q_proj + (mu, Sigma) + avg RoPE",
            "ms_per_call": ms_total, "prologue_ms": ms_stats, "scan_ms": ms_total - ms_stats, "steps": steps,
            "tokens_per_s": S / (ms_total * 1e-3), "prologue_tflops": flops / (ms_stats * 1e-3) / 1e12,
            "prologue_share": ms_stats / ms_total}


def extra_decoding_loop(device, steps_tokens: int, prompt: int = 4096, n_layers: int = 36) -> dict:
    """BASELINE.json configs[3]: DecodingPress(KnormPress, interval 512, target 2048) on Qwen3-8B cache shapes
    (36 layers, Hkv 8, D 128): a 4k prompt, then `steps_tokens` generated tokens. The model's own forward is not the
    path under test: every generated token appends one (k, v) row to each layer's DynamicCache (what attention does)
    and fires the press's forward hook for that layer (decoding_press.py:113-179). Reports the hook cost per layer
    per token when no compaction fires, and the compaction calls."""
    from types import SimpleNamespace

    from transformers import DynamicCache

    from kvpress_b200 import DecodingPress, KnormPress

    Hkv, D, hidden = 8, 128, 4096
    press = DecodingPress(base_press=KnormPress(), compression_interval=512, target_size=2048)
    cache = DynamicCache()
    gd = torch.Generator(device=device).manual_seed(11)
    modules = [SimpleNamespace(layer_idx=i, head_dim=D) for i in range(n_layers)]
    for i in range(n_layers):  # the prefilled prompt
        k = torch.randn((1, Hkv, prompt, D), generator=gd, device=device, dtype=torch.float32).to(torch.bfloat16)
        cache.update(k, k.flip(2), i)
    new_k = torch.randn((1, Hkv, 1, D), generator=gd, device=device, dtype=torch.float32).to(torch.bfloat16)
    hs = torch.zeros((1, 1, hidden), device=device, dtype=torch.bfloat16)
    kwargs = {"hidden_states": hs, "past_key_values": cache}
    out = (None, None)
    hook_s, compact_host_s, n_compact, n_plain = 0.0, 0.0, 0, 0
    comp_ev = []
    torch.cuda.synchronize()
    t_loop = time.perf_counter()
    for t in range(steps_tokens):
        for i in range(n_layers):
            cache.update(new_k, new_k, i)                       # attention appended this token's (k, v)
            len_before = cache.layers[i].keys.shape[2]
            fires = press.layer_step_counts[i] + 1 >= press.compression_interval
            if fires:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            t0 = time.perf_counter()
            press.forward_hook(modules[i], [], kwargs, out)
            dt = time.perf_counter() - t0
            if fires:
                e1.record()
                comp_ev.append((e0, e1, len_before))
                compact_host_s += dt
                n_compact += 1
            else:
                hook_s += dt
                n_plain += 1
    torch.cuda.synchronize()
    wall = time.perf_counter() - t_loop
    dev_us = [a.elapsed_time(b) * 1e3 for a, b, _ in comp_ev]
    sizes = sorted({n for _, _, n in comp_ev})
    final_len = cache.layers[0].keys.shape[2]
    res = {"workload": "decoding_loop_qwen3_8b", "baseline_config_index": 3,
           "description": f"DecodingPress(KnormPress, 512, 2048), {n_layers} layers [1,8,S,128], {prompt}-token prompt + "
                          f"{steps_tokens} generated tokens (cache appends + hooks; model forward not included)",
           "generated_tokens": steps_tokens, "hook_us_per_layer_token_no_compaction": hook_s / max(1, n_plain) * 1e6,
           "compactions": n_compact, "compaction_sizes_before": sizes, "final_cache_len": final_len,
           "compaction_host_us_per_call": compact_host_s / max(1, n_compact) * 1e6,
           "compaction_device_us_per_call_mean": (sum(dev_us) / len(dev_us)) if dev_us else None,
           "compaction_device_us_per_call_min": min(dev_us) if dev_us else None,
           "press_overhead_share_of_loop": (hook_s + compact_host_s) / wall, "loop_wall_s": wall}
    del cache
    torch.cuda.empty_cache()
    return res


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default=os.environ.get("KVP_BENCH_WORKLOAD", DEFAULT_WORKLOAD), choices=list(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-mode", default="auto", choices=["auto", "serial", "staged", "zero_copy"],
                    help="host path: serial = H2D, compress, D2H on one stream; staged = per-kv-head 3-stream pipeline "
                         "(kvpress_b200.host_staging); zero_copy = staged + kept V rows read in place over PCIe")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager C-ABI call only")
    ap.add_argument("--no-extras", action="store_true", help="skip the other BASELINE configs after the headline")
    ap.add_argument("--layers", type=int, default=80, help="layers of the configs[4] pipeline-split extra")
    ap.add_argument("--gen-tokens", type=int, default=1024,
                    help="generated tokens of the configs[3] decoding-loop extra (8192 = the config's full length)")
    ap.add_argument("--no-numa", action="store_true")
    ap.add_argument("--cpu-step-budget", type=float, default=None,
                    help="seconds one CPU call of the reference arm may take (sizes its bounded sample); default: "
                         "chosen so that warmup + steps calls end within ~2 minutes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32 / "
                         "float64, under 64 MB in all: larger outputs as a fixed seeded sample of rows); with the same "
                         "arguments the inputs are the same on every run, so two builds can be compared output by output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    ratio = effective_ratio(w)
    n_kept = w.get("n_kept") or kept_count(w["S"], ratio)
    metric = "KV tokens scored+compacted/sec"
    bytes_per_set = 2 * w["B"] * w["Hkv"] * w["S"] * w["D"] * 2
    n_sets = max(1, min(8, -(-4 * L2_BYTES // bytes_per_set)))
    config = {
        "workload": args.workload, "description": w["label"], "baseline_config_index": w["config_index"],
        "B_per_gpu": w["B"], "Hkv": w["Hkv"], "Hq": w["Hq"], "S": w["S"], "D": w["D"], "n_kept": n_kept,
        "compression_ratio": ratio, "sharding": f"batch over {world} rank(s), no data-path collective",
        # identical in both arms (it describes the workload, not the run): how the GPU arm keeps K/V out of L2
        "l2": (f"{n_sets} rotating input sets x {bytes_per_set / 2**20:.0f} MiB (> L2) so no step re-reads cached K/V"
               if n_sets > 1 else f"inputs {bytes_per_set / 2**20:.0f} MiB per step > 126 MiB L2"),
    }

    # ---------------- reference arm: the reference's CPU implementation, rank 0 only ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        # exactly `steps` timed calls after `warmup` untimed ones; each call is a bounded sample sized so that the
        # whole run ends within ~2 minutes
        per_step = args.cpu_step_budget or max(0.05, min(2.0, 100.0 / (args.steps + max(args.warmup, 1))))
        res = cpu_arm(w, args.warmup, args.steps, per_step)
        line = {
            "impl": "reference", "metric": metric, "value": res["value"], "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["seconds_per_call"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config,
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line), flush=True)
        return

    # ---------------- B200 arm ---------------------------------------------------------------------
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    numa = None if args.no_numa else bind_to_gpu_numa(local_rank)
    torch.cuda.set_device(local_rank)
    device = f"cuda:{local_rank}"
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device(device))

    from kvpress_b200 import native

    native.load()

    # enough distinct input sets that consecutive steps never find their K/V in L2
    sets = [make_inputs(w, device, rank_seed(rank, i)) for i in range(n_sets)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    eager_calls = [lambda s=s: run_native(w, s[0], s[1], s[2], n_kept) for s in sets]
    warm = max(args.warmup, 3)
    timed_loop(eager_calls, warm)
    graphs = None
    if not args.no_graph:
        graphs = [native.capture(c) for c in eager_calls]
        timed_loop([g.replay for g in graphs], warm)
    calls = [g.replay for g in graphs] if graphs is not None else eager_calls
    barrier()
    with ClockSampler(local_rank) as clocks:
        ms_local, host_us, last_out = timed_loop(calls, args.steps)
    barrier()
    ms_per_step = max_over_ranks(ms_local, dist, device)
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = {"dir": args.dump_outputs, "arrays": dump_outputs(args.dump_outputs, w, last_out)}
    eager = None
    if graphs is not None:
        ms_e, host_e, _ = timed_loop(eager_calls, args.steps)
        barrier()
        eager = {"ms_per_step": max_over_ranks(ms_e, dist, device), "host_us_per_call": host_e}
    tokens_per_step = w["B"] * w["S"] * world
    value = whole_job_tokens_per_s(w["B"] * w["S"], world, ms_per_step)

    # roofline of one compress call on one GPU
    peaks = load_peaks()
    abytes = algorithmic_bytes(w, n_kept)
    achieved = abytes / (ms_per_step * 1e-3) / 1e9
    p = native.make_problem(sets[0][0], sets[0][1], n_kept, w["Hq"])
    if w["scorer"] == "knorm_rerotate":  # kvp_knorm_score (1) + kvp_scores_compress_rerotate (generic: 3)
        launches = 1 + native.launches_per_compress(p, 0)
    elif w["scorer"] == "adakv_ea":  # EA score (memset, logits incl. value norms, finalize, sentinel) + 2 x kvp_scores_select (3 each)
        launches = 4 + 2 * native.launches_per_compress(p, 0)
    else:
        scorer_id = {"knorm": 1, "streaming": 2, "snapkv": 3, "expected_attention": 4, "keydiff": 5}[w["scorer"]]
        launches = native.launches_per_compress(p, scorer_id)
    roofline = {
        "bound": "hbm", "kernel": f"kvp_{w['scorer']}_compress ({launches} launches: score, select, compact)",
        "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
        "peak_source": peaks["source"], "algorithmic_bytes_per_launch": abytes, "traffic": None,
    }
    tr = load_traffic(args.workload)
    if tr is not None:
        roofline["traffic"] = tr["dram_bytes_per_call"]
        roofline["traffic_source"] = tr["source"]
        roofline["kernel_us_ncu"] = tr.get("kernel_us")
    flops = algorithmic_flops(w)
    if flops:
        # lower bound on the tensor-core rate of the score stage: all of the step time charged to it
        roofline["tensor"] = {"algorithmic_flops_per_launch": flops, "achieved_tflops_lower_bound": flops / (ms_per_step * 1e-3) / 1e12,
                              "peak_tflops": peaks["bf16_tflops"], "unit": "TFLOP/s"}
    if mufu_bound_us(w):
        roofline["mufu"] = {"bound_us": mufu_bound_us(w), "frac": mufu_bound_us(w) / (ms_per_step * 1e3),
                            "note": "two exact-softmax passes, 16 MUFU.EX2 / clk / SM"}

    # ---------------- e2e: pinned host K/V in, compacted K'/V' out, through the host-buffer API ---------
    e2e = None
    if not args.no_e2e:
        Kh, Vh, extra_h = make_inputs(w, device, 99 + rank, pinned_host=True)
        out_k = torch.empty((w["B"], w["Hkv"], n_kept, w["D"]), dtype=torch.bfloat16).pin_memory()
        out_v = torch.empty_like(out_k).pin_memory()
        out_idx = torch.empty(w["B"] * w["Hkv"] * (w["S"] - n_kept), dtype=torch.int32).pin_memory()
        e2e_steps = max(2, min(args.steps, 8))

        from kvpress_b200 import host_staging

        mode = args.e2e_mode
        if mode == "auto":
            # measured (profiles/r01_e2e_modes.txt): zero_copy > staged > serial wherever V is not read to score
            mode = {"knorm_rerotate": "serial", "adakv_ea": "serial", "expected_attention": "staged"}.get(w["scorer"], "zero_copy")
        if mode != "serial" and w["scorer"] in ("knorm_rerotate", "adakv_ea"):
            raise SystemExit("this workload only has the serial host path")
        if mode == "zero_copy" and w["scorer"] == "expected_attention":
            raise SystemExit("zero_copy needs a scorer that does not read V to score")

        extra_pinned = {k: v.cpu().pin_memory() for k, v in extra_h.items()}  # small operands travel every step too

        def e2e_step():
            extra_d = {k: v.to(device, non_blocking=True) for k, v in extra_pinned.items()}
            if mode == "serial":
                Kd = Kh.to(device, non_blocking=True)
                Vd = Vh.to(device, non_blocking=True)
                k2, v2 = run_native(w, Kd, Vd, extra_d, n_kept)
                if v2 is None:  # head-wise selection: the result is the pruned index list
                    out_idx.copy_(k2.reshape(-1), non_blocking=True)
                    return
                out_k.copy_(k2, non_blocking=True)
                out_v.copy_(v2, non_blocking=True)
                return
            params = dict(extra_d)
            if w["scorer"] == "snapkv":
                params.update(window=64, kernel_size=5)
            if w["scorer"] == "expected_attention":
                params.update(epsilon=0.0, n_sink=4, use_vnorm=True)
            host_staging.compress_host(w["scorer"], Kh, Vh, n_kept, device=device, out_keys=out_k, out_values=out_v,
                                       heads_per_chunk=1, values_zero_copy=(mode == "zero_copy"), **params)

        for _ in range(3):
            e2e_step()
        barrier()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(e2e_steps):
            e2e_step()
        stop.record()
        torch.cuda.synchronize()
        barrier()
        e2e_ms = max_over_ranks(start.elapsed_time(stop), dist, device) / e2e_steps
        small = sum(v.numel() * v.element_size() for v in extra_pinned.values())
        h2d_bytes = small + {"serial": 2 * Kh.numel() * 2, "staged": 2 * Kh.numel() * 2,
                             "zero_copy": (2 * out_k.numel() * 2 if w["scorer"] == "streaming"
                                           else Kh.numel() * 2 + out_v.numel() * 2)}[mode]
        e2e = {
            "value": tokens_per_step / (e2e_ms * 1e-3), "unit": "tokens/s", "ms_per_step": e2e_ms, "steps": e2e_steps,
            "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": (out_idx.numel() * 4 if w["scorer"] == "adakv_ea" else 2 * out_k.numel() * 2),
            "mode": mode, "numa_binding": numa,
            "path": {"serial": "pinned host K,V -> H2D -> kvp_*_compress -> D2H K',V' on one stream",
                     "staged": "kvpress_b200.host_staging.compress_host: per-kv-head chunks, H2D | kvp_*_compress | D2H "
                               "on three streams",
                     "zero_copy": "host_staging.compress_host: K staged per kv-head, kept V rows gathered in place "
                                  "from pinned host memory by the compaction kernel, D2H overlapped"}[mode],
        }
        del Kh, Vh, out_k, out_v, out_idx

    # ---------------- extras: the other BASELINE configs, same process, same timing method ----------
    extras, extras_errors = [], []
    del sets, graphs, calls, eager_calls
    torch.cuda.empty_cache()
    if not args.no_extras:
        def attempt(fn, *a):
            try:
                r = fn(*a)
                if r is not None:
                    extras.append(r)
            except Exception as ex:  # an extra must never cost the headline line
                extras_errors.append(f"{fn.__name__}: {repr(ex)[:200]}")
                torch.cuda.empty_cache()

        xs = max(3, min(args.steps, 20))
        if args.workload == DEFAULT_WORKLOAD:
            attempt(extra_layer_split, device, rank, world, dist, 3, args.layers, peaks)   # every rank takes part
            if world == 1:
                attempt(extra_workload, "snapkv_32k", device, rank, xs, peaks)
                attempt(extra_workload, "knorm_128k", device, rank, xs, peaks)
                attempt(extra_workload, "decoding_knorm", device, rank, 5 * xs, peaks)
                attempt(extra_decoding_loop, device, args.gen_tokens)
                attempt(extra_ea_with_prologue, device, rank, 3)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    cpu_baseline = None
    if not args.no_cpu and world == 1:
        res = cpu_arm(w, 1, 3, per_step_budget_s=4.0)
        cpu_baseline = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}

    line = {
        "metric": metric, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config, "roofline": roofline,
        "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches * args.steps,
        "step_issue": "eager C-ABI call" if args.no_graph else "CUDA-graph replay of the C-ABI call (native.GraphedCall)",
        "host_us_per_call": host_us, "eager": eager,
        "clocks": clocks.summary(), "token_heads_per_s": value * w["Hkv"],
        "extras": extras, "extras_errors": extras_errors,
    }
    if dumped is not None:
        line["dumped_outputs"] = dumped
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
