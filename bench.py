#!/usr/bin/env python
"""bench.py - packed tokens/s of the TouchNet hot path on B200 (contract: see the task statement / DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one packed synthetic audio+text batch per GPU:
    raw waveforms -> fbank -> stack/stride -> input_features            (csrc/frontend.cu)
    TouchAudioForCausalLM forward (projector + 32 decoder layers + lm_head), pack-loss, backward
                                                                         (csrc/gemm.cu, attn_*.cu, elementwise.cu)
on the workload BASELINE.json's metric is quoted on: Llama-3-8B-ASR = TouchAudioForCausalLM around the Llama-3-8B text
config, packed seq_len 8192, one row per GPU (weak scaling), bf16 compute with fp32 master weights and fp32 weight
gradients.  `value` = tokens of all ranks / device time (CUDA events, max over ranks) with inputs resident in HBM;
`e2e` = the same through the public module API with the step's inputs starting in pinned host memory (H2D inside the
timed region) and the loss read back (D2H) every step.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time
from types import SimpleNamespace as NS

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG2E = 1.4426950408889634


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="llama3_8b_asr", choices=sorted(WORKLOADS),
                    help="llama3_8b_asr = the configuration the metric is quoted on (default); qwen2_audio_7b_asr = "
                         "BASELINE config 3 (MHA + q/k/v bias, V=156032, stack 13 / stride 12), a full-size smoke case")
    ap.add_argument("--seq-len", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None, help="packed rows per GPU")
    ap.add_argument("--layers", type=int, default=32, help="debug only: anything but 32 is not the named workload")
    ap.add_argument("--tp", type=int, default=1, help="tensor-parallel degree (BASELINE config 5); default mesh is pure FSDP2")
    ap.add_argument("--cp", type=int, default=1, help="context-parallel degree (BASELINE config 4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--with-optimizer", action="store_true",
                    help="also time fwd + bwd + grad-norm clip + B200AdamW step (extras.with_optimizer; N=1): the optimizer "
                         "kernel writes the bf16 working copies, so this loop has no fp32->bf16 cast kernels")
    ap.add_argument("--no-incumbent", action="store_true",
                    help="skip extras.incumbent (compiled flex_attention / cuBLAS / Liger / HF layer timed next to ours, N=1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32): the loss and a fixed, seeded "
                         "sample of every parameter gradient, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    select_workload(args)
    return args


# ---------------------------------------------------------------------------------------------------------------
# workload
# ---------------------------------------------------------------------------------------------------------------
STACK, STRIDE, MEL = 5, 4, 80          # audio pretrain recipe (examples/audio/pretrain/wenetspeech/run.sh:57)
WORKLOADS = {
    # BASELINE config 2/5 model around the audio projector: the configuration the metric is quoted on
    "llama3_8b_asr": dict(stack=5, stride=4, seq_len=8192, batch=1, name="Llama-3-8B-ASR", text=dict(
        hidden_size=4096, intermediate_size=14336, num_attention_heads=32, num_key_value_heads=8, vocab_size=128256,
        rope_theta=500000.0, attention_bias=False, model_type="llama",
        rope_scaling={"rope_type": "llama3", "factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                      "original_max_position_embeddings": 8192})),
    # BASELINE config 3: Qwen2-Audio-7B init shape (examples/audio/sft/asr/wenetspeech/config/Qwen2-Audio-7B.json:27-51)
    "qwen2_audio_7b_asr": dict(stack=13, stride=12, seq_len=4096, batch=2, name="Qwen2-Audio-7B-shaped ASR", text=dict(
        hidden_size=4096, intermediate_size=11008, num_attention_heads=32, num_key_value_heads=32, vocab_size=156032,
        rope_theta=10000.0, attention_bias=True, model_type="qwen2", rope_scaling=None)),
}
_W = WORKLOADS["llama3_8b_asr"]


def select_workload(args):
    global STACK, STRIDE, _W
    _W = WORKLOADS[args.workload]
    STACK, STRIDE = _W["stack"], _W["stride"]
    args.seq_len = args.seq_len or _W["seq_len"]
    args.batch = args.batch or _W["batch"]


def text_config(layers: int):
    """Default: Llama-3-8B shape (SURVEY 8: L=32, d=4096, H=32, KV=8, hd=128, ffn=14336, V=128256, theta 5e5 + llama3
    scaling)."""
    return NS(num_hidden_layers=layers, head_dim=128, rms_norm_eps=1e-5, tie_word_embeddings=False,
              initializer_range=0.02, pad_token_id=0, **_W["text"])


def asr_config(layers: int):
    return NS(audio_config=NS(input_size=MEL * STACK), text_config=text_config(layers), pad_token_id=0)


def make_host_batch(seed: int, B: int, T: int, vocab: int):
    """One packed audio+text batch in pinned host memory: raw fp32 waveforms + the integer side of the layout."""
    from touchnet_b200 import batching
    buf, placed = batching.plan_audio_text_batch(seed, B, T, vocab, stride=STRIDE, max_s=30.0)
    wav = torch.cat([u["waveform"] for u in placed]).contiguous().pin_memory()
    host = {
        "wav": wav,
        "input_ids": buf["input_ids"].pin_memory(),
        "labels": buf["labels"].pin_memory(),
        "position_ids": buf["position_ids"].pin_memory(),
        "attention_mask": buf["attention_mask"].pin_memory(),
        "sentence_lens": buf["sentence_lens"].pin_memory(),
    }
    meta = {
        "lens": [int(u["waveform"].numel()) for u in placed],
        "dst_rows": [u["row"] * T + u["offset"] for u in placed],
        "frames": [u["frames"] for u in placed],
        "num_sentence": int(buf["num_sentence"]),
        "doc_lens": [],
    }
    doc = buf["attention_mask"]
    for b in range(B):
        ids = doc[b][doc[b] > 0]
        if ids.numel():
            meta["doc_lens"] += torch.bincount(ids)[1:].tolist()
    meta["nonpad_tokens"] = int((doc > 0).sum())
    # compact form for the end-to-end arm (SURVEY 8(f) row 3): int16 PCM as stored on disk (touchnet/bin/make_data.py:202) +
    # per-document tables; the five [B,T] integer buffers are then built ON the device (batching.assemble_on_device)
    plan = batching.plan_documents(batching.synthetic_utterances(seed, vocab, stride=STRIDE, max_s=30.0), B, T, True)
    wav16 = (wav * 32768.0).round().clamp(-32768, 32767).to(torch.int16).contiguous().pin_memory()
    meta["plan"] = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in plan.items()}
    meta["wav_i16"] = wav16
    return host, meta


def dist_util_seed(base, rank):
    from touchnet_b200 import dist_util
    return dist_util.rank_seed(base, rank)


def to_device(host: dict, dev) -> dict:
    return {k: v.to(dev, non_blocking=True) for k, v in host.items()}


def h2d_bytes(host: dict) -> int:
    return int(sum(v.numel() * v.element_size() for v in host.values()))


def e2e_inputs(meta: dict, dev) -> dict:
    """The end-to-end arm's per-step inputs: H2D of the int16 waveforms and the per-document tables, then the [B,T] integer
    buffers assembled by tn_pack_layout_i64 on the device (bit-identical to the host batchers, tests/test_gpu_layout.py)."""
    from touchnet_b200 import batching
    d = batching.assemble_on_device(meta["plan"], dev)
    d["wav"] = meta["wav_i16"].to(dev, non_blocking=True)
    return d


def e2e_h2d_bytes(meta: dict) -> int:
    n = meta["wav_i16"].numel() * 2
    return int(n + sum(v.numel() * v.element_size() for v in meta["plan"].values() if torch.is_tensor(v)))


def run_step(model, d: dict, meta: dict, B: int, T: int, cp_slice=None):
    """frontend -> forward -> pack loss -> backward.  Returns the loss tensor (device).
    cp_slice: this rank's sequence window under context parallelism (every per-token buffer is cut to it, as the
    reference's create_context_parallel_ctx does, ref: touchnet/bin/train.py:363-387)."""
    from touchnet_b200 import frontend
    feats = torch.zeros((B * T, MEL * STACK), dtype=torch.float32, device=d["wav"].device)
    fb, frames = frontend.fbank_batch(d["wav"], meta["lens"], num_mel_bins=MEL)
    frontend.stack_batch(fb, frames, STACK, STRIDE, True, into=feats, dst_rows=meta["dst_rows"])
    feats = feats.view(B, T, -1)
    if cp_slice is not None:
        feats = feats[:, cp_slice].contiguous()
        d = {k: (v[:, cp_slice].contiguous() if v.dim() == 2 and v.shape[1] == T else v) for k, v in d.items()}
    out = model(input_ids=d["input_ids"], input_features=feats, attention_mask=d["attention_mask"],
                position_ids=d["position_ids"])
    # pack loss next to the path (ref: touchnet/loss/cross_entropy.py:12-50), fused CUDA (csrc/loss.cu)
    from touchnet_b200 import loss as tn_loss
    loss, _ = tn_loss.cross_entropy_loss(out.logits, d["labels"], d["sentence_lens"], meta["num_sentence"])
    loss.backward()
    return loss.detach()


# ---------------------------------------------------------------------------------------------------------------
# measurement helpers
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc = gpu_index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # samples under load only (the sampler also sees the idle edges of the region)
        loaded = [x for x in sm if mx is None or x > 0.4 * mx] or sm
        med = loaded[len(loaded) // 2] if loaded else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


class GemmTimer:
    """CUDA events around every launch of our library in the timed region (on the launching stream), summed per kernel
    class afterwards.  GEMM launches carry their algorithmic FLOPs."""

    def __init__(self):
        self.pairs = []
        self.shapes = []
        self._open = None

    def __call__(self, name, phase, args):
        if phase == "pre":
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            flops = 0.0
            if name == "tn_gemm_bf16":
                flops = 2.0 * args[11] * args[12] * args[13]
            elif name == "tn_gemm_swiglu_bf16":
                flops = 4.0 * args[9] * args[10] * args[11]
            elif name == "tn_gemm_qkv_bf16":
                flops = 2.0 * args[15] * args[16] * args[17]
            elif name == "tn_gemm_dswiglu_bf16":
                flops = 2.0 * args[10] * args[11] * args[12]
            shape = None
            if name == "tn_gemm_bf16":
                shape = ("gemm", int(args[2]), int(args[5]), int(args[8]), args[11], args[12], args[13])
            elif name == "tn_gemm_swiglu_bf16":
                shape = ("gemm_swiglu", 0, 0, 0, args[9], 2 * args[10], args[11])
            elif name == "tn_gemm_qkv_bf16":
                shape = ("gemm_qkv_mode%d" % int(args[0]), 0, 0, 0, args[15], args[16], args[17])
            elif name == "tn_gemm_dswiglu_bf16":
                shape = ("gemm_dswiglu", 0, 1, 0, args[10], args[11], args[12])
            self._open = (e, flops, name, shape)
        else:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            self.pairs.append((self._open[0], e1, self._open[1], self._open[2]))
            if self._open[3] is not None:
                self.shapes.append((self._open[0], e1, self._open[1], self._open[3]))

    def summary(self):
        ms = fl = 0.0
        n = 0
        for a, b, f, name in self.pairs:
            if name in ("tn_gemm_bf16", "tn_gemm_swiglu_bf16", "tn_gemm_qkv_bf16", "tn_gemm_dswiglu_bf16"):
                ms += a.elapsed_time(b); fl += f; n += 1
        return ms, fl, n

    def by_shape(self, peak_tflops: float):
        """Per GEMM shape (entry point, operand majorness, fp32 output flag, M, N, K): launches, mean ms, TFLOP/s and the
        fraction of the sustained tensor peak - the per-shape lines behind the aggregate `roofline`."""
        acc = {}
        for a, b, f, shp in self.shapes:
            kind, a_mn, b_mn, f32, M, N, K = shp
            key = f"{kind}{'_aT' if a_mn else ''}{'_bT' if b_mn else ''}{'_f32out' if f32 else ''} M={M} N={N} K={K}"
            e = acc.setdefault(key, [0, 0.0, 0.0])
            e[0] += 1; e[1] += a.elapsed_time(b); e[2] += f
        out = {}
        for k, (n, ms, fl) in sorted(acc.items(), key=lambda kv: -kv[1][1]):
            tf = fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
            out[k] = {"launches": n, "ms_mean": round(ms / n, 4), "tflops": round(tf, 1), "frac": round(tf / peak_tflops, 3)}
        return out

    def by_class(self):
        out = {}
        for a, b, f, name in self.pairs:
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return {k: round(v, 3) for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


def attn_flops_fwd_per_layer(doc_lens, H=32, hd=128):
    """mask-exact: 4*H*hd*sum n_i(n_i+1)/2 (SURVEY 8(d))."""
    return 4.0 * H * hd * sum(n * (n + 1) / 2 for n in doc_lens)


def attn_tile_flops_fwd_per_layer(doc, H=32, hd=128):
    """tile-granular: 4*H*hd*128*128 per (q block, kv block) pair the kernels visit (what the tensor pipe executes)."""
    tiles = 0
    for b in range(doc.shape[0]):
        d = doc[b]
        T = d.numel()
        start = torch.zeros(T, dtype=torch.long)
        change = torch.ones(T, dtype=torch.bool)
        change[1:] = d[1:] != d[:-1]
        idx = torch.arange(T)
        start = torch.cummax(torch.where(change, idx, torch.zeros_like(idx)), 0).values
        for qb in range((T + 127) // 128):
            rows = slice(qb * 128, min(T, (qb + 1) * 128))
            valid = d[rows] > 0
            if valid.any():
                lo = int(start[rows][valid].min()) // 128
                tiles += qb + 1 - lo
    return 4.0 * H * hd * 128 * 128 * tiles


def derived_columns(by_class: dict, steps: int, ms_per_step: float, attn_fwd_flop_step: float, nonpad_tokens: int,
                    tokens_per_step: int, B: int, T: int, layers: int, peaks: dict, text: dict,
                    attn_tile_flop_step: float = 0.0) -> dict:
    """The report columns of BASELINE.md (attention TFLOP/s and MFU, HBM GB/s of the norm / SwiGLU-backward / loss kernels,
    non-pad tokens/s, the reference's own MFU convention) from the per-entry-point device times of the timed region.
    rank 0's rows; never raises (a missing key only drops its column)."""
    out = {}
    try:
        per = {k: v / steps for k, v in by_class.items()}              # ms per step
        peak = float(peaks["bf16_sustained"])
        rows, d, ffn, V = B * T, text["hidden_size"], text["intermediate_size"], text["vocab_size"]
        out["nonpad_tokens_per_s_rank0"] = nonpad_tokens / (ms_per_step * 1e-3)
        if per.get("tn_attn_fwd_bf16"):
            tf = attn_fwd_flop_step / (per["tn_attn_fwd_bf16"] * 1e-3) / 1e12
            out["attn_fwd_tflops_mask_exact"] = tf
            out["attn_fwd_mfu_mask_exact"] = tf / peak
            if attn_tile_flop_step:
                out["attn_fwd_mfu_tile_granular"] = attn_tile_flop_step / (per["tn_attn_fwd_bf16"] * 1e-3) / 1e12 / peak
        if per.get("tn_attn_bwd_bf16"):
            tb = 2.5 * attn_fwd_flop_step / (per["tn_attn_bwd_bf16"] * 1e-3) / 1e12
            out["attn_bwd_tflops_mask_exact_2p5x"] = tb
            out["attn_bwd_mfu_mask_exact"] = tb / peak
            if attn_tile_flop_step:
                out["attn_bwd_mfu_tile_granular_2p5x"] = 2.5 * attn_tile_flop_step / (per["tn_attn_bwd_bf16"] * 1e-3) / 1e12 / peak
        gb = lambda bytes_, ms: bytes_ / (ms * 1e-3) / 1e9
        n_norm = 2 * layers + 1
        if per.get("tn_rmsnorm_fwd_bf16"):
            out["hbm_gbps_rmsnorm_fwd"] = gb(n_norm * rows * d * 4, per["tn_rmsnorm_fwd_bf16"])
        if per.get("tn_rmsnorm_bwd_bf16"):
            out["hbm_gbps_rmsnorm_bwd"] = gb(n_norm * rows * d * 8, per["tn_rmsnorm_bwd_bf16"])
        if per.get("tn_swiglu_bwd_bf16"):
            out["hbm_gbps_swiglu_bwd"] = gb(layers * rows * ffn * 10, per["tn_swiglu_bwd_bf16"])
        if per.get("tn_pack_ce_fwd_bf16"):
            out["hbm_gbps_pack_ce_fwd"] = gb(rows * V * 2, per["tn_pack_ce_fwd_bf16"])
        if per.get("tn_pack_ce_bwd_bf16"):
            out["hbm_gbps_pack_ce_bwd"] = gb(rows * V * 4, per["tn_pack_ce_bwd_bf16"])
        out["hbm_peak_gbps"] = peaks.get("hbm")
        # the reference's own MFU line (touchnet/models/llama/__init__.py:39-54: 6*N_non_embedding + 12*L*H*hd*T per token)
        H = text["num_attention_heads"]
        n_non_emb = layers * (2 * d * H * 128 + 2 * d * text["num_key_value_heads"] * 128 + 3 * d * ffn + 2 * d) + d
        flop_tok = 6 * n_non_emb + 12 * layers * H * 128 * T
        out["mfu_reference_convention_dense_attention_flops"] = flop_tok * tokens_per_step / (ms_per_step * 1e-3) / 1e12 / peak
    except Exception as e:                     # the headline line must never depend on these
        out["derived_columns_error"] = f"{type(e).__name__}: {e}"
    return out


def gemm_traffic():
    """Average DRAM bytes per GEMM launch of the step, from the newest committed ncu capture (profiles/rNN_gemm_traffic.json,
    produced by tools/gemm_traffic.py from an `ncu --metrics dram__bytes_*` run of this very command with --layers 2)."""
    for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                return json.load(open(p))
            except Exception:
                continue
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return {"bf16_sustained": j["bf16_tflops_sustained"], "bf16_burst": j["bf16_tflops"], "hbm": j["hbm_gbs"],
                "source": "measured"}
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "source": "fallback"}


# ---------------------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: the oracle port of the reference's CPU path on a bounded sample
# ---------------------------------------------------------------------------------------------------------------
CPU_SAMPLE_T = 2048


def cpu_reference_step(state):
    """One bounded sample: 1 of the 32 decoder layers, forward + backward, fp32, one packed row of CPU_SAMPLE_T tokens with
    the dense document mask (the only attention the reference runs on CPU, tests/touchnet/models/test_llama.py:93-95),
    plus the fbank+stack frontend for the audio of that row.  Returns seconds."""
    from oracle import frontend_oracle as fo
    from oracle import model_oracle as mo
    cfg, params, x, cos, sin, allow, wavs = state
    t0 = time.perf_counter()
    for w in wavs:
        fo.stack(fo.fbank(w), STACK, STRIDE, True)
    xx = x.clone().requires_grad_(True)
    y = mo.decoder_layer(xx, params, "model.layers.0.", cfg, cos, sin, allow)
    y.square().mean().backward()
    return time.perf_counter() - t0


def _cpu_threads() -> int:
    """Threads the CPU arm uses: the cores this process may run on (cgroup/affinity aware), capped at the physical-core
    count when it can be read - oversubscribing SMT siblings made the round-1 number swing 4x between boxes."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = min(n, phys)
    except Exception:
        pass
    return max(1, n)


def cpu_reference_setup(seed=2025):
    from oracle import model_oracle as mo
    from touchnet_b200 import batching
    torch.set_num_threads(_cpu_threads())
    tc = text_config(1)
    cfg = mo.OracleConfig(hidden_size=tc.hidden_size, intermediate_size=tc.intermediate_size, num_hidden_layers=1,
                          num_attention_heads=tc.num_attention_heads, num_key_value_heads=tc.num_key_value_heads,
                          head_dim=128, vocab_size=8,
                          rope_theta=tc.rope_theta, rope_scaling=tc.rope_scaling)
    g = torch.Generator().manual_seed(seed)
    d, f = cfg.hidden_size, cfg.intermediate_size
    L = "model.layers.0."
    nq, nkv = tc.num_attention_heads * 128, tc.num_key_value_heads * 128
    params = {L + "self_attn.q_proj.weight": torch.randn(nq, d, generator=g) * 0.02,
              L + "self_attn.k_proj.weight": torch.randn(nkv, d, generator=g) * 0.02,
              L + "self_attn.v_proj.weight": torch.randn(nkv, d, generator=g) * 0.02,
              L + "self_attn.o_proj.weight": torch.randn(d, nq, generator=g) * 0.02,
              L + "mlp.gate_proj.weight": torch.randn(f, d, generator=g) * 0.02,
              L + "mlp.up_proj.weight": torch.randn(f, d, generator=g) * 0.02,
              L + "mlp.down_proj.weight": torch.randn(d, f, generator=g) * 0.02,
              L + "input_layernorm.weight": torch.ones(d), L + "post_attention_layernorm.weight": torch.ones(d)}
    for p in params.values():
        p.requires_grad_(True)
    buf, placed = batching.plan_audio_text_batch(seed, 1, CPU_SAMPLE_T, tc.vocab_size, stride=STRIDE, max_s=30.0)
    doc, pos = buf["attention_mask"], buf["position_ids"]
    inv, sc = mo.rope_inv_freq(cfg)
    cos, sin = mo.rope_cos_sin(pos, inv, sc, torch.float32)
    allow = mo.doc_causal_allow(doc)
    x = torch.randn(1, CPU_SAMPLE_T, d, generator=g)
    wavs = [u["waveform"].numpy() for u in placed]
    return (cfg, params, x, cos, sin, allow, wavs)


def cpu_tokens_per_s(sec_per_sample: float) -> float:
    """Extrapolation stated in the sample string: 32 layers cost 32x the measured layer; embeddings/lm_head/loss not
    charged to the CPU arm (favours the CPU)."""
    return CPU_SAMPLE_T / (32.0 * sec_per_sample)


CPU_SAMPLE_DESC = (f"oracle port (fp32 torch, all host threads): fbank+stack of one packed row's audio + 1 of 32 decoder "
                   f"layers fwd+bwd on a {CPU_SAMPLE_T}-token packed row with the dense document mask; tokens/s = "
                   f"{CPU_SAMPLE_T} / (32 x t_sample); embeddings, lm_head and loss not charged")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    state = cpu_reference_setup()
    for _ in range(max(args.warmup, 1)):
        cpu_reference_step(state)
    ts = [cpu_reference_step(state) for _ in range(args.steps)]
    sec = sum(ts) / len(ts)
    val = cpu_tokens_per_s(sec)
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": "packed_tokens_per_sec", "value": val, "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": reference_config(args),
            "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": CPU_SAMPLE_DESC},
            "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def reference_config(args):
    """The CPU arm's OWN configuration (what it really ran), next to the workload it is extrapolated to."""
    t = _W["text"]
    return {"workload": f"CPU sample of {_W['name']}: 1 of 32 decoder layers (d={t['hidden_size']} H={t['num_attention_heads']} "
                        f"KV={t['num_key_value_heads']} ffn={t['intermediate_size']}), fp32, eager attention with the dense "
                        f"document mask, one packed row of {CPU_SAMPLE_T} tokens + fbank80 stack{STACK}/stride{STRIDE} of that "
                        f"row's audio, fwd+bwd; tokens/s extrapolated as {CPU_SAMPLE_T}/(32 x t_sample); embeddings, lm_head "
                        f"and loss not charged",
            "global_batch": 1, "seq_len": CPU_SAMPLE_T, "layers_measured": 1, "layers_extrapolated_to": 32,
            "parallelism": f"host CPU, {_cpu_threads()} threads (torch intra-op), no GPU",
            "extrapolated_to": workload_config(args, args.gpus)["workload"]}


FSDP_COLLECTIVES = "NCCL all-gather / reduce-scatter"


def workload_config(args, n):
    t = _W["text"]
    return {"workload": f"{_W['name']} (TouchAudioForCausalLM, text config L={args.layers} d={t['hidden_size']} "
                        f"H={t['num_attention_heads']} KV={t['num_key_value_heads']} ffn={t['intermediate_size']} "
                        f"V={t['vocab_size']}{' +qkv bias' if t['attention_bias'] else ''}, projector {MEL * STACK}->"
                        f"{t['hidden_size']}), audio+text packed rows, fbank80 stack{STACK}/"
                        f"stride{STRIDE} frontend on GPU, fwd+bwd, fp32 master weights + fp32 weight grads",
            "global_batch": args.batch * n, "seq_len": args.seq_len,
            "parallelism": "single GPU" if n == 1 else
                           f"FSDP2 dp_shard={n // (args.tp * args.cp)} (bf16 params / fp32 reduce, reshard policy "
                           f"{'default' if os.environ.get('TN_FSDP_RESHARD', '0') != '0' else 'never'})"
                           + (f" x TP={args.tp} (+sequence parallel, "
                              f"{'peer-memory GEMM epilogues' if os.environ.get('TN_TP_PEER', '0') != '0' else 'NCCL'})" if args.tp > 1 else "")
                           + (f" x CP={args.cp} ({'K/V halo exchange' if os.environ.get('TN_CP_HALO', '1') != '0' else 'K/V all-gather'}"
                              f", exact document mask)" if args.cp > 1 else "")
                           + f"; FSDP2 collectives: {FSDP_COLLECTIVES}",
            "l2_policy": "inputs larger than L2: every step streams >16 GB of weights through a 126 MB L2"}


# ---------------------------------------------------------------------------------------------------------------
# main arm
# ---------------------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: touchnet_b200 has no CPU path")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"

    from touchnet_b200 import _lib, modeling, ops
    _lib.load()
    sm_margin = int(os.environ.get("TN_SM_MARGIN", "0"))
    _lib.call("tn_set_sm_margin", sm_margin)   # leave SMs to the FSDP2 NCCL kernels so that they overlap the GEMMs
    _lib.call("tn_set_gemm_l2_hints", int(os.environ.get("TN_GEMM_L2_HINTS", "0") != "0"))   # A/B switch
    _lib.call("tn_set_gemm_split_tail", int(os.environ.get("TN_GEMM_SPLIT_TAIL", "1") != "0"))   # A/B switch
    B, T = args.batch, args.seq_len
    cfg = asr_config(args.layers)

    torch.manual_seed(2025)
    with torch.device(dev):
        model = modeling.B200TouchAudioForCausalLM(cfg)
    with torch.no_grad():                     # HF init: normal(0, 0.02), norms = 1 (fp32 master weights)
        for p in model.parameters():
            if p.dim() == 2:
                p.normal_(0.0, 0.02)
    tp, cp = args.tp, args.cp
    assert world % (tp * cp) == 0, f"--tp {tp} x --cp {cp} must divide {world} GPUs"
    dp = world // (tp * cp)
    cp_slice = None
    if world > 1:
        from torch.distributed.fsdp import MixedPrecisionPolicy, fully_shard
        from torch.distributed.device_mesh import init_device_mesh
        # mesh order of the reference: dp_shard outermost, then cp, tp innermost (touchnet/utils/distributed.py:116-157)
        full_mesh = init_device_mesh("cuda", (dp, cp, tp), mesh_dim_names=("dp_shard", "cp", "tp"))
        if tp > 1:
            os.environ.setdefault("TN_TP_PEER", "1")    # block collectives as GEMM epilogues storing into peer memory (validated
            from touchnet_b200 import tensor_parallel   # on 2 x B200, tools/check_tp.py); TN_TP_PEER=0 -> NCCL
            tensor_parallel.apply_tp(model, full_mesh["tp"])
            # loss parallel (the reference recipes' setting, run.sh:140): vocabulary-sharded logits into the pack-loss
            model.language_model.loss_parallel = os.environ.get("TN_TP_LOSS_PARALLEL", "1") != "0"
        if cp > 1:
            from touchnet_b200 import context_parallel
            context_parallel.enable_context_parallel(model, full_mesh["cp"].get_group())
            c = full_mesh["cp"].get_local_rank()
            cp_slice = slice(c * (T // cp), (c + 1) * (T // cp))
        mesh = full_mesh["dp_shard", "cp"]._flatten("dp_shard_cp") if cp > 1 else full_mesh["dp_shard"]
    if world > 1 and mesh.size() > 1:
        mp = MixedPrecisionPolicy(param_dtype=torch.bfloat16, reduce_dtype=torch.float32)
        layers = model.language_model.model.layers       # ref: touchnet/models/helper_func.py:134-202 apply_fsdp
        # reshard policy "never" of the reference (training_fsdp_reshard_after_forward, helper_func.py:141-186): the bf16
        # parameters stay gathered between forward and backward (16 GB per GPU, one all-gather per block per step instead
        # of two; measured +4.5 % at N=2).  TN_FSDP_RESHARD=1 selects the reference's "default" policy instead.
        reshard = os.environ.get("TN_FSDP_RESHARD", "0") != "0"
        for i, layer in enumerate(layers):
            fully_shard(layer, mesh=mesh, mp_policy=mp, reshard_after_forward=(reshard and i < len(layers) - 1))
        fully_shard(model, mesh=mesh, mp_policy=mp, reshard_after_forward=reshard)
        # FSDP2's collectives: default = copy-engine pushes over symmetric memory + one local reduce kernel
        # (touchnet_b200/fsdp_comm.py, mode "push": no SM is taken from the GEMMs; measured +5.7 % at N=2 over NCCL on the same
        # box); TN_FSDP_PEER=0 -> NCCL (the reference's path), =1 -> pull kernels.  Any failure to set it up falls back to NCCL.
        fsdp_mode = os.environ.get("TN_FSDP_PEER", "push")
        global FSDP_COLLECTIVES
        FSDP_COLLECTIVES = "NCCL all-gather / reduce-scatter"
        if fsdp_mode != "0":
            try:
                from touchnet_b200 import fsdp_comm
                fsdp_comm.install(model, mesh.get_group(), dev, max_ctas=int(os.environ.get("TN_FSDP_PEER_CTAS", "32")),
                                  mode="push" if fsdp_mode == "push" else "pull",
                                  direct=os.environ.get("TN_FSDP_DIRECT", "1") != "0")
                FSDP_COLLECTIVES = ("copy-engine pushes over NVLink symmetric memory + local reduce kernel" if fsdp_mode == "push"
                                    else "pull kernels over NVLink symmetric memory")
            except Exception as e:           # symmetric memory unavailable on this box: the reference's NCCL path
                if rank == 0:
                    print(f"[bench] peer-memory FSDP collectives unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
        depth = int(os.environ.get("TN_FSDP_PREFETCH", "0"))
        if depth > 0:                                    # explicit prefetch of the next `depth` blocks' all-gathers
            for i, layer in enumerate(layers):
                layer.set_modules_to_forward_prefetch(list(layers[i + 1:i + 1 + depth]))
                layer.set_modules_to_backward_prefetch(list(reversed(layers[max(0, i - depth):i])))
    model.train()
    # fused lm_head + pack-loss (no [B,T,V] logits): what the "*_b200" TrainSpecs run; TN_FUSED_CE=0 for the A/B
    model.fused_linear_ce = os.environ.get("TN_FUSED_CE", "1") != "0" and tp == 1

    host, meta = make_host_batch(dist_util_seed(2025, rank // (tp * cp)), B, T, cfg.text_config.vocab_size)  # dp coordinate
    resident = to_device(host, dev)
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(inputs):
        model.zero_grad(set_to_none=True)
        ops.invalidate_bf16_cache(model)     # the fp32->bf16 weight cast is part of every step
        return run_step(model, inputs, meta, B, T, cp_slice)

    # ---------------- device-resident arm ----------------
    for _ in range(max(args.warmup, 3)):
        one_step(resident)
    barrier()
    gt = GemmTimer()
    _lib._hooks.append(gt)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = _lib.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        loss = one_step(resident)
    e1.record()
    barrier()
    clocks = sampler.stop()
    _lib._hooks.remove(gt)
    launches = _lib.launch_count - launches0
    ms = e0.elapsed_time(e1)
    gemm_ms, gemm_flops, gemm_n = gt.summary()
    from touchnet_b200 import dist_util
    ms = dist_util.max_over_ranks(ms, dev)
    tokens_per_step = B * T * dp                     # tp / cp ranks share their rows
    value = dist_util.whole_job_tokens_per_s(B * T, args.steps, dp, ms)
    final_loss = float(loss.item())
    if args.dump_outputs:                     # before the later arms overwrite the gradients
        dump_outputs(args.dump_outputs, model, loss, rank)

    # ---------------- end-to-end arm: pinned host inputs, H2D inside, loss read back every step ----------------
    e2e = None
    if not args.no_e2e:
        compact = os.environ.get("TN_E2E_COMPACT", "1") != "0" and cp == 1
        feed = (lambda: e2e_inputs(meta, dev)) if compact else (lambda: to_device(host, dev))
        for _ in range(2):
            float(one_step(feed()).item())
        barrier()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(args.steps):
            l = one_step(feed())
            _ = float(l.item())                                  # D2H of the step's result
        t1.record()
        barrier()
        ms2 = t0.elapsed_time(t1)
        ms2 = dist_util.max_over_ranks(ms2, dev)
        e2e = {"value": tokens_per_step * args.steps / (ms2 * 1e-3), "unit": "tokens/s",
               "h2d_bytes_per_step": e2e_h2d_bytes(meta) if compact else h2d_bytes(host), "d2h_bytes_per_step": 4,
               "inputs": ("pinned host int16 waveforms + per-document tables; [B,T] id / label / position / mask buffers built "
                          "on the device (tn_pack_layout_i64), fbank from int16") if compact else
                         "pinned host fp32 waveforms + five host-built [B,T] int64 buffers"}

    with_opt = None
    if args.with_optimizer and world == 1:
        # fwd + bwd + clip + AdamW (touchnet/utils/optimizer.py:127-172, distributed.py:426-491 equivalents, csrc/optim.cu):
        # the clip coefficient is applied inside the AdamW kernel, which also writes next step's bf16 weights
        from touchnet_b200 import optim as tn_optim
        opt = tn_optim.B200AdamW(model.parameters(), lr=1e-5, betas=(0.9, 0.95), weight_decay=0.1)

        def opt_step():
            model.zero_grad(set_to_none=True)
            l = run_step(model, resident, meta, B, T, cp_slice)      # no cache invalidation: the optimizer refreshed the copies
            tn_optim.clip_grad_norm_(model.parameters(), 1.0, defer_to=opt)
            opt.step()
            return l
        for _ in range(3):
            opt_step()
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for _ in range(args.steps):
            opt_step()
        o1.record()
        barrier()
        ms3 = o0.elapsed_time(o1)
        with_opt = {"value": tokens_per_step * args.steps / (ms3 * 1e-3), "unit": "tokens/s", "ms_per_step": ms3 / args.steps,
                    "what": "fwd + bwd + fused grad-norm clip + B200AdamW step, fp32 master weights and moments; no "
                            "fp32->bf16 cast kernels in the loop (the AdamW kernel writes the bf16 working copies)",
                    "mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
        del opt
    if os.environ.get("TN_TRACE"):            # diagnostic: device timeline of ONE more step (not part of any number)
        trace_one_step(lambda: one_step(resident), os.environ["TN_TRACE"], rank, barrier)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    gemm_tflops = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    n_layers = args.layers
    attn_fwd = attn_flops_fwd_per_layer(meta["doc_lens"]) * n_layers
    line = {
        "metric": "packed_tokens_per_sec", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args, world),
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "roofline": {"bound": "tensor", "achieved": gemm_tflops, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                     "frac": gemm_tflops / peaks["bf16_sustained"],
                     "traffic": (gemm_traffic() or {}).get("avg_dram_bytes_per_gemm_launch"),
                     "algorithmic_bytes_per_launch": (gemm_traffic() or {}).get("avg_algorithmic_bytes_per_gemm_launch"),
                     "kernel": "tn::gemm_pair_kernel<A_MN,B_MN,EPI> (all GEMM launches of the timed region)",
                     "launches": gemm_n, "share_of_step": gemm_ms / ms if ms > 0 else None,
                     "by_shape": gt.by_shape(peaks["bf16_sustained"]),
                     "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']}); burst {peaks['bf16_burst']}"},
        "extras": {"nonpad_tokens_per_step_rank0": meta["nonpad_tokens"], "docs_rank0": len(meta["doc_lens"]),
                   "attn_fwd_tflop_mask_exact_per_step_rank0": attn_fwd / 1e12, "loss": final_loss,
                   "parity": {"loss_rank0": final_loss,
                              "note": "rank 0's batch and the weights are the same at every N (seed 2025, no optimizer step): under "
                                      "the default FSDP2 mesh this value equals the N=1 line's bit for bit - a driver-visible "
                                      "check that the sharded run computes the same function (tp / cp meshes print the loss of "
                                      "their own shard layout)"},
                   "model_tflop_per_step_rank0": gemm_flops / args.steps / 1e12,
                   "ms_by_entry_point_timed_region": gt.by_class(),
                   "mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30, "with_optimizer": with_opt,
                   "report_columns_rank0": derived_columns(gt.by_class(), args.steps, ms / args.steps, attn_fwd,
                                                           meta["nonpad_tokens"], B * T, B, T, n_layers, peaks, _W["text"],
                                                           attn_tile_flops_fwd_per_layer(host["attention_mask"],
                                                                                         _W["text"]["num_attention_heads"])
                                                           * n_layers)},
    }
    if world == 1 and not args.no_cpu_baseline:
        state = cpu_reference_setup()
        cpu_reference_step(state)
        ts = [cpu_reference_step(state) for _ in range(2)]
        sec = sum(ts) / len(ts)
        line["cpu_baseline"] = {"value": cpu_tokens_per_s(sec), "unit": "tokens/s", "cores": torch.get_num_threads(),
                                "kind": "port", "sample": CPU_SAMPLE_DESC}
    if world == 1 and not args.no_incumbent:
        # the kernels the reference's GPU path actually resolves to (flex_attention, cuBLAS, Liger, HF eager layer), same box,
        # same shapes, after our model is freed; never part of `value` / `--impl reference` (tools/incumbent.py)
        try:
            del model, resident, loss
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            from tools import incumbent
            line["extras"]["incumbent"] = incumbent.measure(budget_s=150.0)
        except Exception as e:
            line["extras"]["incumbent"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


DUMP_SAMPLE = 32768            # gradient elements written per parameter: ~30 MB for the 32-layer workloads
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, model, loss, rank):
    """What a caller of the timed step receives, as `out_dir/<name>.npy` in float32: `loss` (shape [1]) and
    `grad.<parameter name>`, the parameter's gradient at DUMP_SAMPLE flat indices drawn with a seed derived from the name
    (sorted; the whole gradient when it is no larger).  Sharded gradients are gathered first, so every rank calls this;
    rank 0 writes."""
    import zlib
    import numpy as np
    arrays = {"loss": loss.detach().float().reshape(1).cpu()}
    for name, p in model.named_parameters():
        if p.grad is None:
            continue
        grad = p.grad.full_tensor() if hasattr(p.grad, "full_tensor") else p.grad
        flat = grad.detach().reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randint(flat.numel(), (DUMP_SAMPLE,), generator=g).sort().values
            flat = flat[idx.to(flat.device)]
        arrays["grad." + name] = flat.float().cpu()
    if rank != 0:
        return
    total = sum(a.numel() * 4 for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total / 2**20:.1f} MB exceeds {DUMP_LIMIT_BYTES >> 20} MB")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def trace_one_step(step_fn, path, rank, barrier):
    """Kineto timeline of one step on every rank (so collectives progress); rank 0 writes `path` (csv.gz: name, stream,
    start_us, dur_us of every kernel / memcpy).  Used to see what FSDP2's streams overlap with (profiles/README.md)."""
    import gzip, tempfile
    from torch.profiler import profile, ProfilerActivity
    barrier()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step_fn()
        torch.cuda.synchronize()
    barrier()
    if rank != 0:
        return
    with tempfile.TemporaryDirectory() as td:
        tp = os.path.join(td, "t.json")
        prof.export_chrome_trace(tp)
        ev = json.load(open(tp))["traceEvents"]
    rows = [(e["ts"], e.get("dur", 0), e.get("args", {}).get("stream", -1), e["name"][:70].replace(",", ";"))
            for e in ev if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
    rows.sort()
    t0 = rows[0][0] if rows else 0
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with gzip.open(path, "wt") as f:
        f.write("name,stream,start_us,dur_us\n")
        for ts, dur, st, name in rows:
            f.write(f"{name},{st},{ts - t0:.1f},{dur:.1f}\n")


if __name__ == "__main__":
    main()
