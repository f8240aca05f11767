"""bench.py — SCAIL-14B denoising steps/sec at 512p/81f (config A of BASELINE.json / SURVEY §8d).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one sampler step of the reference (sgm/modules/diffusionmodules/sampling.py:950-963): the
CFG-duplicated batch-2 DiT forward over the ref || noise || pose sequence (N = 27 904 tokens, 40 blocks,
hidden 5120), CFG combine and the Euler update.  `value` = steps/s with inputs resident in HBM; `e2e` = the
same step through scail_b200.sampler.HostStep (pinned host -> device inputs, device -> host latent) timed
inside the region; `fwd_per_s` (extra key) = value * 2 is the b=1-forward rate BASELINE.md's targets are
quoted on (SURVEY F3).  Random-init weights of the 14B architecture, synthetic inputs (no network).

N > 1: one process per GPU (torchrun); strong scaling (the step is fixed).  Default layout for even N
(`--parallel auto`): the two CFG branches on the two halves of the ranks, context parallel over the token dimension
inside each half with one NCCL K/V all-gather per block (scail_b200.parallel.HybridParallel); `--parallel cp` = pure
context parallel over all ranks.  Every N > 1 line carries `cp_check_rel` (2 blocks of step 0 vs a single-GPU recompute on
rank 0) and `latent_checksum` (equal to the 1-GPU line's for the same --steps/--warmup).

--impl reference: the reference's own CPU implementation of the path cannot travel to the GPU box
(/root/reference is absent there), so this arm times the oracle port (oracle/dit_oracle.py, fp32, all host
threads) on a bounded sample — ONE full-width block at the full N = 27 904, b=1 (SURVEY §8d(ii)) — and scales it
by the 40 layers x 2 CFG branches it stands for (machine-readable: cpu_baseline.extrapolated / .extrapolation_factor).

--impl torchlib: the SAME step (same weights, same inputs, same N) on the PyTorch library path the reference
actually runs on a GPU (cuBLASLt F.linear, flash/cuDNN SDPA, F.layer_norm; baseline/torchlib.py).  The default arm
also times it after its own timed region and reports `library_baseline`, plus per-kernel `kernel_compare`
(ours vs cuBLAS / SDPA at the step's shapes) and `vae_decode` (config 5, ours vs cuDNN conv3d) at N=1.

--dump-outputs DIR (GPU arms): after the timed steps, rank 0 writes the fp32 latent the last timed step returned as
DIR/latent.npy.  Weights and inputs are seeded, so two builds run with the same arguments can be compared output for
output.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: importing the package must not write __pycache__ into it

import torch  # noqa: E402

D, F, HEADS, LAYERS, TEXT_DIM = 5120, 13824, 40, 40, 4096
T_LAT, H_LAT, W_LAT = 21, 64, 64  # 512x512, 81 frames
N_TEXT, N_CLIP = 512, 257
NCU_ATTN_DRAM_BYTES = 1.723713e9 + 0.555318e9  # per self-attention launch (b=2, 40 heads, N=27904), profiles/r02_ncu_summary.md


def seq_len(t=None, h=None, w=None):
    """ref + noise + pose tokens; defaults are read at CALL time so that --latent reaches every caller."""
    t, h, w = (T_LAT if t is None else t), (H_LAT if h is None else h), (W_LAT if w is None else w)
    return h * w // 4 + t * h * w // 4 + t * (h // 2) * (w // 2) // 4


def block_flops(n, d=D, f=F):
    """SURVEY §8d, per batch element."""
    return n * (12 * d * d + 4 * d * f) + 2 * (N_TEXT + N_CLIP) * d * 2 * d + 4 * n * n * d + 4 * n * (N_TEXT + N_CLIP) * d


def forward_flops(n):
    return LAYERS * block_flops(n) + 2 * n * 80 * D + 2 * n * D * 64


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            atexit.register(self.proc.terminate)  # the poller never ends by itself: stop it even if the run raises
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        time.sleep(0.05)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_inputs(seed=0):
    """SURVEY §8d C2: x~N(0,1) fp32; ref/pose ~N(0,1); ctx ~N(0,1) with padding rows zeroed; uncond = one EOS row."""
    g = torch.Generator().manual_seed(seed)
    bf = torch.bfloat16
    ctx = torch.randn(1, N_TEXT, TEXT_DIM, generator=g)
    ctx[:, 77:] = 0
    unc = torch.zeros(1, N_TEXT, TEXT_DIM)
    unc[:, 0] = torch.randn(TEXT_DIM, generator=g)
    return dict(x=torch.randn(1, T_LAT, 16, H_LAT, W_LAT, generator=g),
                ref_concat=torch.randn(1, 1, 16, H_LAT, W_LAT, generator=g).to(bf),
                concat_smpl_render=torch.randn(1, T_LAT, 16, H_LAT // 2, W_LAT // 2, generator=g).to(bf),
                context_cond=ctx.to(bf), context_uncond=unc.to(bf),
                image_clip_features=torch.randn(1, N_CLIP, 1280, generator=g).to(bf))


def build_model(device, layers=LAYERS, seed=1234):
    from scail_b200.dit import DiffusionTransformer
    torch.manual_seed(seed)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device(device):
            m = DiffusionTransformer(hidden_size=D, num_attention_heads=HEADS, inner_hidden_size=F, num_layers=layers,
                                     text_dim=TEXT_DIM, time_embed_dim=D)
    finally:
        torch.set_default_dtype(prev)
    return m.eval()


_ORACLE_BLOCK_CACHE = {}


def _oracle_block_inputs(n, g):
    if "sd" in _ORACLE_BLOCK_CACHE:  # ~0.8 G fp32 weights: drawn once per process, not once per timed step
        return _ORACLE_BLOCK_CACHE["sd"]
    sd = {}
    def lin(name, o, i):
        sd[name + ".weight"] = torch.randn(o, i, generator=g) * 0.02
        sd[name + ".bias"] = torch.zeros(o)
    p = "transformer.layers.0."
    lin(p + "attention.query_key_value", 3 * D, D); lin(p + "attention.dense", D, D)
    lin(p + "cross_attention.query", D, D); lin(p + "cross_attention.key_value", 2 * D, D); lin(p + "cross_attention.dense", D, D)
    lin(p + "mlp.dense_h_to_4h", F, D); lin(p + "mlp.dense_4h_to_h", D, F)
    lin("mixins.adaln_layer.clip_feature_key_value_list.0", 2 * D, D)
    sd[p + "post_cross_attention_layernorm.weight"], sd[p + "post_cross_attention_layernorm.bias"] = torch.ones(D), torch.zeros(D)
    for nm in ("query", "key", "cross_query", "cross_key", "clip_feature_key"):
        sd[f"mixins.adaln_layer.{nm}_layernorm_list.0.weight"] = torch.ones(D)
    sd["mixins.adaln_layer.adaLN_modulations.0"] = torch.randn(1, 6, D, generator=g) / D ** 0.5
    _ORACLE_BLOCK_CACHE["sd"] = sd
    return sd


def cpu_baseline(threads=None, budget_s=150.0):
    """Oracle port (fp32, torch CPU kernels incl. the library SDPA the reference calls, all host threads) on a bounded
    sample.  Preferred sample (SURVEY §8d(ii)): ONE full-width block at the FULL sequence length, b=1 — the extrapolation is
    then only x (40 layers x 2 CFG branches).  A calibration block on a 9x32x32 latent predicts its cost first; if the
    prediction exceeds `budget_s` on this host the reduced sample itself is reported, FLOP-scaled (and says so)."""
    from oracle import dit_oracle as O
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    O.USE_LIBRARY_SDPA = True  # F.scaled_dot_product_attention (what sat/transformer_defaults.py:67-72 calls): no N x N matrix
    g = torch.Generator().manual_seed(0)
    sd = _oracle_block_inputs(0, g)
    text, clip = torch.randn(1, N_TEXT, D, generator=g), torch.randn(1, N_CLIP, D, generator=g)
    emb = torch.randn(1, 6 * D, generator=g) * 0.1

    def run(t, h, w):
        n = seq_len(t, h, w)
        x = torch.randn(1, n, D, generator=g)
        cos, sin = O.rope_tables(128, t, h // 2, w // 2, 21, 150, 150)
        with torch.no_grad():
            t0 = time.time()
            O.block(sd, 0, x, emb, HEADS, cos, sin, text, clip)
            return n, time.time() - t0

    with torch.no_grad():
        run(4, 16, 16)  # warm-up (thread pool, allocator)
        n_s, dt_s = run(9, 32, 32)
    step_flops = 2 * forward_flops(seq_len())
    pred_full = dt_s * block_flops(seq_len()) / block_flops(n_s)
    if pred_full <= budget_s:
        n, dt = run(T_LAT, H_LAT, W_LAT)
        factor = step_flops / block_flops(n)
        sample = (f"oracle/dit_oracle.py fp32: 1 full-width block (d=5120, f=13824, 40 heads), b=1, FULL latent "
                  f"{T_LAT}x{H_LAT}x{W_LAT} (N={n} tokens) took {dt:.2f} s on {threads} threads; EXTRAPOLATED x{factor:.1f} "
                  f"(40 layers x 2 CFG branches + embed/final) to one sampler step; fp32 14B weights (64.6 GB) do not fit host RAM")
        kind_note = "full-N block"
    else:
        n, dt = n_s, dt_s
        factor = step_flops / block_flops(n)
        sample = (f"oracle/dit_oracle.py fp32: 1 full-width block, b=1, REDUCED latent 9x32x32 (N={n}) took {dt:.2f} s on {threads} "
                  f"threads (the full-N block was predicted at {pred_full:.0f} s > {budget_s:.0f} s budget); EXTRAPOLATED by FLOPs x{factor:.0f}")
        kind_note = "reduced-N block"
    est_step_s = dt * factor
    return {"value": 1.0 / est_step_s, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample,
            "sample_kind": kind_note, "sample_seconds": dt, "sample_tokens": n, "extrapolated": True,
            "extrapolation_factor": factor, "est_step_seconds": est_step_s}


CPU_ARM_BUDGET_S = 360.0  # host seconds the timed steps of `--impl reference` may spend on full-N blocks (K <= 3: full-N, ~80 s each on 128 threads)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for i in range(args.warmup + args.steps):
        # warm-up iterations use the reduced sample; the timed ones share ~3 minutes of host time, so the full-N block
        # (SURVEY 8d(ii)) is used when its predicted cost fits and the FLOP-scaled reduced block otherwise (the line says which)
        cb = cpu_baseline(budget_s=CPU_ARM_BUDGET_S / max(args.steps, 1) if i >= args.warmup else 0.0)
        if i >= args.warmup:
            vals.append(cb)
    v = statistics.mean(c["value"] for c in vals)
    cb = dict(vals[-1], value=v)
    print(json.dumps({"impl": "reference", "metric": "denoising steps/sec (SCAIL-14B, 512p/81f)", "value": v,
                      "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                      "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus, parallelism_name(args.gpus, args.parallel)),
                      "cpu_baseline": cb, "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0,
                                                  "d2h_bytes_per_step": 0}}))


def _time_cuda(fn, iters, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def kernel_compare(dev):
    """Ours vs the library kernel the reference would launch, at the step's shapes (b=2 rows = 2 x N), isolated, CUDA events."""
    from scail_b200 import ops
    n = seq_len()
    M = 2 * n
    res = {}
    for name, (N, K, epi) in {"qkv": (3 * D, D, 0), "attn_out": (D, D, 2), "fc1": (F, D, 1), "fc2": (D, F, 2)}.items():
        a = torch.randn(M, K, device=dev, dtype=torch.bfloat16)
        w = torch.randn(N, K, device=dev, dtype=torch.bfloat16) * 0.01
        b = torch.randn(N, device=dev, dtype=torch.bfloat16)
        out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        kw = dict(gate=torch.randn(2, N, device=dev, dtype=torch.bfloat16), residual=out, rows_per_batch=n) if epi == 2 else {}
        ms = _time_cuda(lambda: ops.gemm(a, w, b, out=out, epilogue=epi, **kw), 20, 3)
        ms_t = _time_cuda(lambda: torch.nn.functional.linear(a, w, b), 20, 3)
        lin = torch.nn.functional.linear
        if epi == 1:    # what the reference launches for the same math: F.linear then nn.GELU(tanh)
            lib = lambda: torch.nn.functional.gelu(lin(a, w, b), approximate="tanh")
        elif epi == 2:  # RowParallelLinear (matmul, + bias) then x + gate * y  (dit_video_crossattn_sc_xc.py:1036,1050)
            g3, r3 = kw["gate"].view(2, 1, N), out.view(2, n, N)
            lib = lambda: r3 + g3 * (lin(a, w) + b).view(2, n, N)
        else:
            lib = lambda: lin(a, w, b)
        ms_l = _time_cuda(lib, 20, 3)
        res["gemm_" + name] = {"ours_ms": round(ms, 3), "cublas_ms": round(ms_t, 3), "library_same_math_ms": round(ms_l, 3),
                               "ours_tflops": round(2 * M * N * K / ms / 1e9, 1), "ours_over_cublas": round(ms_t / ms, 3),
                               "ours_over_library_same_math": round(ms_l / ms, 3),
                               "note": "ours = one launch incl. the fused bias" + ("+GELU" if epi == 1 else "+gate+residual" if epi == 2 else "")
                                       + " epilogue; cublas_ms = F.linear alone; library_same_math_ms = F.linear plus the elementwise "
                                         "ops the reference runs after it; 20 back-to-back launches each (power cap settled)"}
        del a, w, out
    qkv = torch.randn(M, 3 * D, device=dev, dtype=torch.bfloat16)
    out = torch.empty(M, D, device=dev, dtype=torch.bfloat16)
    ms = _time_cuda(lambda: ops.attention(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], out, 2, HEADS, n, n), 3, 1)
    q4 = qkv.view(2, n, 3, HEADS, 128)
    qh, kh, vh = (q4[:, :, i].transpose(1, 2) for i in range(3))
    ms_t = _time_cuda(lambda: torch.nn.functional.scaled_dot_product_attention(qh, kh, vh), 3, 1)
    fl = 4 * 2 * HEADS * n * n * 128
    res["self_attention"] = {"ours_ms": round(ms, 3), "sdpa_ms": round(ms_t, 3), "ours_tflops": round(fl / ms / 1e9, 1),
                             "ours_over_sdpa": round(ms_t / ms, 3)}
    return res


VAE_TFLOP_A, VAE_MIN_BYTES_A = 180.5, 107.3e9  # SURVEY §8d: algorithmic FLOPs / minimum fused traffic of the decode @ 21x64x64


def vae_decode_bench(dev, peaks):
    """BASELINE.json config 5: Wan2.1 VAE decode of a [16,21,64,64] latent -> [3,81,512,512], random weights (seed 7)."""
    from baseline import torchlib
    from scail_b200.wan_vae import WanVAE
    torch.manual_seed(7)
    vae = WanVAE(dim=96, device=dev)
    z = torch.randn(16, T_LAT, H_LAT, W_LAT, device=dev).to(torch.bfloat16)
    with torch.no_grad():
        ms = min(_time_cuda(lambda: vae.decode([z]), 1, 1) for _ in range(3))
        try:
            ms_lib = min(_time_cuda(lambda: torchlib.vae_decode(vae, z), 1, 1) for _ in range(2))
        except Exception as e:  # a library failure must not take the product's line down with it
            ms_lib = None
            lib_err = repr(e)[:200]
    scale = (T_LAT * H_LAT * W_LAT) / (21 * 64 * 64)
    tf = VAE_TFLOP_A * scale / ms * 1e3
    out = {"workload": f"Wan2.1 VAE decode, latent {T_LAT}x{H_LAT}x{W_LAT} -> {4 * (T_LAT - 1) + 1} frames {8 * H_LAT}x{8 * W_LAT}",
           "ms": ms, "tflops": tf, "frac_of_bf16_burst_peak": tf / peaks["bf16_tflops"],
           "frac_of_bf16_sustained_peak": tf / peaks["bf16_tflops_sustained"], "algorithmic_tflop": VAE_TFLOP_A * scale,
           "library_ms": ms_lib, "library": "F.conv3d bf16 channels_last_3d (cuDNN) + F.normalize/silu/interpolate (baseline/torchlib.py)",
           "ours_over_library": (ms_lib / ms) if ms_lib else None}
    if ms_lib is None:
        out["library_error"] = lib_err
    return out


def cp_consistency_check(model, d, cond, uc, sig, rank, dist, plan=None, layers=2):
    """N > 1: the first `layers` blocks of step 0 computed (a) context-parallel over all ranks and (b) on rank 0 alone with
    the single-GPU path; returns relL2 of (a) vs (b) on rank 0 (None elsewhere) so the scaling run carries correctness."""
    from scail_b200 import sampler
    ad = model.mixins["adaln_layer"]
    x0 = d["x"].clone()
    a = sampler.sampler_step(model, x0.clone(), sig[0], sig[1], cond, uc, 4.0, plan=plan, _num_layers=layers)
    rel = None
    if rank == 0:
        cp, ad.cp = ad.cp, None
        try:
            b = sampler.sampler_step(model, x0.clone(), sig[0], sig[1], cond, uc, 4.0, _num_layers=layers)
        finally:
            ad.cp = cp
        dsig = float(sig[1]) - float(sig[0])
        va, vb = (a - x0) / dsig, (b - x0) / dsig
        rel = float((va - vb).norm() / vb.norm())
    dist.barrier()
    return rel


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy in float32, all of them together within DUMP_MAX_BYTES.  A tensor over its
    share is replaced by a fixed seeded sample of its flattened elements (the same positions on every run of one shape)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_MAX_BYTES // len(arrays) // 4
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > share:
            idx = torch.randint(a.numel(), (share,), generator=torch.Generator().manual_seed(0)).sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def parallelism_name(n_gpus, mode="auto"):
    if n_gpus <= 1:
        return "single"
    if mode == "auto":
        mode = "cfgxcp" if n_gpus % 2 == 0 else "cp"
    if mode == "cfgxcp":
        return f"cfg2xcp{n_gpus // 2}" if n_gpus > 2 else "cfg2"
    return f"cp{n_gpus}"


def workload_config(n_gpus, parallelism=None):
    return {"workload": f"SCAIL-14B one sampler step (CFG batch-2 DiT forward + CFG + Euler), latent {T_LAT}x{H_LAT}x{W_LAT} "
                        f"({8 * H_LAT}x{8 * W_LAT}, {4 * (T_LAT - 1) + 1} frames), N={seq_len()} tokens (ref | noise | pose), 40 blocks, "
                        "d=5120, 40 heads x 128, MLP 13824, text 512 + CLIP 257 keys",
            "global_batch": 2, "seq_len": seq_len(), "parallelism": parallelism or parallelism_name(n_gpus),
            "l2_policy": "inputs larger than L2 (32 GB weights, >5 GB activations per step)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torchlib"])
    ap.add_argument("--parallel", default="auto", choices=["auto", "cp", "cfgxcp"],
                    help="N > 1 layout: cp = tokens sharded over all ranks (one K/V all-gather per block); cfgxcp = the two CFG "
                         "branches on the two halves of the ranks, context parallel inside each half (default when N is even)")
    ap.add_argument("--no-extras", action="store_true", help="skip library_baseline / kernel_compare / vae_decode (profiling runs)")
    ap.add_argument("--layers", type=int, default=LAYERS, help=argparse.SUPPRESS)  # debugging only; default = full model
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--latent", default=None, help="TxHxW latent override, e.g. 21x64x112 (the reference's default 512x896); "
                    "the default 21x64x64 is the BASELINE.json config")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the latent the last timed step "
                    "returned as DIR/latent.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arms (--impl ours|torchlib)")
    if args.latent:
        global T_LAT, H_LAT, W_LAT
        T_LAT, H_LAT, W_LAT = (int(v) for v in args.latent.lower().split("x"))
    if args.impl == "reference":
        return run_reference_arm(args)

    from scail_b200 import ops, sampler
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep stdout to the one JSON line (some images default to NCCL_DEBUG=VERSION)
        dist.init_process_group("nccl", device_id=dev)
    model = build_model(dev, layers=args.layers)
    plan = None
    par = "single"
    if world > 1:
        from scail_b200.parallel import ContextParallel, HybridParallel
        mode = args.parallel if args.parallel != "auto" else ("cfgxcp" if world % 2 == 0 else "cp")
        if mode == "cfgxcp":
            plan = HybridParallel()
            model.mixins["adaln_layer"].cp = plan.cp
            par = f"cfg2xcp{plan.cp_size}" if plan.cp_size > 1 else "cfg2"
        else:
            model.mixins["adaln_layer"].cp = ContextParallel(dist.group.WORLD)
            par = f"cp{world}"
    host = synthetic_inputs()
    d = {k: v.to(dev) for k, v in host.items()}
    cond = dict(crossattn=d["context_cond"], ref_concat=d["ref_concat"], concat_smpl_render=d["concat_smpl_render"],
                image_clip_features=d["image_clip_features"])
    uc = dict(crossattn=d["context_uncond"])
    sig = sampler.make_flow_timesteps(50, 5.0)
    x = d["x"].clone()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lib_arm = args.impl == "torchlib"
    if lib_arm:
        assert world == 1, "--impl torchlib is the single-GPU library baseline"
        from baseline import torchlib

    def step(i):
        j = i % 50
        if lib_arm:
            x.copy_(torchlib.sampler_step(model, x, sig[j], sig[j + 1], cond, uc, 4.0))
        else:
            sampler.sampler_step(model, x, sig[j], sig[j + 1], cond, uc, 4.0, plan=plan)

    cp_check = None
    with torch.no_grad():
        if world > 1:
            cp_check = cp_consistency_check(model, d, cond, uc, sig, rank, dist, plan)
        for i in range(args.warmup):
            step(i)
        # ---- timed region: device-resident inputs ----
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        ops.ATTN_EVENTS = []
        barrier()
        launches0 = ops.LAUNCHES
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            step(args.warmup + i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / args.steps
        launches = (ops.LAUNCHES - launches0) // args.steps
        attn_ms = [a.elapsed_time(b) for a, b in ops.ATTN_EVENTS]
        ops.ATTN_EVENTS = None
        # ---- e2e: host buffers through the public API ----
        hs = sampler.HostStep(model, host, dev, step_fn=torchlib.sampler_step if lib_arm else None, plan=plan)
        hs(sig[0], sig[1])
        barrier()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(args.steps):
            hs(sig[i % 50], sig[i % 50 + 1])
        t1.record()
        barrier()
        e2e_ms = t0.elapsed_time(t1) / args.steps
        clk = clocks.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
    if rank != 0:
        return
    peaks, peak_src = measured_peaks()
    n = seq_len()
    step_flops = 2 * forward_flops(n) * args.layers / LAYERS
    # self-attention work of one rank per step = 40 layers x 4*B*H*(N/P)*N*128; at N>1 the two CFG branches are
    # separate launches (80 per step), so the per-launch figures are derived from the per-step totals
    n_attn = len(attn_ms) // args.steps if attn_ms else 0
    attn_flops = (4 * 2 * HEADS * (n / world) * n * 128) * args.layers / max(n_attn, 1)
    attn_avg = statistics.mean(attn_ms) if attn_ms else None
    value = 1000.0 / ms
    out = {"metric": "denoising steps/sec (SCAIL-14B, 512p/81f)", "value": value, "unit": "steps/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "bf16", "data": "synthetic (random-init 14B weights, seeded N(0,1) inputs)",
           "config": workload_config(world, par), "fwd_per_s": 2 * value,
           "step_tflops": step_flops / 1e12, "achieved_tflops_per_gpu": step_flops / world / ms / 1e9,
           "frac_of_bf16_sustained_peak": step_flops / world / ms / 1e9 / peaks["bf16_tflops_sustained"],
           "frac_of_bf16_burst_peak": step_flops / world / ms / 1e9 / peaks["bf16_tflops"],
           "gpu_launches": launches, "clocks": clk,
           "e2e": {"value": 1000.0 / e2e_ms, "unit": "steps/s", "h2d_bytes_per_step": hs.h2d_bytes,
                   "d2h_bytes_per_step": hs.d2h_bytes},
           "roofline": {"kernel": f"attention_fwd_kernel (self-attention, {n_attn} launches/step)", "bound": "tensor",
                        "achieved": attn_flops / attn_avg / 1e9 if attn_avg else None,
                        "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                        "frac": attn_flops / attn_avg / 1e9 / peaks["bf16_tflops_sustained"] if attn_avg else None,
                        "traffic": NCU_ATTN_DRAM_BYTES if (world == 1 and args.latent is None) else None,
                        "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this "
                                          "launch shape (profiles/r02_ncu_summary.md); algorithmic Q+K+V+O bytes = 2.286e9",
                        "peak_source": peak_src + ", sustained figure (kernel timed inside a long step)",
                        "algorithmic_flops_per_launch": attn_flops, "avg_launch_ms": attn_avg,
                        "share_of_step": sum(attn_ms) / args.steps / ms if attn_ms else None}}
    out["latent_checksum"] = float(x.double().abs().mean())  # same seeded inputs => comparable across N and across arms
    if args.dump_outputs:  # x still holds the last timed step's output: the e2e run above used its own buffers
        dump_outputs(args.dump_outputs, {"latent": x})
    if cp_check is not None:
        out["cp_check_rel"] = cp_check
    if args.layers != LAYERS:
        out["INVALID"] = f"debug run with {args.layers} layers"
    if lib_arm:
        out["impl"] = "torchlib"
        out["gpu_launches"] = 0
        out["roofline"] = None
        out["note"] = "PyTorch library path (cuBLASLt / flash-cuDNN SDPA / F.layer_norm), baseline/torchlib.py; none of this repo's kernels"
    elif world == 1 and not args.no_extras:
        try:  # an extra must never take the headline line down with it
            from baseline import torchlib
            with torch.no_grad():
                xl = d["x"].clone()
                fn = lambda: torchlib.sampler_step(model, xl, sig[10], sig[11], cond, uc, 4.0)
                lib_ms = _time_cuda(fn, 2, 1)
                # parity of the two arms on the bench's own inputs and weights (all 40 blocks, N = 27 904): the DiT velocity of
                # each CFG branch, ours vs the library chain (both bf16; neither is the fp32 truth)
                x2 = torch.cat([d["x"], d["x"]], 0)
                ts = torch.full((2,), float(sig[10]) * 1000.0, device=dev, dtype=torch.float32)
                ctx = sampler.prepare_context(cond, uc)
                v_o = model(x2, timesteps=ts, context=ctx, ref_concat=cond["ref_concat"], concat_smpl_render=cond["concat_smpl_render"],
                            image_clip_features=cond["image_clip_features"]).float()
                v_l = torchlib.dit_forward(model, x2, ts, ctx, cond["ref_concat"], cond["concat_smpl_render"],
                                           cond["image_clip_features"]).float()
                rel = [float((v_o[i] - v_l[i]).norm() / v_l[i].norm()) for i in range(2)]
                del x2, v_o, v_l
            out["library_baseline"] = {"steps_per_s": 1000.0 / lib_ms, "ms_per_step": lib_ms, "ours_over_library": lib_ms / ms,
                                       "what": "the same step (weights, inputs, N, bf16) on the PyTorch library path the reference runs "
                                               "on a GPU: F.linear (cuBLASLt), F.scaled_dot_product_attention, F.layer_norm; baseline/torchlib.py",
                                       "velocity_rel_l2_ours_vs_library": {"uncond": rel[0], "cond": rel[1]}}
            del xl
        except Exception as e:
            out["library_baseline"] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()
        try:  # SURVEY §8f rank 3: the same step with the forward captured in a CUDA graph (3 host launches per step)
            with torch.no_grad():
                xg = d["x"].clone()
                gs = sampler.GraphedStep(model, xg, cond, uc, 4.0)
                g_ms = _time_cuda(lambda: gs(sig[10], sig[11]), 2, 1)
            out["cuda_graph"] = {"steps_per_s": 1000.0 / g_ms, "ms_per_step": g_ms, "kernels_in_graph": gs.kernels_in_graph,
                                 "host_launches_per_step": 3, "vs_eager": ms / g_ms}
            del gs, xg
        except Exception as e:
            out["cuda_graph"] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()
        for key, fn in (("kernel_compare", lambda: kernel_compare(dev)), ("vae_decode", lambda: vae_decode_bench(dev, peaks))):
            try:  # an extra must never take the headline line down with it
                out[key] = fn()
            except Exception as e:
                out[key] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
    if not args.no_cpu_baseline and world >= 1 and not lib_arm:
        out["cpu_baseline"] = cpu_baseline()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
