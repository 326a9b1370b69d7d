"""Headline benchmark: Flux denoise it/s (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c5] [--impl ours|reference|reference-gpu]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" is one denoise step of the hot path (Flux.forward over all 19+38 blocks + the Euler update) for one sample
per GPU (batch-parallel across GPUs, weak scaling).  Default workload = BASELINE.json configs[1] (c2: Flux-dev
1024x1024, batch 1); --config selects the other BASELINE configurations:

    c2  Flux-dev     1024x1024  T=512  guidance        S=4608
    c3  Flux-schnell 1024x1024  T=256  no guidance     S=4352
    c4  Flux-dev      768x768   T=512  + merged LoRA   S=2816   (rank-16 LoRA fused on the device into every block linear)
    c5  Flux-dev     1536x1536  T=512  quantize_modulation=False (bf16 Modulation.lin)   S=9728

Weights are synthetic (seeded N(0, 0.02^2), quantised with the reference flow, input scales calibrated by >= 13 eager
steps on rank 0 and replicated with one NCCL broadcast); latents / text embeddings are synthetic tensors of the
published shapes.

--dump-outputs DIR writes the latent the timed loop returned after its last step (what a caller of
DenoiseSession.step_device receives) to DIR/latent.npy (DIR/latent_rank<r>.npy with several GPUs), float32.  Weights
and inputs are seeded, so two builds run with the same arguments can be compared output for output.  It covers
--impl ours only and is refused with the other arms: those time the reference's own modules as a baseline (a bounded
block sample on the host CPU, or a child process on the GPU), which do not change with this package's builds.

One JSON line on stdout (rank 0):
  value         sample-steps/s over all GPUs, latents resident in HBM (CUDA-graph replay per step)
  e2e           the same through DenoiseSession.step_host (pinned host latents, H2D + step + D2H per step)
  roofline      tcgen05 FP8 GEMM kernels: algorithmic FLOP/s from CUDA events around every launch of an instrumented
                pass, against the FP8 tensor-pipe ceiling MEASURED on this box in the same run (fluxb200_fp8_mma_probe)
  vae_decode    one AutoEncoder.decode of the config's image size through our kernels (SURVEY 8f N4), with the reference's
                cuDNN decode on the same GPU beside it when gpu_reference ran
  text_encoders the T5-XXL / CLIP-L text encoders through conditioner.accelerate and the Hugging Face modules themselves
  gpu_reference the UNMODIFIED reference modules (oracle/_ref) timed on the same GPU: eager, and torch.compile'd blocks
  cpu_baseline  the reference's bf16 blocks on the host cores (bounded sample)

--impl reference        the reference's own bf16 modules on the host CPU (all threads it can use), each step a bounded
                        sample (1 DoubleStreamBlock + 2 SingleStreamBlocks = 1/19 of the block stack of a step)
--impl reference-gpu    the reference's own fp8 modules on cuda:0 (eager or compiled), same harness (used for gpu_reference)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = {
    "c2": dict(model="Flux-dev", res=1024, text_len=512, guidance=True, qmod=True, lora=False, num_steps=28),
    "c3": dict(model="Flux-schnell", res=1024, text_len=256, guidance=False, qmod=True, lora=False, num_steps=4),
    "c4": dict(model="Flux-dev", res=768, text_len=512, guidance=True, qmod=True, lora=True, num_steps=28),
    "c5": dict(model="Flux-dev", res=1536, text_len=512, guidance=True, qmod=False, lora=False, num_steps=50),
}


def geometry(cfg):
    L = (cfg["res"] // 16) ** 2
    return L, L + cfg["text_len"]


def algorithmic_flops(cfg):
    """Per sample per step (SURVEY.md section 8d): fp8 GEMM, bf16 attention, bf16 modulation GEMV (c5 only)."""
    _, S = geometry(cfg)
    f8 = 1.29101e10 * S + (6.456e9 if cfg["qmod"] else 0.0)
    return f8, 700416.0 * S * S, (0.0 if cfg["qmod"] else 6.456e9)


def metric_name(cfg):
    return f"{cfg['model']} {cfg['res']}x{cfg['res']} denoise it/s"


def workload(cfg, what):
    L, S = geometry(cfg)
    extra = " + rank-16 LoRA merged into every block linear" if cfg["lora"] else ""
    extra += ", quantize_modulation=False (bf16 Modulation.lin)" if not cfg["qmod"] else ""
    return f"{cfg['model']} {cfg['res']}x{cfg['res']} denoise step (19 double + 38 single blocks, S={S}){extra}, {what}"


def config_block(cfg, key, world, extra=None):
    L, S = geometry(cfg)
    d = {"workload": workload(cfg, "batch 1 per GPU"), "baseline_config": key, "resolution": [cfg["res"], cfg["res"]],
         "seq_len": S, "text_len": cfg["text_len"], "global_batch": world,
         "parallelism": f"dp{world} (image batch, replicated fp8 weights)",
         "l2": "inputs larger than L2: ~12 GB of weights stream per step (L2 is 126 MB)"}
    d.update(extra or {})
    return d


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.path = gpu_index, None, f"/tmp/fluxb200_clocks_{os.getpid()}.csv"

    def __enter__(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:  # noqa: BLE001
                self.proc.kill()
            self.f.close()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "power_w_max": None, "reasons": [], "samples": 0}
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            rows = [[c.strip() for c in r] for r in rows if len(r) >= 9]
            if not rows:
                return out
            sm = [float(r[1]) for r in rows]
            busy = [s for s, r in zip(sm, rows) if float(r[3]) > 300.0] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=float(rows[0][2]),
                       power_w_max=max(float(r[3]) for r in rows), samples=len(rows))
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for i, n in enumerate(names):
                if any(r[5 + i].lower().startswith("active") for r in rows):
                    out["reasons"].append(n)
        except Exception as ex:  # noqa: BLE001
            out["error"] = str(ex)
        return out


def gemm_traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum per f8_gemm_kernel launch, averaged over the GEMM launches of one
    c2 step, from the newest committed ncu capture (profiles/r*_gemm_traffic.json, written by tools/ncu_traffic.py from
    `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` over tools/profile_step.py).  None if absent."""
    for name in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return float(json.load(f)["dram_bytes_per_launch"]), name
        except (OSError, KeyError, ValueError):
            continue
    return None, None


# ------------------------------------------------------------------------------------------------
# reference arms (bench.py is one of the places allowed to execute oracle/): the UNMODIFIED reference modules staged in
# oracle/_ref when present, else the oracle port
# ------------------------------------------------------------------------------------------------
def init_reference_weights(ref, net, seed=1234):
    """The synthetic checkpoint recipe of SURVEY.md section 8(d) on reference modules (plain torch)."""
    dev = next(net.parameters()).device
    g = torch.Generator(device=dev).manual_seed(seed)
    mod_lins = {id(m.lin) for m in net.modules() if isinstance(m, ref.fm.Modulation)}
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.Linear):
                is_mod = id(m) in mod_lins
                m.weight.copy_(torch.randn(m.weight.shape, device=dev, generator=g) * (0.01 if is_mod else 0.02))
                if m.bias is not None:
                    if is_mod:
                        m.bias.zero_()
                    else:
                        m.bias.copy_(torch.randn(m.bias.shape, device=dev, generator=g) * 0.02)
            elif isinstance(m, ref.fm.RMSNorm):
                m.scale.copy_(1 + 0.05 * torch.randn(m.scale.shape, device=dev, generator=g))


def reference_inputs(cfg, device, hidden=3072, dtype=torch.bfloat16):
    from oracle import flux_oracle as O

    L, S = geometry(cfg)
    g = torch.Generator().manual_seed(0)
    side = cfg["res"] // 16
    ids = torch.cat((torch.zeros(1, cfg["text_len"], 3, dtype=dtype), O.make_img_ids(1, side, side, dtype)), 1)
    return dict(img=torch.randn(1, L, hidden, generator=g).to(dtype).to(device),
                txt=torch.randn(1, cfg["text_len"], hidden, generator=g).to(dtype).to(device),
                vec=torch.randn(1, hidden, generator=g).to(dtype).to(device), ids=ids.to(device))


def cpu_sample_reference(cfg):
    """1 DoubleStreamBlock + 2 SingleStreamBlocks of the reference (bf16, flow_dtype=bfloat16 / no quantisation) at the
    config's full sequence length = exactly 1/19 of the block stack of one denoise step.  Returns (run, kind)."""
    from oracle import ref_loader as R

    inp = reference_inputs(cfg, "cpu")
    if R.available():
        ref = R.load()
        D, H = 3072, 24
        torch.manual_seed(0)
        dbl = ref.fm.DoubleStreamBlock(D, H, mlp_ratio=4.0, qkv_bias=True, dtype=torch.bfloat16).to(torch.bfloat16).eval()
        sgl = [ref.fm.SingleStreamBlock(D, H, mlp_ratio=4.0, dtype=torch.bfloat16).to(torch.bfloat16).eval()
               for _ in range(2)]
        for m in [dbl] + sgl:
            init_reference_weights(ref, m, seed=5)
        pe = ref.fm.EmbedND(128, 10_000, [16, 56, 56], torch.bfloat16)(inp["ids"])

        def run():
            with torch.inference_mode():
                img, txt = dbl(img=inp["img"], txt=inp["txt"], vec=inp["vec"], pe=pe)
                x = torch.cat((txt, img), 1)
                for b in sgl:
                    x = b(x, vec=inp["vec"], pe=pe)
            return x

        return run, "reference"
    # oracle port of the same blocks (oracle/_ref not staged)
    from oracle import flux_oracle as O

    g = torch.Generator().manual_seed(5)
    D, H, MLP, bf = 3072, 24, 12288, torch.bfloat16

    def lin(prefix, n, k, std=0.02):
        return {prefix + "weight": (torch.randn(n, k, generator=g) * std).to(bf),
                prefix + "bias": (torch.randn(n, generator=g) * 0.02).to(bf)}

    p = {}
    for s in ("img", "txt"):
        p.update(lin(f"d.{s}_mod.lin.", 6 * D, D, 0.01))
        p.update(lin(f"d.{s}_attn.qkv.", 3 * D, D))
        p.update(lin(f"d.{s}_attn.proj.", D, D))
        p.update(lin(f"d.{s}_mlp.0.", MLP, D))
        p.update(lin(f"d.{s}_mlp.2.", D, MLP))
        p[f"d.{s}_attn.norm.query_norm.scale"] = torch.ones(128, dtype=bf)
        p[f"d.{s}_attn.norm.key_norm.scale"] = torch.ones(128, dtype=bf)
    p.update(lin("s.modulation.lin.", 3 * D, D, 0.01))
    p.update(lin("s.linear1.", 3 * D + MLP, D))
    p.update(lin("s.linear2.", D, D + MLP))
    p["s.norm.query_norm.scale"] = torch.ones(128, dtype=bf)
    p["s.norm.key_norm.scale"] = torch.ones(128, dtype=bf)
    pe = O.embed_nd(inp["ids"], [16, 56, 56], 10_000, bf)

    def run():
        with torch.inference_mode():
            i2, t2 = O.double_block(inp["img"], inp["txt"], inp["vec"], pe, p, "d.", H)
            x = torch.cat((t2, i2), 1)
            for _ in range(2):
                x = O.single_block(x, inp["vec"], pe, p, "s.", H)
        return x

    return run, "port"


def pick_threads(run, budget_s=40.0):
    """The reference uses whatever torch's intra-op pool gives it; on many-core hosts the all-cores setting is not the
    fastest for these GEMM sizes (oversubscription / NUMA).  Try a few pool sizes once each, keep the fastest."""
    n = os.cpu_count() or 1
    cands = sorted({c for c in (n, n // 2, n // 4, 32, 16) if 1 <= c <= n}, reverse=True)
    best, best_t, t_begin = n, float("inf"), time.perf_counter()
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        if time.perf_counter() - t_begin > budget_s:
            break
    torch.set_num_threads(best)
    return best, best_t


def cpu_reference_measure(cfg, steps, warmup, tune=True):
    run, kind = cpu_sample_reference(cfg)
    threads = os.cpu_count() or 1
    fixed = os.environ.get("FLUXB200_BENCH_THREADS")  # pin the pool size (skips the search)
    if fixed:
        threads, tune = max(1, min(int(fixed), threads)), False
    torch.set_num_threads(threads)
    if tune:
        threads, _ = pick_threads(run)
    for _ in range(warmup):
        run()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
    sample_s = sum(times) / len(times)
    step_s = 19.0 * sample_s  # 19 x (1 double + 2 single) = the 19 + 38 blocks of a step
    return dict(value=1.0 / step_s, sample_s=sample_s, step_s=step_s, threads=threads, kind=kind, times=times)


def run_reference_arm(args, cfg, rank):
    """--impl reference: the reference's own CPU implementation of the path (its bf16 blocks, all host threads it can
    use), honouring --steps / --warmup; each step is the bounded sample described in cpu_sample_reference."""
    if rank != 0:
        return
    from oracle import ref_loader as R

    t0 = time.perf_counter()
    m = cpu_reference_measure(cfg, max(1, args.steps), max(0, args.warmup))
    wall = time.perf_counter() - t0
    L, S = geometry(cfg)
    sample = (f"each timed step = 1 DoubleStreamBlock + 2 SingleStreamBlocks of the "
              f"{'unmodified reference modules (oracle/_ref)' if m['kind'] == 'reference' else 'oracle port'}, bf16, B=1, "
              f"S={S} = 1/19 of the block stack of one denoise step; it/s = 1 / (19 x {m['sample_s']:.3f} s); "
              f"{m['threads']} threads (fastest of the pool sizes tried), {R.cpu_info()['model']}")
    line = {
        "impl": "reference", "metric": metric_name(cfg), "value": m["value"], "unit": "it/s",
        "n_gpus": args.gpus, "steps": max(1, args.steps), "warmup": max(0, args.warmup),
        "ms_per_step": m["sample_s"] * 1e3, "ms_per_full_step_extrapolated": m["step_s"] * 1e3,
        "sample_fraction_of_step": 1.0 / 19.0,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": config_block(cfg, args.config, max(1, args.gpus)),
        "cpu_baseline": {"value": m["value"], "unit": "it/s", "cores": m["threads"], "kind": m["kind"], "sample": sample},
        "e2e": {"value": m["value"], "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": wall,
    }
    print(json.dumps(line), flush=True)


VAE_PARAMS = dict(resolution=256, in_channels=3, ch=128, out_ch=3, ch_mult=[1, 2, 4, 4], num_res_blocks=2, z_channels=16,
                  scale_factor=0.3611, shift_factor=0.1159)  # util.py:178-188


def vae_decode_flops(res):
    """Multiply-add flops of Decoder.forward (modules/autoencoder.py:256-283) for a res x res image, convolutions and the
    mid-block attention (conv_in from the 16 real latent channels, conv_out to the 3 real image channels)."""
    h = res // 8
    ch, mult = VAE_PARAMS["ch"], VAE_PARAMS["ch_mult"]
    c = ch * mult[-1]
    px = h * h
    f = 2 * px * 16 * c * 9  # conv_in
    res_block = lambda cin, cout, p: 2 * p * 9 * (cin * cout + cout * cout) + (2 * p * cin * cout if cin != cout else 0)
    f += 2 * res_block(c, c, px) + 4 * 2 * px * c * c + 4 * px * px * c  # mid: two ResnetBlocks, q/k/v/proj_out, QK^T + PV
    for lvl in reversed(range(len(mult))):
        cout = ch * mult[lvl]
        for _ in range(VAE_PARAMS["num_res_blocks"] + 1):
            f += res_block(c, cout, px)
            c = cout
        if lvl != 0:
            px *= 4
            f += 2 * px * 9 * c * c  # Upsample.conv
    return f + 2 * px * 9 * c * 3  # conv_out


def time_cuda(fn, iters, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def vae_latent(cfg, dev):
    g = torch.Generator(device=dev).manual_seed(5)
    return torch.randn(1, 16, cfg["res"] // 8, cfg["res"] // 8, device=dev, generator=g) * 1.2


def measure_vae_ours(cfg, dev):
    """SURVEY.md 8f N4 beside the headline metric: one AutoEncoder.decode of the config's image size through this package's
    kernels (seeded synthetic VAE weights)."""
    from flux_fp8_api_b200 import _cabi as cabi, autoencoder as A, pipeline as PL

    ae = A.AutoEncoder(A.AutoEncoderParams(**VAE_PARAMS))
    PL.init_synthetic_vae_weights(ae, seed=77)
    ae = ae.to(dev, torch.bfloat16).eval()
    z = vae_latent(cfg, dev)
    with torch.inference_mode():
        ae.decode(z)
        n0 = cabi.LAUNCHES
        ae.decode(z)
        calls = cabi.LAUNCHES - n0
        ms = time_cuda(lambda: ae.decode(z), 5)
    fl = vae_decode_flops(cfg["res"])
    return {"workload": f"AutoEncoder.decode, 1 x {cfg['res']}x{cfg['res']} (modules/autoencoder.py:330-333 under bf16 autocast)",
            "ms": ms, "tflops": fl / (ms * 1e-3) / 1e12, "flop": fl, "c_abi_calls": calls, "dtype": "bf16, fp32 accumulate"}


def measure_text_encoders(dev):
    """SURVEY.md 8f N4 beside the headline metric: the two text encoders of a request (t5-v1_1-xxl encoder, 512 tokens;
    clip-vit-large-patch14 text tower, 77 tokens; seeded weights) through conditioner.accelerate, and the Hugging Face
    modules themselves (what the reference's HFEmbedder runs, modules/conditioner.py:109-113) on the same GPU."""
    import math

    from transformers import CLIPTextConfig, CLIPTextModel, T5Config, T5EncoderModel

    from flux_fp8_api_b200 import conditioner as CD

    def init(m, gain):
        g = torch.Generator(device=dev).manual_seed(17)
        with torch.no_grad():
            for k, p in sorted(m.state_dict().items()):
                if p.dtype.is_floating_point:
                    if "norm" in k and k.endswith("weight"):
                        p.copy_(1.0 + 0.1 * torch.randn(p.shape, device=dev, generator=g))
                    else:
                        p.copy_(torch.randn(p.shape, device=dev, generator=g) * (gain / math.sqrt(p.shape[-1]) if p.dim() > 1 else 0.05))

    out = {}
    with torch.device(dev):
        models = (("t5-v1_1-xxl encoder, 512 tokens", lambda: T5EncoderModel(T5Config(
                       vocab_size=32128, d_model=4096, d_kv=64, d_ff=10240, num_layers=24, num_heads=64, dropout_rate=0.0,
                       feed_forward_proj="gated-gelu", is_encoder_decoder=False, use_cache=False, tie_word_embeddings=False)), 512, 0.5),
                  ("clip-vit-large-patch14 text, 77 tokens", lambda: CLIPTextModel(CLIPTextConfig(
                       vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12, num_attention_heads=12,
                       max_position_embeddings=77, hidden_act="quick_gelu", eos_token_id=2, bos_token_id=0, pad_token_id=1)), 77, 1.0))
        for name, build, S, gain in models:
            m = build().to(torch.bfloat16).eval()
            init(m, gain)
            ids = torch.randint(3, 30000, (1, S), device=dev)
            ours = CD.accelerate(m)
            with torch.inference_mode():
                ms = time_cuda(lambda: ours(input_ids=ids, attention_mask=None, output_hidden_states=False), 5)
                ms_hf = time_cuda(lambda: m(input_ids=ids, attention_mask=None, output_hidden_states=False), 5)
            out[name] = {"ms": ms, "hugging_face_ms": ms_hf, "speedup_ours_over_hugging_face": ms_hf / ms}
            del m, ours
            torch.cuda.empty_cache()
    return out


def measure_vae_reference(ref, cfg, dev):
    """The unmodified reference AutoEncoder on the same GPU, as flux_pipeline.py:431-434 runs it."""
    from oracle import vae_oracle as V

    if ref.ae is None:
        return None
    rae = ref.ae.AutoEncoder(ref.ae.AutoEncoderParams(**VAE_PARAMS))
    rae.load_state_dict(V.synthetic_state(rae, seed=77), strict=False)
    rae = rae.to(dev, torch.bfloat16).eval()
    z = vae_latent(cfg, dev)

    def run():
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16, cache_enabled=False):
            return rae.decode(z)

    with torch.inference_mode():
        return time_cuda(run, 3)


def run_reference_gpu_arm(args, cfg):
    """--impl reference-gpu: the unmodified reference fp8 modules on cuda:0 -- F8Linear (torch._scaled_mm), eager
    elementwise ops, F.scaled_dot_product_attention -- in the denoise loop of flux_pipeline.py:627-651; mode `compiled`
    first does what FluxPipeline.compile does with compile_blocks=True (block.compile() on every block, :215-219)."""
    import types

    from oracle import ref_loader as R

    if not R.available():
        print(json.dumps({"impl": "reference-gpu", "unavailable": "oracle/_ref not staged"}), flush=True)
        return
    ref = R.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L, S = geometry(cfg)
    params = dict(in_channels=64, vec_in_dim=768, context_in_dim=4096, hidden_size=3072, mlp_ratio=4.0, num_heads=24,
                  depth=19, depth_single_blocks=38, axes_dim=[16, 56, 56], theta=10_000, qkv_bias=True,
                  guidance_embed=cfg["guidance"])
    spec = R.model_spec(ref, params, False, cfg["qmod"], False)
    t0 = time.perf_counter()
    with torch.device(dev), torch.inference_mode():
        net = ref.fm.Flux(spec, dtype=torch.bfloat16).to(torch.bfloat16)
        init_reference_weights(ref, net)
    net.eval()
    ref.f8.quantize_flow_transformer_and_dispatch_float8(
        net, dev, offload_flow=False, swap_linears_with_cublaslinear=False, flow_dtype=torch.bfloat16,
        quantize_modulation=cfg["qmod"], quantize_flow_embedder_layers=False)
    g = torch.Generator(device=dev).manual_seed(0)
    side = cfg["res"] // 16
    from oracle import flux_oracle as O

    req = dict(img=torch.randn(1, L, 64, device=dev, generator=g).to(torch.bfloat16),
               img_ids=O.make_img_ids(1, side, side, torch.bfloat16, dev),
               txt=(0.15 * torch.randn(1, cfg["text_len"], 4096, device=dev, generator=g)).to(torch.bfloat16),
               txt_ids=torch.zeros(1, cfg["text_len"], 3, dtype=torch.bfloat16, device=dev),
               y=torch.randn(1, 768, device=dev, generator=g).to(torch.bfloat16),
               guidance=torch.full((1,), 3.5, device=dev, dtype=torch.bfloat16) if cfg["guidance"] else None)
    sched = O.get_schedule(28, L, shift=cfg["guidance"])

    def loop(k):
        img = req["img"]
        t_vec = torch.full((1,), sched[0], dtype=img.dtype, device=dev)
        for i in range(k):
            t_curr, t_prev = sched[i % 28], sched[i % 28 + 1]
            t_vec.fill_(t_curr)
            pred = net(img=img, img_ids=req["img_ids"], txt=req["txt"], txt_ids=req["txt_ids"], y=req["y"],
                       timesteps=t_vec, guidance=req["guidance"])
            img = img + (t_prev - t_curr) * pred
        return img

    err = None
    with torch.inference_mode():
        loop(14)  # > 12 calls: freezes every F8Linear input scale (float8_quantize.py:238-246)
        assert R.all_frozen(ref, net)
        if args.mode == "compiled":
            try:
                for block in list(net.double_blocks) + list(net.single_blocks):
                    block.compile()
                loop(2)
            except Exception as ex:  # noqa: BLE001
                err = f"{type(ex).__name__}: {str(ex)[:300]}"
        setup_s = time.perf_counter() - t0
        if err is None:
            loop(max(3, args.warmup))
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            loop(args.steps)
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / args.steps
    line = {"impl": "reference-gpu", "mode": args.mode, "metric": metric_name(cfg), "unit": "it/s", "steps": args.steps,
            "warmup": max(3, args.warmup), "setup_s": round(setup_s, 1), "torch": torch.__version__,
            "config": config_block(cfg, args.config, 1)}
    if args.mode == "eager":
        try:
            del net
            torch.cuda.empty_cache()
            line["vae_decode_ms"] = measure_vae_reference(ref, cfg, dev)
        except Exception as ex:  # noqa: BLE001
            line["vae_decode_error"] = f"{type(ex).__name__}: {str(ex)[:200]}"
    if err is None:
        line.update(value=1000.0 / ms, ms_per_step=ms)
    else:
        line.update(value=None, error=err)
    print(json.dumps(line), flush=True)


def gpu_reference_block(args, timeout_eager=420, timeout_compiled=900):
    """Run the reference-gpu arm in child processes (its 24 GB bf16 build and torch.compile state stay out of this
    process; a failure or time-out of the reference cannot take the bench down)."""
    out = {}
    modes = {"eager": ["eager"], "compiled": ["compiled"], "both": ["eager", "compiled"], "none": []}[args.gpu_reference]
    for mode in modes:
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference-gpu", "--mode", mode, "--config", args.config,
               "--steps", str(min(args.steps, 20)), "--warmup", str(args.warmup)]
        env = dict(os.environ)
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        t0 = time.perf_counter()
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, env=env,
                               timeout=timeout_eager if mode == "eager" else timeout_compiled)
            lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            out[mode] = json.loads(lines[-1]) if lines else {"error": (r.stderr or "no output")[-300:]}
        except subprocess.TimeoutExpired:
            out[mode] = {"error": f"timed out after {timeout_eager if mode == 'eager' else timeout_compiled} s"}
        except Exception as ex:  # noqa: BLE001
            out[mode] = {"error": repr(ex)[:300]}
        out[mode]["wall_s"] = round(time.perf_counter() - t0, 1)
        out[mode].pop("config", None)
    return out


# ------------------------------------------------------------------------------------------------
def synthetic_lora(params, rank=16, seed=11):
    """SURVEY.md section 8(d), c4: rank-16 LoRA over every block linear, BFL key layout, lora_down ~ N(0, 1/16),
    lora_up ~ N(0, 0.01^2)."""
    g = torch.Generator().manual_seed(seed)
    D, MLP = params.hidden_size, int(params.hidden_size * params.mlp_ratio)
    shapes = {}
    for i in range(params.depth):
        for s in ("img", "txt"):
            shapes[f"double_blocks.{i}.{s}_attn.qkv"] = (3 * D, D)
            shapes[f"double_blocks.{i}.{s}_attn.proj"] = (D, D)
            shapes[f"double_blocks.{i}.{s}_mlp.0"] = (MLP, D)
            shapes[f"double_blocks.{i}.{s}_mlp.2"] = (D, MLP)
    for i in range(params.depth_single_blocks):
        shapes[f"single_blocks.{i}.linear1"] = (3 * D + MLP, D)
        shapes[f"single_blocks.{i}.linear2"] = (D, D + MLP)
    sd = {}
    for key, (n, k) in shapes.items():
        sd[f"{key}.lora_A.weight"] = (torch.randn(rank, k, generator=g) / 16.0).to(torch.bfloat16)   # "down"
        sd[f"{key}.lora_B.weight"] = (torch.randn(n, rank, generator=g) * 0.01).to(torch.bfloat16)   # "up"
    return sd


def measure_fp8_peak(ops, cabi, dev):
    """The tcgen05 kind::f8f6f4 ceiling of THIS box: fluxb200_fp8_mma_probe = the bare MMA loop of the product GEMM tiling
    (cta_group::2, M = 256, N = 256, K = 32), operands resident in shared memory, no TMA / epilogue / global traffic.
    burst = best single ~0.3 ms launch after a pause; sustained = back-to-back launches for ~1.5 s (the power-capped
    regime the step runs in)."""
    import ctypes as C

    lib = cabi.load()
    flops = C.c_double(0.0)

    def launch(tiles):
        cabi.check(lib.fluxb200_fp8_mma_probe(tiles, C.byref(flops), cabi.stream_ptr()), "fluxb200_fp8_mma_probe")
        return flops.value

    for _ in range(2):
        launch(40)
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(8):
        time.sleep(0.05)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        f_burst = launch(40)
        e.record()
        torch.cuda.synchronize()
        best = min(best, s.elapsed_time(e))
    reps = max(8, int(1500.0 / (best * 10)))
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        f_sus = launch(400)
    e.record()
    torch.cuda.synchronize()
    sustained_ms = s.elapsed_time(e) / reps
    return {"fp8_tflops_burst": f_burst / (best * 1e-3) / 1e12, "fp8_tflops_sustained": f_sus / (sustained_ms * 1e-3) / 1e12,
            "burst_launch_ms": best, "sustained_launches": reps, "sustained_launch_ms": sustained_ms,
            "how": "fluxb200_fp8_mma_probe: tcgen05.mma.cta_group::2.kind::f8f6f4 M=256 N=256 K=32 issued back to back on "
                   "all 74 SM pairs, operands resident in shared memory (no TMA, no epilogue), CUDA events"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=28)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--mode", default="eager", choices=["eager", "compiled"], help="--impl reference-gpu only")
    ap.add_argument("--gpu-reference", default="both", choices=["none", "eager", "compiled", "both"],
                    help="time the unmodified reference modules on the same GPU after our arm (rank 0, N=1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-vae", action="store_true",
                    help="skip the VAE decode and text-encoder measurements (SURVEY 8f N4) beside the metric")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the latent of the last timed step as DIR/latent.npy (float32; --impl ours only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return
    if args.impl == "reference-gpu":
        if rank == 0:
            run_reference_gpu_arm(args, cfg)
        return
    if args.warmup < 3:
        args.warmup = 3

    from flux_fp8_api_b200 import _cabi, model as M, ops, parallel as PAR, pipeline as PL

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback "
                         "(use --impl reference for the CPU baseline arm)")
    rank, local_rank, world = PAR.init_distributed("nccl")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ops.device_check()
    peaks, peaks_src = measured_peaks()
    L_IMG, S_TOTAL = geometry(cfg)
    F8_FLOPS, ATTN_FLOPS, MOD_BF16_FLOPS = algorithmic_flops(cfg)

    # ---- model: synthetic weights -> reference quantisation flow -> calibrate on rank 0 -> one broadcast
    spec = (M.flux_dev_spec if cfg["guidance"] else M.flux_schnell_spec)(quantize_modulation=cfg["qmod"])
    net = PL.build_synthetic_flux(spec, dev, seed=1234)
    req = PL.synthetic_request(spec.params, cfg["res"], cfg["res"], 1, cfg["text_len"], dev, seed=0, sample_offset=rank)
    if not cfg["guidance"]:
        req["guidance"] = None
    lora_info = None
    if cfg["lora"]:
        t0 = time.perf_counter()
        net.load_lora(synthetic_lora(spec.params), scale=1.0, name="synthetic-rank16")
        torch.cuda.synchronize()
        lora_info = {"rank": 16, "layers": 19 * 8 + 38 * 2, "fuse_s": round(time.perf_counter() - t0, 2),
                     "how": "Flux.load_lora -> on-device fuse (fluxb200_lora_fuse) before calibration"}
    bcast_bytes, bcast_ms = 0, 0.0
    if rank == 0:
        if cfg["guidance"]:
            PL.calibrate(net, req, num_steps=13, shift=True)
        else:  # schnell: 4 runs of 4 steps, mirroring flux_pipeline.py:207-210
            for _ in range(4):
                PL.denoise(net, dict(req), PL.get_schedule(4, L_IMG, shift=False))
    if world > 1:
        if rank != 0:  # allocate scale buffers so shapes agree, then receive rank 0's state
            for m in net.modules():
                if isinstance(m, M.F8Linear):
                    z = torch.zeros((), dtype=torch.float32, device=dev)
                    m.input_scale, m.input_scale_reciprocal = z.clone(), z.clone()
        torch.cuda.synchronize()
        PAR.barrier()
        t0 = time.perf_counter()
        bcast_bytes = PAR.broadcast_state(net, src=0)
        torch.cuda.synchronize()
        bcast_ms = (time.perf_counter() - t0) * 1e3
        PAR.frozen_flags_sync(net)
    assert PL.all_frozen(net)

    sess = PL.DenoiseSession(net, req, use_graph=not args.no_graph)
    sched = PL.get_schedule(max(cfg["num_steps"], 1), L_IMG, shift=cfg["guidance"])
    nsch = len(sched) - 1

    # launches per step (counted while running one eager-launch step)
    before = _cabi.LAUNCHES
    with torch.inference_mode():
        tv = torch.full((1,), sched[0], dtype=torch.bfloat16, device=dev)
        net(img=req["img"], img_ids=req["img_ids"], txt=req["txt"], txt_ids=req["txt_ids"], y=req["y"], timesteps=tv,
            guidance=req["guidance"])
    launches_per_step = _cabi.LAUNCHES - before

    def timed_loop(step_fn, steps):
        torch.cuda.synchronize()
        PAR.barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = step_fn(steps)
        e.record()
        torch.cuda.synchronize()
        PAR.barrier()
        return PAR.max_over_ranks(s.elapsed_time(e), dev), out

    # ---- value: latents resident in HBM
    def device_steps(k):
        img = req["img"]
        for i in range(k):
            img = sess.step_device(img, sched[i % nsch], sched[i % nsch + 1])
        return img

    device_steps(args.warmup)
    with ClockSampler(local_rank) as clocks:
        ms_total, latent = timed_loop(device_steps, args.steps)
    clock_info = clocks.summary()
    if args.dump_outputs:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "latent.npy" if world == 1 else f"latent_rank{rank}.npy"
        np.save(os.path.join(args.dump_outputs, name), latent.float().cpu().numpy())
    del latent
    ms_per_step = ms_total / args.steps
    value = world * 1000.0 / ms_per_step

    # ---- e2e: host buffers in, host buffers out, every step
    host_img = torch.empty(req["img"].shape, dtype=req["img"].dtype, pin_memory=True)
    host_img.copy_(req["img"])

    def host_steps(k):
        h = host_img
        for i in range(k):
            h = sess.step_host(h, sched[i % nsch], sched[i % nsch + 1])
        return h

    host_steps(2)
    e2e_ms = timed_loop(host_steps, args.steps)[0] / args.steps
    e2e_value = world * 1000.0 / e2e_ms

    # ---- roofline: CUDA events around every kernel launch of an eager-launch pass + the measured FP8 ceiling
    roof = None
    if rank == 0:
        fp8_probe = measure_fp8_peak(ops, _cabi, dev)
        ops.KERNEL_TIMELINE = []
        eager = PL.DenoiseSession(net, req, use_graph=False)
        with torch.inference_mode():
            for i in range(3):
                if i == 1:
                    ops.KERNEL_TIMELINE.clear()
                eager.step_device(req["img"], sched[0], sched[1])
        torch.cuda.synchronize()
        tl, ops.KERNEL_TIMELINE = ops.KERNEL_TIMELINE, None
        agg = {}
        for kind, flops, s, e, *_ in tl:
            a = agg.setdefault(kind, [0.0, 0.0, 0])
            a[0] += flops
            a[1] += s.elapsed_time(e)
            a[2] += 1
        gf, gms, gn = agg["f8_gemm"]
        af, ams, an = agg["attention"]
        hbm = {}
        for kind in ("ln_mod_quant", "modulation_batched"):
            if kind in agg:
                bts, ms_, cnt = agg[kind]
                hbm[kind] = {"achieved": bts / (ms_ * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": bts / (ms_ * 1e-3) / 1e9 / peaks["hbm_gbs"], "launches_per_step": cnt // 2,
                             "ms_per_step": ms_ / 2}
        fp8_peak = fp8_probe["fp8_tflops_sustained"]
        # The event-timed pass launches eagerly: the host-side gaps between its launches let the power-capped GPU
        # clock higher than it does inside the back-to-back CUDA-graph step.  `achieved` therefore charges the kernel
        # its SHARE of the event-timed launches applied to the timed graph step (the in-step rate); the raw
        # event-timed rate is reported beside it.
        timed_ms = sum(a[1] for a in agg.values()) / 2
        gemm_share = (gms / 2) / timed_ms
        attn_share = (ams / 2) / timed_ms
        gemm_ms_in_step = gemm_share * ms_per_step
        attn_ms_in_step = attn_share * ms_per_step
        achieved = (gf / 2) / (gemm_ms_in_step * 1e-3) / 1e12
        attn_achieved = (af / 2) / (attn_ms_in_step * 1e-3) / 1e12
        traffic, traffic_src = gemm_traffic_per_launch()
        roof = {
            "bound": "tensor", "kernel": "f8_gemm_kernel (tcgen05 kind::f8f6f4)", "achieved": achieved,
            "peak": fp8_peak, "unit": "TFLOP/s", "frac": achieved / fp8_peak,
            "traffic": traffic if args.config == "c2" else None, "traffic_source": traffic_src,
            "peak_source": "measured in this run on this GPU: sustained tcgen05 kind::f8f6f4 issue rate of the GEMM "
                           "kernel's own tiling (fluxb200_fp8_mma_probe); MEASURED_PEAKS.json has no fp8 row",
            "fp8_peak_probe": fp8_probe,
            "frac_of_burst_peak": achieved / fp8_probe["fp8_tflops_burst"],
            "frac_of_2x_bf16_sustained": achieved / (2.0 * peaks["bf16_tflops_sustained"]),
            "frac_of_nominal_4500": achieved / 4500.0,
            "method": "algorithmic flops of all GEMM launches of a step / (share of the CUDA-event-timed launch time "
                      "x graph-replay ms per step)",
            "achieved_event_timed_eager": gf / (gms * 1e-3) / 1e12,
            "launches_per_step": gn // 2, "gemm_ms_per_step": gemm_ms_in_step, "gemm_share_of_step": gemm_share,
            "gemm_ms_per_step_event_timed_eager": gms / 2,
            "attention": {"achieved": attn_achieved, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                          "frac": attn_achieved / peaks["bf16_tflops_sustained"],
                          "peak_source": f"bf16_tflops_sustained, {peaks_src}",
                          "achieved_event_timed_eager": af / (ams * 1e-3) / 1e12,
                          "launches_per_step": an // 2, "ms_per_step": attn_ms_in_step, "share_of_step": attn_share},
            "hbm_kernels": hbm,
            "step_tensor_frac": (F8_FLOPS / (fp8_peak * 1e12) + ATTN_FLOPS / (peaks["bf16_tflops_sustained"] * 1e12))
                                / (ms_per_step * 1e-3),
            "fp8_pipe_util_nominal": F8_FLOPS / (ms_per_step * 1e-3) / 4.5e15,
            "fp8_pipe_util_measured_peak": F8_FLOPS / (ms_per_step * 1e-3) / (fp8_peak * 1e12),
        }

    # ---- the unmodified reference on the same GPU (rank 0, N=1 only): the GPU-vs-GPU number SURVEY 8(d) asks for
    gpu_ref = None
    h2d_bytes, d2h_bytes = sess.h2d_bytes_per_step, sess.d2h_bytes_per_step
    vae = None
    text = None
    if rank == 0 and world == 1 and not args.no_vae:
        vae = measure_vae_ours(cfg, dev)
        try:
            text = measure_text_encoders(dev)
        except Exception as ex:  # noqa: BLE001  (transformers missing / changed: the headline line must still print)
            text = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
    if rank == 0 and world == 1 and args.gpu_reference != "none":
        del sess
        torch.cuda.empty_cache()
        gpu_ref = gpu_reference_block(args)
        for mode, r in gpu_ref.items():
            if r.get("value"):
                r["speedup_ours_over_reference"] = value / r["value"]
        ref_vae = (gpu_ref.get("eager") or {}).get("vae_decode_ms")
        if vae is not None and ref_vae:
            vae["reference_gpu_ms"] = ref_vae
            vae["speedup_ours_over_reference"] = ref_vae / vae["ms"]

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        m = cpu_reference_measure(cfg, 2, 1)
        cpu = {"value": m["value"], "unit": "it/s", "cores": m["threads"], "kind": m["kind"],
               "sample": f"2 x (1 DoubleStreamBlock + 2 SingleStreamBlocks, bf16, S={S_TOTAL}) through the "
                         f"{'unmodified reference modules' if m['kind'] == 'reference' else 'oracle port'} = 1/19 of a "
                         f"step each; step = 19 x {m['sample_s']:.3f} s"}

    if rank == 0:
        line = {
            "metric": metric_name(cfg), "value": value, "unit": "it/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "fp8 (e5m2 activations x e4m3 weights, fp32 accumulate; bf16 attention)" + (
                "" if cfg["qmod"] else "; bf16 modulation"),
            "data": "synthetic",
            "config": config_block(cfg, args.config, world, {
                "cuda_graph": not args.no_graph, "weights": "seeded synthetic, reference quantise+calibrate flow",
                "lora": lora_info}),
            "e2e": {"value": e2e_value, "unit": "it/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
            "gpu_launches": launches_per_step * args.steps,
            "gpu_launches_per_step": launches_per_step,
            "clocks": clock_info,
            "roofline": roof,
            "gpu_reference": gpu_ref,
            "vae_decode": vae,
            "text_encoders": text,
            "cpu_baseline": cpu,
            "broadcast": {"bytes": bcast_bytes, "ms": bcast_ms},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
