"""Mint the stored outputs of the UNMODIFIED reference that the parity tests compare against, so that the tests run
from a plain checkout (the reference itself is never part of the repository):

    tests/golden/reference_surface.json   signatures, parameter fields and state-dict shapes of the reference's classes
    tests/golden/reference_flux_full.pt   full-depth Flux (every config of tests/test_gpu_reference.py): the reference's
                                          calibrated input scales, byte checksums of its state and of the forward's
                                          inputs, a sample of its output and its own SDPA-backend-to-backend spread
    tests/golden/reference_vae_full.pt    full-size VAE decode / encode: byte checksums of the state and the input,
                                          samples of the reference's bf16-autocast and fp32 outputs and the
                                          whole-tensor distance between the two
    tests/golden/reference_tiny_gpu.pt    the reference container running a save_prequantized file of the tiny model

    python oracle/reference_golden.py surface DIR      # CPU, needs oracle/_ref (python oracle/fetch_ref.py)
    python oracle/reference_golden.py gpu DIR          # B200, needs oracle/_ref

TEST INFRASTRUCTURE ONLY.  `sample` and `state_bytesum` are shared with the tests, which apply them to this package's
outputs and inputs.  The first m elements of sample(t, n) are sample(t, m), so a stored sample may be cut short.
"""
from __future__ import annotations

import dataclasses
import inspect
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BF16 = torch.bfloat16
DEV = "cuda"

FLUX_SAMPLES = 8192
VAE_SAMPLES = 4096
SAMPLE_STRIDE = 1_000_003  # prime, coprime to the size of every sampled tensor

# name: (resolution, text_len, guidance_embed, quantize_modulation, batch, activation fp8 dtype)
FLUX_CONFIGS = {
    "c2-dev-1024": (1024, 512, True, True, 1, torch.float8_e5m2),
    "c2-dev-1024-e4m3": (1024, 512, True, True, 1, torch.float8_e4m3fn),
    "c3-schnell-1024": (1024, 256, False, True, 1, torch.float8_e5m2),
    "c4-dev-768": (768, 512, True, True, 2, torch.float8_e5m2),
    "c5-dev-1536-bf16mod": (1536, 512, True, False, 1, torch.float8_e5m2),
}

VAE_PARAMS = dict(resolution=256, in_channels=3, ch=128, out_ch=3, ch_mult=[1, 2, 4, 4], num_res_blocks=2, z_channels=16,
                  scale_factor=0.3611, shift_factor=0.1159)
# name: (state seed, latent seed, batch, height, width)
VAE_DECODE_CASES = {
    "decode-1024": (77, 78, 1, 1024, 1024),
    "decode-768": (77, 78, 1, 768, 768),
    "decode-1536": (77, 78, 1, 1536, 1536),
    "decode-5x128x192": (91, 92, 5, 128, 192),
    "decode-2x720x1280": (91, 92, 2, 720, 1280),
}
VAE_ENCODE_SEEDS = (93, 94)  # state seed, image seed; 1 x 1024 x 1024


def sample(t: torch.Tensor, n: int) -> torch.Tensor:
    """n elements of t at the flat positions k * SAMPLE_STRIDE mod t.numel(), k = 0 .. n-1 (all of t when it is
    smaller), on the CPU.  The stride is coprime to the size, so the positions are distinct, and it is not a multiple of
    any row width, so they cover every row, column and channel rather than lining up on a few columns."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= n:
        return flat.cpu().clone()
    if math.gcd(SAMPLE_STRIDE, flat.numel()) != 1:
        raise ValueError(f"sample: {flat.numel()} elements share a factor with the stride {SAMPLE_STRIDE}")
    idx = (torch.arange(n, dtype=torch.int64, device=flat.device) * SAMPLE_STRIDE) % flat.numel()
    return flat[idx].cpu()


def state_bytesum(sd) -> int:
    """Exact, order-independent checksum of a state dict: the byte sum of every tensor, weighted by its rank in the
    sorted key list (so a tensor under the wrong key changes it)."""
    total = 0
    for i, k in enumerate(sorted(sd)):
        v = sd[k]
        if v is None:
            continue
        total += (i + 1) * int(v.detach().contiguous().reshape(-1).view(torch.uint8).to(torch.int64).sum().item())
    return total


def f8_names(net, f8_class) -> list:
    return [n for n, m in net.named_modules() if isinstance(m, f8_class)]


def vae_decode_latent(seed, B, height, width):
    return torch.randn(B, 16, height // 8, width // 8, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed)) * 1.2


def vae_encode_image(seed):
    return (torch.rand(1, 3, 1024, 1024, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed)) * 2 - 1).to(BF16)


def flux_call(name):
    """(params, request, the free-running forward's arguments) of a full-depth config; shared with the tests."""
    from flux_fp8_api_b200 import model as M, pipeline as PL

    res, text_len, guidance, qmod, batch, in_dt = FLUX_CONFIGS[name]
    params = M.FluxParams(guidance_embed=guidance)
    req = PL.synthetic_request(params, res, res, batch, text_len, DEV, seed=3)
    if not guidance:
        req["guidance"] = None
    sched = PL.get_schedule(28, req["img"].shape[1], shift=guidance)
    t = torch.full((batch,), sched[3], dtype=BF16, device=DEV)
    call = dict(img=req["img"], img_ids=req["img_ids"], txt=req["txt"], txt_ids=req["txt_ids"], timesteps=t, y=req["y"],
                guidance=req["guidance"])
    return params, req, call


# ------------------------------------------------------------------------------------------------
def _params(fn):
    return [[p.name, int(p.kind), repr(p.default) if not isinstance(p.default, torch.dtype) else str(p.default)]
            for p in inspect.signature(fn).parameters.values()]


def surface(out_dir):
    from oracle import ref_loader as R

    ref = R.load()
    sig = {}
    for name in ("F8Linear", "recursive_swap_linears", "quantize_flow_transformer_and_dispatch_float8"):
        sig[f"float8_quantize.{name}"] = _params(getattr(ref.f8, name))
    for name in ("attention", "rope", "apply_rope", "EmbedND", "QKNorm", "Modulation", "DoubleStreamBlock",
                 "SingleStreamBlock"):
        sig[f"flux_model.{name}"] = _params(getattr(ref.fm, name))
    for meth in ("get_lora", "has_lora", "load_lora", "unload_lora", "from_pretrained", "forward"):
        sig[f"flux_model.Flux.{meth}"] = _params(getattr(ref.fm.Flux, meth))
    ae_init = {name: [p.name for p in inspect.signature(getattr(ref.ae, name).__init__).parameters.values()]
               for name in ("AttnBlock", "ResnetBlock", "Upsample", "Downsample", "Encoder", "Decoder", "DiagonalGaussian",
                            "AutoEncoder")}
    ae_params = dict(resolution=64, in_channels=3, ch=64, out_ch=3, ch_mult=[1, 2, 4, 4], num_res_blocks=2, z_channels=16,
                     scale_factor=0.3611, shift_factor=0.1159)
    ae_state = {k: list(v.shape) for k, v in ref.ae.AutoEncoder(ref.ae.AutoEncoderParams(**ae_params)).state_dict().items()}
    blob = {"signatures": sig, "autoencoder_init": ae_init,
            "autoencoder_params_fields": sorted(ref.ae.AutoEncoderParams.model_fields),
            "autoencoder_state_shapes": {"params": ae_params, "shapes": ae_state}}
    with open(os.path.join(out_dir, "reference_surface.json"), "w") as f:
        json.dump(blob, f, indent=0, sort_keys=True)


# ------------------------------------------------------------------------------------------------
def _stats(a, b):
    d = (a.float() - b.float()).abs()
    return [d.mean().item(), d.max().item()]


def gpu_flux(ref):
    from torch.nn.attention import SDPBackend, sdpa_kernel

    from flux_fp8_api_b200 import model as M, pipeline as PL
    from oracle import ref_loader as R

    backends = [("cudnn", SDPBackend.CUDNN_ATTENTION), ("flash", SDPBackend.FLASH_ATTENTION),
                ("efficient", SDPBackend.EFFICIENT_ATTENTION), ("math", SDPBackend.MATH)]
    out = {}
    for name, (res, text_len, guidance, qmod, batch, in_dt) in FLUX_CONFIGS.items():
        params, req, call = flux_call(name)
        seed_net = PL.build_synthetic_flux(M.FluxSpec(params=params, quantize_modulation=qmod), DEV, seed=7, quantize=False)
        theirs = R.build_reference_flux(ref, dataclasses.asdict(params), seed_net.state_dict(), DEV,
                                        quantize_modulation=qmod, input_float8_dtype=in_dt)
        del seed_net
        torch.cuda.empty_cache()
        L = req["img"].shape[1]
        PL.denoise(theirs, dict(req), PL.get_schedule(13, L, shift=guidance))  # the reference's own calibration
        assert R.all_frozen(ref, theirs)
        names = f8_names(theirs, ref.f8.F8Linear)
        mods = dict(theirs.named_modules())
        scales = torch.stack([torch.stack([mods[n].input_scale.float().reshape(()), mods[n].input_scale_reciprocal.float().reshape(())])
                              for n in names]).cpu()
        with torch.inference_mode():
            y_ref = theirs(**call)
            floor = {}
            for bname, backend in backends:
                try:
                    with sdpa_kernel([backend]):
                        floor[bname] = _stats(theirs(**call), y_ref)
                except RuntimeError:
                    continue
        out[name] = {"n_f8": len(names), "scales": scales, "state_bytesum": state_bytesum(theirs.state_dict()),
                     "inputs_bytesum": state_bytesum(call),
                     "y_shape": list(y_ref.shape), "y_ref": sample(y_ref, FLUX_SAMPLES), "ref_vs_ref": floor}
        print(name, {k: v for k, v in out[name].items() if k not in ("scales", "y_ref")}, flush=True)
        del theirs, y_ref
        torch.cuda.empty_cache()
    return out


def gpu_vae(ref):
    from oracle import vae_oracle as V

    out = {}

    def build(seed, prefixes):
        rae = ref.ae.AutoEncoder(ref.ae.AutoEncoderParams(**VAE_PARAMS))
        sd = V.synthetic_state(rae, seed=seed, prefixes=prefixes)
        rae.load_state_dict(sd, strict=prefixes != ("decoder.",))
        return rae.to(DEV, BF16).eval(), state_bytesum(sd)

    for name, (sseed, zseed, B, height, width) in VAE_DECODE_CASES.items():
        rae, sd_sum = build(sseed, ("decoder.",))
        z = vae_decode_latent(zseed, B, height, width)
        with torch.inference_mode():
            with torch.autocast(device_type="cuda", dtype=BF16, cache_enabled=False):  # flux_pipeline.py:431-434
                y_ref = rae.decode(z)
            y32 = rae.float().decode(z)
        floor = (y_ref.float() - y32).abs()
        out[name] = {"state_bytesum": sd_sum, "inputs_bytesum": state_bytesum({"z": z}),
                     "shape": list(y_ref.shape), "y_ref": sample(y_ref, VAE_SAMPLES), "y32": sample(y32, VAE_SAMPLES),
                     "floor_mean": floor.mean().item(), "floor_max": floor.max().item()}
        print(name, out[name]["shape"], out[name]["floor_mean"], out[name]["floor_max"], flush=True)
        del rae, y_ref, y32, floor
        torch.cuda.empty_cache()
    rae, sd_sum = build(VAE_ENCODE_SEEDS[0], ("decoder.", "encoder."))
    img = vae_encode_image(VAE_ENCODE_SEEDS[1])
    with torch.inference_mode():
        with torch.autocast(device_type="cuda", dtype=BF16, cache_enabled=False):
            m_ref = rae.encoder(img)
        m32 = rae.float().encoder(img.float())
    floor = (m_ref.float() - m32).abs()
    out["encode-1024"] = {"state_bytesum": sd_sum, "inputs_bytesum": state_bytesum({"img": img}),
                          "shape": list(m_ref.shape), "m_ref": sample(m_ref, VAE_SAMPLES), "m32": sample(m32, VAE_SAMPLES),
                          "floor_mean": floor.mean().item(), "floor_max": floor.max().item()}
    print("encode-1024", out["encode-1024"]["floor_mean"], out["encode-1024"]["floor_max"], flush=True)
    return out


def gpu_tiny_prequantized(ref, tmp_path):
    """The reference container loads a save_prequantized file of the tiny golden model the way util.load_flow_model does
    (load_sft + load_state_dict(assign=True), util.py:245-256) and runs it on its library kernels."""
    from safetensors.torch import load_file

    from flux_fp8_api_b200 import model as M, pipeline as PL
    from oracle import ref_loader as R

    gold = torch.load(os.path.join(ROOT, "tests", "golden", "flux_tiny.pt"))
    spec = M.FluxSpec(params=M.FluxParams(**gold["tiny"]), prequantized_flow=True)
    with torch.device(DEV):
        net = M.Flux(spec, dtype=BF16)
    net.load_state_dict({k: v.to(DEV) for k, v in gold["state"].items()}, strict=True, assign=True)
    path = os.path.join(tmp_path, "tiny.f8.safetensors")
    PL.save_prequantized(net.eval(), path, spec)
    with torch.device("meta"):
        theirs = ref.fm.Flux(R.model_spec(ref, gold["tiny"], prequantized_flow=True), dtype=BF16)
    missing, unexpected = theirs.load_state_dict(load_file(path, device="cpu"), strict=False, assign=True)
    assert not missing and not unexpected
    theirs = theirs.to(DEV).eval()
    assert R.all_frozen(ref, theirs)
    with torch.inference_mode():
        y_ref = theirs(**{k: v.to(DEV) for k, v in gold["inputs"].items()})
    return {"y_ref": y_ref.cpu()}


def gpu(out_dir):
    import tempfile

    from oracle import ref_loader as R

    ref = R.load()
    with tempfile.TemporaryDirectory() as tmp:
        torch.save(gpu_tiny_prequantized(ref, tmp), os.path.join(out_dir, "reference_tiny_gpu.pt"))
    torch.save(gpu_vae(ref), os.path.join(out_dir, "reference_vae_full.pt"))
    torch.save(gpu_flux(ref), os.path.join(out_dir, "reference_flux_full.pt"))


if __name__ == "__main__":
    what, out_dir = sys.argv[1], sys.argv[2]
    os.makedirs(out_dir, exist_ok=True)
    {"surface": surface, "gpu": gpu}[what](out_dir)
