"""GPU (-m gpu): parity against the REAL reference, run on the same B200.

The unmodified reference modules (float8_quantize.py, modules/flux_model.py) are staged under oracle/_ref by
oracle/fetch_ref.py and imported through oracle/ref_loader.py -- SURVEY.md section 8(c): "the parity target is the
reference fp8 path run on the B200 box with the same torch" (cuBLASLt `_scaled_mm`, GPU SDPA, GPU layer_norm/rms_norm).

For every BASELINE config (c2..c5) at FULL width and FULL depth (19 double + 38 single blocks):

1. the reference Flux is built from seeded synthetic bf16 weights, quantised with the reference's own
   quantize_flow_transformer_and_dispatch_float8 and calibrated by 13 reference denoise steps; its state_dict() is
   loaded, strict, into this package's Flux (prequantized_flow=True) -- the drop-in claim, checked with real data;
2. LAYER teacher forcing: every reference F8Linear call (304 per forward) and every attention() call (57) is replayed
   through our kernel on the reference's own input -- identical fp8 operand bytes, so what remains is accumulation
   order: bar = bit-identical on >= 90 % of elements, <= 1 bf16 ulp at the output range everywhere;
3. BLOCK teacher forcing: each of the 57 reference blocks hands ITS inputs to our fused block.  Inside a block four
   quantise points turn 1-ulp bf16 differences into flipped e5m2 / e4m3 codes, so the bar cannot be "2 ulp": it is the
   reference's OWN spread on the same block input when it dispatches to a different SDPA backend (reference-vs-reference
   floor, measured in the same hook), and the flip rate of every fp8 operand is measured against the reference's own
   quantised inputs and reported;
4. FREE-RUNNING forward at full depth: ours vs reference, against reference (default SDPA) vs reference (other
   backend): the three must be mutually equidistant.

Results are printed and written to gpurun_out/parity_<config>.json (summarised in profiles/r2_parity_reference.md).

These checks drive the reference's own modules, so they run where oracle/_ref is staged.  The free-running comparison
also runs from a plain checkout, against the reference's output stored by oracle/reference_golden.py
(test_full_depth_output_matches_the_stored_reference_output).
"""
import contextlib
import dataclasses
import json
import os

import pytest
import torch

from oracle import ref_loader as R
from oracle import reference_golden as G

pytestmark = pytest.mark.gpu
needs_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref not staged (python oracle/fetch_ref.py)")
BF16 = torch.bfloat16
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CONFIGS = G.FLUX_CONFIGS  # name: (resolution, text_len, guidance_embed, quantize_modulation, batch, input dtype)


def stats(a, b):
    """(mean |a-b|, max |a-b|, fraction differing) of two same-shape tensors, in fp32."""
    d = (a.float() - b.float()).abs()
    return d.mean().item(), d.max().item(), (d > 0).float().mean().item()


def sdpa_backends():
    from torch.nn.attention import SDPBackend

    return [("cudnn", SDPBackend.CUDNN_ATTENTION), ("flash", SDPBackend.FLASH_ATTENTION),
            ("efficient", SDPBackend.EFFICIENT_ATTENTION), ("math", SDPBackend.MATH)]


@contextlib.contextmanager
def sdpa(backend):
    from torch.nn.attention import sdpa_kernel

    with sdpa_kernel([backend]):
        yield


def build_pair(name):
    """(reference module ns, reference Flux [calibrated], our Flux carrying the reference's state, request, schedule)."""
    from flux_fp8_api_b200 import model as M, pipeline as PL

    res, text_len, guidance, qmod, batch, in_dt = CONFIGS[name]
    ref = R.load()
    params = M.FluxParams(guidance_embed=guidance)
    spec = M.FluxSpec(params=params, quantize_modulation=qmod)
    seed_net = PL.build_synthetic_flux(spec, DEV, seed=7, quantize=False)
    theirs = R.build_reference_flux(ref, dataclasses.asdict(params), seed_net.state_dict(), DEV,
                                    quantize_modulation=qmod, input_float8_dtype=in_dt)
    del seed_net
    torch.cuda.empty_cache()
    req = PL.synthetic_request(params, res, res, batch, text_len, DEV, seed=3)
    if not guidance:
        req["guidance"] = None
    L = req["img"].shape[1]
    PL.denoise(theirs, dict(req), PL.get_schedule(13, L, shift=guidance))  # the reference's own warm-up calibration
    assert R.all_frozen(ref, theirs)
    with torch.device(DEV):
        ours = M.Flux(M.FluxSpec(params=params, prequantized_flow=True, quantize_modulation=qmod), dtype=BF16).to(BF16)
    missing, unexpected = ours.load_state_dict(theirs.state_dict(), strict=True)
    assert not missing and not unexpected
    ours.eval()
    if in_dt != torch.float8_e5m2:
        PL.set_input_float8_dtype(ours, in_dt)
    assert PL.all_frozen(ours)
    return ref, theirs, ours, req, PL.get_schedule(28, L, shift=guidance)


@needs_ref
@pytest.mark.parametrize("name", list(CONFIGS))
def test_full_depth_parity_against_the_reference_on_this_gpu(name, lib):
    from flux_fp8_api_b200 import blocks as B

    ref, theirs, ours, req, sched = build_pair(name)
    in_dt = CONFIGS[name][5]
    t = torch.full((req["img"].shape[0],), sched[3], dtype=BF16, device=DEV)
    call = dict(img=req["img"], img_ids=req["img_ids"], txt=req["txt"], txt_ids=req["txt_ids"], timesteps=t, y=req["y"],
                guidance=req["guidance"])
    report = {"config": name, "layers": [], "attention": [], "blocks": []}
    hooks, state = [], {"live": True}
    xq_of = {}  # reference F8Linear module -> its quantised input of the current block

    # ---- layer teacher forcing: every reference F8Linear / attention call replayed through our kernel ------------
    our_mods = dict(ours.named_modules())

    def lin_hook(qual):
        mine = our_mods[qual]

        def hook(mod, args, out):
            if not state["live"]:
                return
            x = args[0]
            xq_of[mod] = mod.to_fp8_saturated(x, mod.input_scale, mod.input_max_value).to(mod.input_float8_dtype)
            got = mine(x)
            mean, mx, frac = stats(got, out)
            report["layers"].append({"layer": qual, "shape": [int(x.numel() // x.shape[-1]), mod.out_features,
                                                              mod.in_features],
                                     "mean": mean, "max": mx, "frac_diff": frac, "amax": out.abs().max().item()})
        return hook

    for qual, mod in theirs.named_modules():
        if isinstance(mod, ref.f8.F8Linear):
            hooks.append(mod.register_forward_hook(lin_hook(qual)))

    ref_attention = ref.fm.attention

    def attention_probe(q, k, v, pe):
        out = ref_attention(q, k, v, pe=pe)
        if state["live"]:
            got = B.attention(q.contiguous(), k.contiguous(), v.contiguous(), pe)
            mean, mx, frac = stats(got, out)
            report["attention"].append({"mean": mean, "max": mx, "frac_diff": frac, "amax": out.abs().max().item()})
        return out

    ref.fm.attention = attention_probe

    # ---- block teacher forcing + reference-vs-reference floor + fp8 flip rates ------------------------------------
    def flips(tap, block, names):
        out = {}
        for n in names:
            mod = block
            for part in n.split("."):
                mod = getattr(mod, part)
            theirs_q = xq_of.get(mod)
            mine_q = tap.get(n)
            if theirs_q is None or mine_q is None:
                continue
            out[n] = (theirs_q.reshape(-1).view(torch.uint8) != mine_q.reshape(-1).view(torch.uint8)).float().mean().item()
        return out

    def floor_of(mod, kwargs, args, out_ref):
        """reference-vs-reference: the same block, same inputs, every other SDPA backend that runs here."""
        res = {}
        state["live"] = False
        try:
            for bname, backend in sdpa_backends():
                try:
                    with sdpa(backend):
                        alt = mod(*args, **kwargs)
                except RuntimeError:
                    continue
                alt = alt if isinstance(alt, tuple) else (alt,)
                ref_o = out_ref if isinstance(out_ref, tuple) else (out_ref,)
                a, b = torch.cat([x.float().flatten() for x in alt]), torch.cat([x.float().flatten() for x in ref_o])
                res[bname] = stats(a, b)[:2]
        finally:
            state["live"] = True
        return res

    def block_hook(kind, idx, mine, names):
        def hook(mod, args, kwargs, out):
            if not state["live"]:
                return
            B.TAP = tap = {}
            try:
                got = mine(*args, **kwargs)
            finally:
                B.TAP = None
            got_t = got if isinstance(got, tuple) else (got,)
            ref_t = out if isinstance(out, tuple) else (out,)
            a = torch.cat([x.float().flatten() for x in got_t])
            b = torch.cat([x.float().flatten() for x in ref_t])
            mean, mx, frac = stats(a, b)
            report["blocks"].append({"block": f"{kind}{idx}", "mean": mean, "max": mx, "frac_diff": frac,
                                     "amax": b.abs().max().item(), "rms": b.pow(2).mean().sqrt().item(),
                                     "flips": flips(tap, mod, names), "floor": floor_of(mod, kwargs, args, out)})
            xq_of.clear()
        return hook

    dnames = [f"{s}_{l}" for s in ("img", "txt") for l in ("attn.qkv", "attn.proj", "mlp.0", "mlp.2")]
    for i, blk in enumerate(theirs.double_blocks):
        hooks.append(blk.register_forward_hook(block_hook("double", i, ours.double_blocks[i], dnames), with_kwargs=True))
    for i, blk in enumerate(theirs.single_blocks):
        hooks.append(blk.register_forward_hook(block_hook("single", i, ours.single_blocks[i], ["linear1", "linear2"]),
                                               with_kwargs=True))
    try:
        with torch.inference_mode():
            y_ref = theirs(**call)
    finally:
        for h in hooks:
            h.remove()
        ref.fm.attention = ref_attention

    def dump():
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", f"parity_{name}.json"), "w") as f:
            json.dump(report, f)

    dump()
    # ---- free-running forward at full depth: ours / reference / reference on another SDPA backend ----------------
    with torch.inference_mode():
        y_ours = ours(**call)
        free = {"ours_vs_ref": stats(y_ours, y_ref)[:2], "ref_amax": y_ref.abs().max().item(),
                "ref_rms": y_ref.float().pow(2).mean().sqrt().item(), "ref_vs_ref": {}}
        for bname, backend in sdpa_backends():
            try:
                with sdpa(backend):
                    y_alt = theirs(**call)
            except RuntimeError:
                continue
            free["ref_vs_ref"][bname] = stats(y_alt, y_ref)[:2]
            free.setdefault("ours_vs_ref_alt", {})[bname] = stats(y_ours, y_alt)[:2]
    report["free_running"] = free
    assert torch.isfinite(y_ours.float()).all()

    dump()

    # ---- bars -------------------------------------------------------------------------------------------------------
    n_f8 = sum(isinstance(m, ref.f8.F8Linear) for m in theirs.modules())
    assert len(report["layers"]) >= n_f8 - 8  # every block linear ran (embedder / final-layer linears are nn.Linear)
    assert len(report["attention"]) == 57 and len(report["blocks"]) == 57
    worst_layer = max(report["layers"], key=lambda r: r["max"] / max(r["amax"], 1e-6))
    print(f"[{name}] layers: {len(report['layers'])} F8Linear calls, worst max|d|/amax = "
          f"{worst_layer['max'] / worst_layer['amax']:.3e} ({worst_layer['layer']}), "
          f"mean frac_diff = {sum(r['frac_diff'] for r in report['layers']) / len(report['layers']):.4f}")
    for r in report["layers"]:
        # identical operand bytes: only fp32 accumulation order differs -> at most 1 bf16 ulp at the output range
        assert r["max"] <= 2.0 ** -7 * max(1.0, r["amax"]), r
        assert r["frac_diff"] <= 0.10, r
    for r in report["attention"]:
        assert r["max"] <= 2 * 2.0 ** -7 * max(1.0, r["amax"]), r  # bf16 P (ours / flash) vs the backend's rounding

    flip_all = [v for r in report["blocks"] for v in r["flips"].values()]
    ratios = []
    for r in report["blocks"]:
        fused = [v for k, v in r["floor"].items()]
        assert fused, "no alternative SDPA backend ran: cannot measure the reference-vs-reference floor"
        floor_mean = max(v[0] for v in fused)
        floor_max = max(v[1] for v in fused)
        ratios.append(r["mean"] / max(floor_mean, 1e-9))
        # our error on the reference's own block input stays within the reference's own backend-to-backend spread
        assert r["mean"] <= 1.5 * floor_mean + 2.0 ** -10 * max(1.0, r["rms"]), r
        assert r["max"] <= 2.0 * floor_max + 2.0 ** -6 * max(1.0, r["amax"]), r
    print(f"[{name}] blocks: ours/floor mean-error ratio median {sorted(ratios)[len(ratios) // 2]:.2f}, "
          f"max {max(ratios):.2f}; fp8 operand flip rate mean {sum(flip_all) / max(len(flip_all), 1):.4f}, "
          f"max {max(flip_all) if flip_all else 0:.4f}")
    rr = free["ref_vs_ref"]
    floor_free = max(v[0] for v in rr.values())
    print(f"[{name}] free-running 57 blocks: ours-ref mean/max = {free['ours_vs_ref'][0]:.4f}/{free['ours_vs_ref'][1]:.4f}; "
          f"ref-vs-ref = { {k: (round(v[0], 4), round(v[1], 4)) for k, v in rr.items()} }; ref rms {free['ref_rms']:.3f}")
    assert free["ours_vs_ref"][0] <= 1.25 * floor_free + 1e-3
    del theirs, ours
    torch.cuda.empty_cache()


@pytest.mark.parametrize("name", list(CONFIGS))
def test_full_depth_output_matches_the_stored_reference_output(name, golden_dir, lib):
    """Self-contained form of the free-running check above, against what oracle/reference_golden.py stored from the
    reference on a B200: this package's quantisation of the same seeded weights, given the reference's calibrated input
    scales, reproduces the reference's state byte for byte, and our full-depth output on a fixed sample of positions
    stays within the reference's own spread between SDPA backends.  The input checksum comes first, so a change to how
    the request or the schedule is generated names itself instead of showing up as a parity failure."""
    from flux_fp8_api_b200 import f8linear, model as M, pipeline as PL

    gold = torch.load(os.path.join(golden_dir, "reference_flux_full.pt"))[name]
    _, _, _, qmod, _, in_dt = CONFIGS[name]
    params, _, call = G.flux_call(name)
    assert G.state_bytesum(call) == gold["inputs_bytesum"], f"{name}: the forward's inputs differ from the reference's"
    net = PL.build_synthetic_flux(M.FluxSpec(params=params, quantize_modulation=qmod), DEV, seed=7)
    names = G.f8_names(net, f8linear.F8Linear)
    assert len(names) == gold["n_f8"]
    sd = net.state_dict()
    for n, (s, r) in zip(names, gold["scales"].to(DEV)):
        sd[f"{n}.input_scale"], sd[f"{n}.input_scale_reciprocal"] = s.clone(), r.clone()
    del net
    with torch.device(DEV):
        ours = M.Flux(M.FluxSpec(params=params, prequantized_flow=True, quantize_modulation=qmod), dtype=BF16).to(BF16)
    missing, unexpected = ours.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    del sd
    ours.eval()
    if in_dt != torch.float8_e5m2:
        PL.set_input_float8_dtype(ours, in_dt)
    assert PL.all_frozen(ours)
    assert G.state_bytesum(ours.state_dict()) == gold["state_bytesum"]
    with torch.inference_mode():
        y = ours(**call)
    assert list(y.shape) == gold["y_shape"] and torch.isfinite(y.float()).all()
    d = (G.sample(y, gold["y_ref"].numel()).float() - gold["y_ref"].float()).abs()
    floor_free = max(v[0] for v in gold["ref_vs_ref"].values())
    print(f"[{name}] free-running 57 blocks, {d.numel()} sampled outputs: ours-ref mean/max = {d.mean().item():.4f}/"
          f"{d.max().item():.4f}; ref-vs-ref = {gold['ref_vs_ref']}")
    assert d.mean().item() <= 1.25 * floor_free + 1e-3
    del ours
    torch.cuda.empty_cache()
