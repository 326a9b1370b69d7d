"""The reference-side binding (flux_fp8_api_b200.reference_binding, quoted in INTEGRATION.md) executed against the
staged UNMODIFIED reference (oracle/_ref, see oracle/fetch_ref.py); the signature and state-layout checks run against the
reference's surface stored in tests/golden/reference_surface.json.

CPU part: the staged files are byte-identical to the reference tree they were staged from; after bind() the reference's own `Flux` container
builds over the B200 classes, has exactly the reference's state-dict keys, and loads a reference-minted prequantised
state dict.  GPU part (-m gpu): that container -- the reference's own Flux.forward driving our blocks -- gives the same
output as this package's Flux and matches the reference-minted golden; LoRA load / unload through the reference-named
entry points round-trips.
"""
import os
import types

import pytest
import torch

from oracle import ref_loader as R

BF16 = torch.bfloat16
needs_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref not staged (run python oracle/fetch_ref.py)")


@pytest.fixture()
def bound():
    from flux_fp8_api_b200 import reference_binding as RB

    ref = R.load()
    saved = RB.bind(ref.f8, ref.fm, ref.lora, replace_container=False)
    yield ref
    RB.unbind(saved)


@needs_ref
def test_staged_reference_is_the_unmodified_reference():
    m = R.verify_manifest()  # sha256 vs MANIFEST.json, and vs /root/reference where that exists
    assert set(m["files"]) == {"float8_quantize.py", "modules/flux_model.py", "lora_loading.py", "modules/autoencoder.py"}
    ref = R.load()
    assert ref.fm.__file__.startswith(R.REF_DIR) and ref.f8.__file__.startswith(R.REF_DIR)
    # nothing of it is tracked by git
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tracked = subprocess.run(["git", "ls-files", "oracle/_ref"], cwd=root, capture_output=True, text=True).stdout.strip()
    assert tracked == ""


def test_autoencoder_surface_matches_the_reference(golden_dir):
    """Constructor signatures, state-dict keys and shapes of the decode half (SURVEY.md 8f N4), against the reference's
    as stored in tests/golden/reference_surface.json (oracle/reference_golden.py)."""
    import inspect
    import json

    from flux_fp8_api_b200 import autoencoder as A

    with open(os.path.join(golden_dir, "reference_surface.json")) as f:
        gold = json.load(f)
    for name, theirs in gold["autoencoder_init"].items():
        assert [p.name for p in inspect.signature(getattr(A, name).__init__).parameters.values()] == theirs, name
    assert sorted(A.AutoEncoderParams.model_fields) == gold["autoencoder_params_fields"]
    params, theirs = gold["autoencoder_state_shapes"]["params"], gold["autoencoder_state_shapes"]["shapes"]
    ours = A.AutoEncoder(A.AutoEncoderParams(**params)).state_dict()
    assert {k: list(v.shape) for k, v in ours.items()} == theirs
    # a reference checkpoint (its keys and shapes) loads the way util.py:285 loads it
    ckpt = {k: torch.zeros(shape) for k, shape in theirs.items()}
    missing, unexpected = A.AutoEncoder(A.AutoEncoderParams(**params)).load_state_dict(ckpt, strict=False)
    assert not missing and not unexpected


@needs_ref
def test_bind_redirects_the_autoencoder_and_a_reference_checkpoint_loads():
    """bind(..., autoencoder=modules.autoencoder): the name util.load_autoencoder constructs (util.py:281) is ours, a state
    dict minted by the reference class loads with strict=False exactly as util.py:285 loads it, unbind restores."""
    from flux_fp8_api_b200 import autoencoder as A, reference_binding as RB

    ref = R.load()
    params = dict(resolution=64, in_channels=3, ch=64, out_ch=3, ch_mult=[1, 2], num_res_blocks=1, z_channels=16,
                  scale_factor=0.3611, shift_factor=0.1159)
    orig = ref.ae.AutoEncoder
    theirs = orig(ref.ae.AutoEncoderParams(**params))
    saved = RB.bind(ref.f8, ref.fm, ref.lora, replace_container=False, autoencoder=ref.ae)
    try:
        assert ref.ae.AutoEncoder is A.AutoEncoder and ref.ae.Decoder is A.Decoder
        built = ref.ae.AutoEncoder(ref.ae.AutoEncoderParams(**params))  # the reference's own params class
        missing, unexpected = built.load_state_dict(theirs.state_dict(), strict=False, assign=True)
        assert not missing and not unexpected
        assert torch.equal(built.decoder.conv_in.weight, theirs.decoder.conv_in.weight)
        assert built.scale_factor == theirs.scale_factor and built.shift_factor == theirs.shift_factor
        with pytest.raises(Exception):
            built.decode(torch.zeros(1, 16, 8, 8))  # CPU tensors: no fallback
    finally:
        RB.unbind(saved)
    assert ref.ae.AutoEncoder is orig


def test_signatures_match_the_reference(golden_dir):
    """Every replaced reference function / class / Flux method keeps the reference's signature, as stored in
    tests/golden/reference_surface.json (oracle/reference_golden.py)."""
    import inspect
    import json

    from flux_fp8_api_b200 import blocks, f8linear, model

    with open(os.path.join(golden_dir, "reference_surface.json")) as f:
        theirs = json.load(f)["signatures"]

    def params(fn):
        return [[p.name, int(p.kind), repr(p.default) if not isinstance(p.default, torch.dtype) else str(p.default)]
                for p in inspect.signature(fn).parameters.values()]

    for name in ("F8Linear", "recursive_swap_linears", "quantize_flow_transformer_and_dispatch_float8"):
        assert params(getattr(f8linear, name)) == theirs[f"float8_quantize.{name}"], name
    for name in ("attention", "rope", "apply_rope", "EmbedND", "QKNorm", "Modulation", "DoubleStreamBlock",
                 "SingleStreamBlock"):
        assert params(getattr(blocks, name)) == theirs[f"flux_model.{name}"], name
    for meth in ("get_lora", "has_lora", "load_lora", "unload_lora", "from_pretrained", "forward"):
        assert [p[0] for p in params(getattr(model.Flux, meth))] == [p[0] for p in theirs[f"flux_model.Flux.{meth}"]], meth
    # block forwards: the reference's positional / keyword names first (extras are optional keyword hand-downs)
    assert [p[0] for p in params(blocks.DoubleStreamBlock.forward)][:5] == ["self", "img", "txt", "vec", "pe"]
    assert [p[0] for p in params(blocks.SingleStreamBlock.forward)][:4] == ["self", "x", "vec", "pe"]


@needs_ref
def test_bind_redirects_and_unbind_restores():
    from flux_fp8_api_b200 import blocks, f8linear, reference_binding as RB

    ref = R.load()
    orig = (ref.f8.F8Linear, ref.fm.DoubleStreamBlock, ref.fm.Flux, ref.lora.apply_lora_to_model)
    saved = RB.bind(ref.f8, ref.fm, ref.lora, replace_container=False)
    try:
        assert ref.f8.F8Linear is f8linear.F8Linear and ref.fm.DoubleStreamBlock is blocks.DoubleStreamBlock
        assert ref.f8.Modulation is blocks.Modulation and ref.lora.F8Linear is f8linear.F8Linear
        assert ref.fm.Flux is orig[2]  # replace_container=False keeps the reference's own container
    finally:
        RB.unbind(saved)
    assert (ref.f8.F8Linear, ref.fm.DoubleStreamBlock, ref.fm.Flux, ref.lora.apply_lora_to_model) == orig


@needs_ref
def test_reference_container_over_b200_classes_loads_reference_state(bound, golden_dir):
    """util.load_flow_model's sequence (meta-device construction, load_state_dict(assign=True), util.py:245-256) with
    the reference's own Flux class, whose blocks / F8Linear are now the B200 ones."""
    from flux_fp8_api_b200 import blocks, f8linear

    ref = bound
    gold = torch.load(os.path.join(golden_dir, "flux_tiny.pt"))
    spec = R.model_spec(ref, gold["tiny"], prequantized_flow=True)
    with torch.device("meta"):
        net = ref.fm.Flux(spec, dtype=BF16)
    assert type(net).__module__ == "modules.flux_model"
    assert isinstance(net.double_blocks[0], blocks.DoubleStreamBlock)
    assert isinstance(net.single_blocks[0].linear1, f8linear.F8Linear)
    missing, unexpected = net.load_state_dict(gold["state"], strict=True, assign=True)
    assert not missing and not unexpected
    assert set(net.state_dict().keys()) == set(gold["state"].keys())
    lin = net.double_blocks[0].img_attn.qkv
    assert lin.frozen and lin.float8_data.dtype == torch.float8_e4m3fn and lin.weight.numel() == 1
    assert torch.equal(lin.input_scale, gold["state"]["double_blocks.0.img_attn.qkv.input_scale"])
    # and there is no CPU compute path behind it: a forward on CPU tensors raises loudly
    with pytest.raises(RuntimeError):
        net.double_blocks[0](img=gold["block_in"]["img"], txt=gold["block_in"]["txt"], vec=gold["block_in"]["vec"],
                             pe=gold["block_in"]["pe"])


@needs_ref
@pytest.mark.gpu
def test_reference_forward_over_b200_blocks_matches_our_flux_and_the_golden(bound, golden_dir, lib):
    import flux_fp8_api_b200.f8linear as f8
    from flux_fp8_api_b200 import model as M

    ref = bound
    gold = torch.load(os.path.join(golden_dir, "flux_tiny.pt"))
    with torch.device("cuda"):
        theirs = ref.fm.Flux(R.model_spec(ref, gold["tiny"], prequantized_flow=True), dtype=BF16)
        ours = M.Flux(M.FluxSpec(params=M.FluxParams(**gold["tiny"]), prequantized_flow=True), dtype=BF16)
    for net in (theirs, ours):
        net.load_state_dict({k: v.cuda() for k, v in gold["state"].items()}, strict=True, assign=True)
        net.eval()
    inp = {k: v.cuda() for k, v in gold["inputs"].items()}
    f8.SCALE_SEMANTICS = "cpu"  # the golden was minted on the CPU
    try:
        with torch.inference_mode():
            ours.batch_modulation = False  # the reference container runs every Modulation on its own
            y_ref_container = theirs(**inp)
            y_ours = ours(**inp)
            # same blocks, same kernels; the containers differ in the embedders / final layer (the reference's run as
            # torch library calls, ours as weight-streaming GEMV launches: fp32 summation order)
            assert (y_ref_container.float() - y_ours.float()).abs().max().item() <= 2.0 ** -4
            # the reference container recomputes pe every step: alternate two grids with the same token count
            # (the stale-cos/sin scenario of VERDICT r1 "What's weak" #2) and check against fresh evaluations
            ids2 = inp["img_ids"].clone()
            ids2[..., 1], ids2[..., 2] = inp["img_ids"][..., 2] * 2, inp["img_ids"][..., 1]
            a1 = theirs(**inp)
            b1 = theirs(**{**inp, "img_ids": ids2})
            a2 = theirs(**inp)
            b2 = theirs(**{**inp, "img_ids": ids2})
            assert torch.equal(a1, a2) and torch.equal(b1, b2) and not torch.equal(a1, b1)
        assert (y_ours.float().cpu() - gold["y_fp8"].float()).abs().max().item() <= 2.0 ** -4
        # the reference container also runs under the CUDA-graph session (it has no denoise_step / request cache)
        from flux_fp8_api_b200 import pipeline as PL

        req = {k: v for k, v in inp.items() if k != "timesteps"}
        sched = PL.get_schedule(3, req["img"].shape[1])
        g = PL.DenoiseSession(theirs, req, use_graph=True).run(sched)
        e = PL.DenoiseSession(theirs, req, use_graph=False).run(sched)
        assert torch.isfinite(g.float()).all() and torch.equal(g, e)
    finally:
        f8.SCALE_SEMANTICS = "cuda"


@needs_ref
@pytest.mark.gpu
def test_lora_through_the_reference_named_entry_points(bound, golden_dir, lib):
    """Flux.load_lora / unload_lora of the REFERENCE container (modules/flux_model.py:631-670) call
    lora_loading.apply_lora_to_model / remove_lora_from_module, which bind() pointed at the on-device fuse."""
    ref = bound
    gold = torch.load(os.path.join(golden_dir, "flux_tiny.pt"))
    with torch.device("cuda"):
        net = ref.fm.Flux(R.model_spec(ref, gold["tiny"], prequantized_flow=True), dtype=BF16)
    net.load_state_dict({k: v.cuda() for k, v in gold["state"].items()}, strict=True, assign=True)
    net.eval()
    g = torch.Generator().manual_seed(3)
    D = gold["tiny"]["hidden_size"]
    lora = {"double_blocks.0.img_attn.proj.lora_A.weight": (torch.randn(8, D, generator=g) * 0.05).to(BF16),
            "double_blocks.0.img_attn.proj.lora_B.weight": (torch.randn(D, 8, generator=g) * 0.05).to(BF16)}
    lin = net.double_blocks[0].img_attn.proj
    before = lin.float8_data.clone()
    ptr = lin.float8_data.data_ptr()
    net.load_lora(lora, scale=1.0, name="probe")
    assert net.has_lora("probe") and lin.float8_data.data_ptr() == ptr
    assert not torch.equal(lin.float8_data.view(torch.uint8), before.view(torch.uint8))
    net.unload_lora("probe")
    assert not net.loras
    changed = (lin.float8_data.view(torch.uint8) != before.view(torch.uint8)).float().mean().item()
    assert changed < 0.2  # back to the original up to the e4m3 re-quantisation of the round trip
