"""GPU (-m gpu): the VAE decode kernels (SURVEY.md 8f N4) against torch fp32 references of the same ops, the oracle's
golden vectors, and the outputs of the UNMODIFIED reference AutoEncoder run on a B200 under torch.autocast("cuda",
torch.bfloat16) exactly as flux_pipeline.py:423-438 runs it, and in fp32 (stored by oracle/reference_golden.py)."""
import json
import math
import os

import pytest
import torch
import torch.nn.functional as F

from flux_fp8_api_b200 import autoencoder as A
from flux_fp8_api_b200 import ops
from oracle import reference_golden as G
from oracle import vae_oracle as V

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16
DEV = "cuda"
ULP = 2.0 ** -7  # one bf16 ulp relative to a value's binade top


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(shape, device=DEV, generator=g) * scale).to(BF16)


def _conv_ref(x_nhwc, weight, bias, residual_nhwc, pad):
    """The arithmetic the kernel promises, from an fp32-accumulated torch convolution of the same bf16 operands."""
    acc = F.conv2d(x_nhwc.permute(0, 3, 1, 2).float(), weight.float(), None, padding=pad)
    h = acc.to(BF16)
    if bias is not None:
        h = (h.float() + bias.float().view(1, -1, 1, 1)).to(BF16)
    if residual_nhwc is not None:
        h = (h.float() + residual_nhwc.permute(0, 3, 1, 2).float()).to(BF16)
    return acc, h  # NCHW


def _close_in_ulps(out, ref, acc_scale, what, max_ulps=2.0, max_frac=0.02):
    d = (out.float() - ref.float()).abs()
    tol = max_ulps * ULP * max(acc_scale, 1e-6)
    frac = (d > 0).float().mean().item()
    assert d.max().item() <= tol, f"{what}: max|d| {d.max().item():.4g} > {tol:.4g}"
    assert frac <= max_frac, f"{what}: {frac:.4f} of the elements differ"


@pytest.mark.parametrize("B,H,W,Cin,N,k,res", [
    (1, 8, 8, 64, 64, 3, False),        # one partial tile, BN = 64
    (2, 16, 16, 128, 256, 3, True),     # two images, residual, BN = 256
    (1, 12, 96, 64, 128, 3, False),     # W = 96 (768 px images): 32-wide strips; H not a multiple of the strip height
    (3, 20, 24, 64, 192, 3, True),      # nothing divides anything: clipped tiles in x, y and N (192 of a 256 tile)
    (1, 64, 64, 256, 256, 1, True),     # 1x1 (nin_shortcut / q / k / v / proj_out)
    (1, 128, 128, 512, 512, 3, False),  # the decoder's 128 x 128 x 512 convolutions at full size
    (1, 256, 256, 128, 128, 3, True),   # 128-channel level
])
def test_conv2d_nhwc_matches_fp32_convolution_of_the_same_bf16_operands(B, H, W, Cin, N, k, res):
    x = _rand((B, H, W, Cin), 1)
    w = _rand((N, Cin, k, k), 2, 1.0 / math.sqrt(Cin * k * k))
    b = _rand((N,), 3, 0.1)
    r = _rand((B, H, W, N), 4) if res else None
    out = ops.conv2d_nhwc(x, ops.pack_conv_weight(w), b, k * k, residual=r)
    acc, ref = _conv_ref(x, w, b, r, k // 2)
    _close_in_ulps(out.permute(0, 3, 1, 2), ref, ref.float().abs().max().item(), f"conv {B}x{H}x{W} {Cin}->{N} k{k}")


def test_conv2d_padded_input_channels_and_nchw_output():
    """conv_in (16 latent channels zero-padded to 64) and conv_out (3 output channels, NCHW image)."""
    z = torch.randn(2, 16, 24, 40, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
    x = ops.vae_latent_prep(z, 0.3611, 0.1159)
    expect = (z / 0.3611 + 0.1159).to(BF16)  # eager torch on the same GPU: AutoEncoder.decode's first line
    assert torch.equal(x[..., :16].permute(0, 3, 1, 2), expect) and not x[..., 16:].any()
    w = _rand((512, 16, 3, 3), 6, 1.0 / 12.0)
    b = _rand((512,), 7, 0.1)
    out = ops.conv2d_nhwc(x, ops.pack_conv_weight(w), b, 9)
    _, ref = _conv_ref(x[..., :16], w, b, None, 1)
    _close_in_ulps(out.permute(0, 3, 1, 2), ref, ref.float().abs().max().item(), "conv_in")

    h = _rand((2, 24, 40, 128), 8)
    w3 = _rand((3, 128, 3, 3), 9, 1.0 / 34.0)
    b3 = _rand((3,), 10, 0.1)
    img = ops.conv2d_nhwc(h, ops.pack_conv_weight(w3), b3, 9, out_mode=2)
    _, ref3 = _conv_ref(h, w3, b3, None, 1)
    assert img.shape == (2, 3, 24, 40)
    _close_in_ulps(img, ref3, ref3.float().abs().max().item(), "conv_out")


def test_dense_gemm_modes_scores_fp32_and_transposed_operand():
    """The attention block's three products: q k^T scaled (fp32 out), v^T (NCHW out with padded rows), P v."""
    S, Cn = 320, 256  # 320 positions: not a multiple of 128; K of the P v product padded to 320 -> 320 (already % 64)
    q, k = _rand((S, Cn), 11), _rand((S, Cn), 12)
    sc = ops.conv2d_nhwc(q.view(1, 1, S, Cn), k, None, 1, out_mode=1, alpha=0.0625).view(S, S)
    ref = (q.float() @ k.float().t()) * 0.0625
    assert (sc - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()
    p = ops.softmax_rows(sc)
    pref = torch.softmax(ref, -1)
    assert (p.float() - pref).abs().max().item() <= ULP * pref.max().item() * 1.5
    v = _rand((S, Cn), 13)
    o = ops.conv2d_nhwc(p.view(1, 1, S, S), v.t().contiguous(), None, 1).view(S, Cn)
    oref = p.float() @ v.float()
    _close_in_ulps(o, oref.to(BF16), oref.abs().max().item(), "P v")


@pytest.mark.parametrize("C,swish", [(64, True), (128, True), (256, False), (512, True)])
def test_group_norm_swish_is_the_fp32_formula_rounded_once(C, swish):
    x = _rand((2, 24, 20, C), 20, 2.0) + 0.5
    gamma, beta = (1 + 0.1 * _rand((C,), 21).float()).to(BF16), _rand((C,), 22, 0.1)
    y = ops.group_norm_nhwc(x, gamma, beta, 1e-6, swish)
    ref = F.group_norm(x.permute(0, 3, 1, 2).float(), 32, gamma.float(), beta.float(), eps=1e-6)
    if swish:
        ref = ref * torch.sigmoid(ref)
    ref = ref.to(BF16).permute(0, 2, 3, 1)
    d = (y.float() - ref.float()).abs()
    assert d.max().item() <= 2 * ULP * ref.float().abs().max().item()
    assert (d > 0).float().mean().item() < 0.03  # a few results sit on a rounding boundary


def test_conv_epilogue_statistics_equal_the_standalone_reduction():
    """GroupNorm fed by the producing convolution's fused sums == GroupNorm reducing the stored tensor itself."""
    for (B, H, W, Cin, N) in ((2, 40, 24, 128, 256), (4, 20, 36, 64, 1024), (3, 16, 48, 256, 512), (1, 128, 128, 128, 128)):
        x = _rand((B, H, W, Cin), 50)
        w = _rand((N, Cin, 3, 3), 51, 1.0 / math.sqrt(Cin * 9))
        b, r = _rand((N,), 52, 0.3), _rand((B, H, W, N), 53)
        st = torch.empty((B, 32, 2), dtype=torch.float64, device=DEV)
        y = ops.conv2d_nhwc(x, ops.pack_conv_weight(w), b, 9, residual=r, gn_stats=st)
        yf = y.float().reshape(B, H * W, 32, N // 32)
        ref = torch.stack([yf.double().sum((1, 3)), (yf.double() ** 2).sum((1, 3))], -1)
        assert torch.allclose(st, ref, rtol=1e-6, atol=1e-3), (st - ref).abs().max()
        gamma, beta = (1 + 0.1 * _rand((N,), 54).float()).to(BF16), _rand((N,), 55, 0.1)
        fused = ops.group_norm_nhwc(y, gamma, beta, 1e-6, True, stats=st)
        alone = ops.group_norm_nhwc(y, gamma, beta, 1e-6, True)
        d = (fused.float() - alone.float()).abs()
        assert d.max().item() <= ULP * alone.float().abs().max().item() and (d > 0).float().mean().item() < 1e-3
    with pytest.raises(ValueError):
        ops.conv2d_nhwc(_rand((5, 8, 8, 64), 56), ops.pack_conv_weight(_rand((64, 64, 3, 3), 57)), None, 9,
                        gn_stats=torch.empty((5, 32, 2), dtype=torch.float64, device=DEV))  # more images than the epilogue keeps


def test_upsample2x_is_nearest():
    x = _rand((2, 6, 10, 64), 30)
    y = ops.upsample2x_nhwc(x)
    ref = F.interpolate(x.permute(0, 3, 1, 2).float(), scale_factor=2.0, mode="nearest").to(BF16).permute(0, 2, 3, 1)
    assert torch.equal(y, ref)


def _tiny(golden_dir):
    g = torch.load(os.path.join(golden_dir, "vae_tiny.pt"))
    m = A.AutoEncoder(A.AutoEncoderParams(**g["params"]))
    sd = V.synthetic_state(m, g["state_seed"])
    assert V.state_checksum(sd) == g["state_checksum"]
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith("encoder.") for k in missing)
    return g, m.to(DEV, BF16).eval(), sd


def test_tiny_decoder_against_the_golden_vectors(golden_dir):
    """ours vs (a) the oracle's CUDA-autocast restatement, (b) the reference's own fp32 output: our distance to the fp32
    reference must not exceed the autocast arithmetic's own distance to it."""
    g, m, _ = _tiny(golden_dir)
    with torch.inference_mode():
        y = m.decode(g["z"].to(DEV)).float().cpu()
    ref32, auto = g["y_ref_fp32"], g["y_oracle_autocast"].float()
    floor = (auto - ref32).abs().mean().item()
    ours = (y - ref32).abs().mean().item()
    vs_auto = (y - auto).abs()
    print(f"tiny VAE: ours-vs-fp32 {ours:.4g}, autocast-oracle-vs-fp32 {floor:.4g}, ours-vs-oracle mean {vs_auto.mean().item():.4g} "
          f"max {vs_auto.max().item():.4g}")
    assert torch.isfinite(y).all()
    assert ours <= 1.25 * floor
    assert vs_auto.mean().item() <= floor


def test_tiny_blocks_teacher_forced_on_the_reference_activations(golden_dir):
    """mid.block_1 and mid.attn_1 on the reference's own (fp32) inputs: one block deep, so the bound is bf16 arithmetic."""
    g, m, _ = _tiny(golden_dir)
    h0, h1, h2 = g["h_conv_in"].to(DEV), g["h_mid_block_1"].to(DEV), g["h_mid_attn_1"].to(DEV)
    with torch.inference_mode():
        o1 = m.decoder.mid.block_1(h0.to(BF16)).float()
        o2 = m.decoder.mid.attn_1(h1.to(BF16)).float()
    for name, o, ref in (("mid.block_1", o1, h1), ("mid.attn_1", o2, h2)):
        d = (o - ref).abs()
        print(f"{name}: mean|d| {d.mean().item():.4g} max {d.max().item():.4g} on amax {ref.abs().max().item():.4g}")
        assert d.max().item() <= 6 * ULP * ref.abs().max().item()
        assert d.mean().item() <= 0.6 * ULP * ref.abs().max().item()


def test_loud_failures():
    x = _rand((1, 8, 8, 48), 40)
    with pytest.raises(ValueError):
        ops.conv2d_nhwc(x, _rand((64, 9 * 48), 41), None, 9)  # Cin not a multiple of 64
    with pytest.raises(ValueError):
        ops.conv2d_nhwc(_rand((1, 8, 8, 64), 42), _rand((64, 9 * 64), 43).float(), None, 9)  # fp32 weights
    m = A.AutoEncoder(A.AutoEncoderParams(resolution=64, in_channels=3, ch=64, out_ch=3, ch_mult=[1, 2], num_res_blocks=1,
                                          z_channels=16, scale_factor=1.0, shift_factor=0.0))
    with pytest.raises(ValueError):
        m.to(DEV, BF16).decode(torch.zeros(1, 4, 8, 8, device=DEV))
    with pytest.raises(ValueError):
        m.encode(torch.zeros(1, 4, 64, 64, device=DEV))
    with pytest.raises(ValueError):
        ops.conv2d_nhwc(x.new_zeros((1, 8, 8, 64)), _rand((64, 64), 44), None, 1, stride=2)  # stride 2 is the 3x3 Downsample only


def _ours(state_seed, prefixes=("decoder.",)):
    """Flux's VAE (ch 128, ch_mult 1-2-4-4) with the seeded state oracle/reference_golden.py gave the reference, and the
    byte checksum of that state."""
    ours = A.AutoEncoder(A.AutoEncoderParams(**G.VAE_PARAMS))
    sd = V.synthetic_state(ours, seed=state_seed, prefixes=prefixes)
    ours.load_state_dict(sd, strict=prefixes != ("decoder.",))
    return ours.to(DEV, BF16).eval(), G.state_bytesum(sd)


def _timed(fn, n=3):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        out = fn()
    e.record()
    torch.cuda.synchronize()
    return out, s.elapsed_time(e) / n


def _against_the_stored_reference(golden_dir, case, state_sum, inputs, out, ours_key, ref_key, ref32_key):
    """|ours - reference fp32| and |ours - reference bf16 autocast| against the reference's own bf16-vs-fp32 distance,
    all on the sample of positions the reference's outputs were stored at (G.sample: spread over every row, column and
    channel).  The state and input checksums come first, so a change to how they are generated names itself."""
    gold = torch.load(os.path.join(golden_dir, "reference_vae_full.pt"))[case]
    assert state_sum == gold["state_bytesum"], f"{case}: the seeded VAE state differs from the one the reference ran"
    assert G.state_bytesum(inputs) == gold["inputs_bytesum"], f"{case}: the input differs from the one the reference ran"
    assert list(out.shape) == gold["shape"] and out.dtype == BF16
    ref, ref32 = gold[ref_key].float(), gold[ref32_key].float()
    mine = G.sample(out, ref.numel()).float()
    floor, d32, d_ref = (ref - ref32).abs(), (mine - ref32).abs(), (mine - ref).abs()
    rep = {"case": case, "reference_autocast_vs_fp32": {"mean": floor.mean().item(), "max": floor.max().item(),
                                                        "mean_whole": gold["floor_mean"], "max_whole": gold["floor_max"]},
           f"{ours_key}_vs_fp32": {"mean": d32.mean().item(), "max": d32.max().item()},
           f"{ours_key}_vs_reference_autocast": {"mean": d_ref.mean().item(), "max": d_ref.max().item()}}
    return floor, d32, d_ref, rep


@pytest.mark.parametrize("res", [1024, 768, 1536])
def test_full_size_decode_against_the_reference_on_this_gpu(res, golden_dir):
    """Flux's VAE (ch 128, ch_mult 1-2-4-4) at full resolution: ours vs the reference's decode under CUDA autocast and in
    fp32, as oracle/reference_golden.py stored them from the unmodified reference on a B200, with the reference's own
    bf16-vs-fp32 distance as the floor; ours timed with CUDA events."""
    ours, state_sum = _ours(77)
    z = G.vae_decode_latent(78, 1, res, res)
    with torch.inference_mode():
        y_ours, ms_ours = _timed(lambda: ours.decode(z))
    floor, d_32, d_ref, rep = _against_the_stored_reference(golden_dir, f"decode-{res}", state_sum, {"z": z}, y_ours, "ours",
                                                            "y_ref", "y32")
    rep["ms_ours"] = ms_ours
    print(json.dumps(rep))
    assert torch.isfinite(y_ours).all()
    # as close to the fp32 answer as the reference's own bf16 run is (25 % slack: two bf16 runs are not the same run)
    assert d_32.mean().item() <= 1.25 * floor.mean().item()
    assert d_32.max().item() <= 1.5 * floor.max().item()
    # and no further from the reference's bf16 run than that run is from fp32 (both are bf16 perturbations of the same thing)
    assert d_ref.mean().item() <= 1.5 * floor.mean().item()


@pytest.mark.parametrize("B,height,width", [(5, 128, 192), (2, 720, 1280)])
def test_decoder_shapes_outside_the_fast_paths_against_the_reference(B, height, width, golden_dir):
    """Batch 5 (more images than the convolution epilogue keeps statistics for: the GroupNorms reduce by themselves) and a
    720 x 1280 image (latent 90 x 160: strips of 32 pixels, rows clipped, 14 400 attention positions) -- same bars as the
    full-size test, against the stored reference outputs."""
    ours, state_sum = _ours(91)
    z = G.vae_decode_latent(92, B, height, width)
    with torch.inference_mode():
        y = ours.decode(z)
    assert y.shape == (B, 3, height, width)
    floor, d32, _, rep = _against_the_stored_reference(golden_dir, f"decode-{B}x{height}x{width}", state_sum, {"z": z}, y,
                                                       "ours", "y_ref", "y32")
    print(json.dumps(rep))
    assert torch.isfinite(y).all()
    assert d32.mean().item() <= 1.25 * floor.mean().item() and d32.max().item() <= 1.5 * floor.max().item()


def test_decode_is_reproducible_run_to_run(golden_dir):
    """Same weights, same latent -> the same bits, for the fused-statistics path and the stand-alone GroupNorm reduction
    (64-channel level of the tiny model): partial sums are combined in a fixed order inside a block, fp64 across blocks."""
    g, m, _ = _tiny(golden_dir)
    z = g["z"].to(DEV)
    with torch.inference_mode():
        y0 = m.decode(z).clone()
        for _ in range(4):
            assert torch.equal(m.decode(z), y0)


def test_packed_weights_follow_parameter_updates(golden_dir):
    """The kernel-layout weight cache is keyed on parameter storage / version: load_state_dict and in-place edits are seen,
    also for a model built and loaded under inference_mode (no version counters there: invalidate_packed)."""
    g, m, sd = _tiny(golden_dir)
    z = g["z"].to(DEV)
    with torch.inference_mode():
        y0 = m.decode(z).clone()
    with torch.no_grad():
        m.decoder.conv_out.weight.mul_(2.0)  # version bump
        m.decoder.conv_out.bias.zero_()
    with torch.inference_mode():
        y1 = m.decode(z).clone()
    assert not torch.equal(y0, y1)
    m.load_state_dict({k: v.to(DEV) for k, v in sd.items()}, strict=False)  # copies in place: version bump again
    with torch.inference_mode():
        assert torch.equal(m.decode(z), y0)
        m2 = A.AutoEncoder(A.AutoEncoderParams(**g["params"])).to(DEV, BF16)
        m2.load_state_dict({k: v.to(DEV) for k, v in sd.items()}, strict=False)
        assert torch.equal(m2.decode(z), y0)
        m2.decoder.conv_out.weight.mul_(2.0)  # inference tensor: no version counter
        A.invalidate_packed(m2)
        assert not torch.equal(m2.decode(z), y0)


@pytest.mark.parametrize("B,H,W,Cin,N", [(1, 16, 16, 64, 64), (2, 64, 64, 128, 128), (1, 256, 256, 128, 128), (1, 30, 44, 64, 256),
                                         (1, 17, 23, 64, 64)])
def test_downsample_convolution_stride_2(B, H, W, Cin, N):
    """Downsample.forward (autoencoder.py:106-110): F.pad(x, (0, 1, 0, 1)) then 3x3 stride 2 padding 0, through the TMA box
    with element stride 2 (odd sizes included: the pad column / row is the TMA unit's out-of-bounds zero)."""
    x = _rand((B, H, W, Cin), 60)
    w = _rand((N, Cin, 3, 3), 61, 1.0 / math.sqrt(Cin * 9))
    b = _rand((N,), 62, 0.1)
    out = ops.conv2d_nhwc(x, ops.pack_conv_weight(w), b, 9, stride=2)
    acc = F.conv2d(F.pad(x.permute(0, 3, 1, 2).float(), (0, 1, 0, 1)), w.float(), None, stride=2)
    ref = (acc.to(BF16).float() + b.float().view(1, -1, 1, 1)).to(BF16)
    assert out.shape == (B, ref.shape[2], ref.shape[3], N)
    _close_in_ulps(out.permute(0, 3, 1, 2), ref, ref.float().abs().max().item(), f"downsample {B}x{H}x{W} {Cin}->{N}")


def test_tiny_encoder_against_the_golden_moments(golden_dir):
    g = torch.load(os.path.join(golden_dir, "vae_tiny.pt"))
    m = A.AutoEncoder(A.AutoEncoderParams(**g["params"]))
    m.load_state_dict(V.synthetic_state(m, g["state_seed"], prefixes=("decoder.", "encoder.")), strict=True)
    m = m.to(DEV, BF16).eval()
    with torch.inference_mode():
        mom = m.encoder(g["img"].to(DEV)).float().cpu()
        torch.manual_seed(5)
        z = m.encode(g["img"].to(DEV))
    ref32, auto = g["moments_ref_fp32"], g["moments_oracle_autocast"].float()
    floor, mine = (auto - ref32).abs().mean().item(), (mom - ref32).abs().mean().item()
    print(f"tiny encoder moments: ours-vs-fp32 {mine:.4g}, autocast-oracle-vs-fp32 {floor:.4g}")
    assert mom.shape == ref32.shape and mine <= 1.25 * floor
    assert z.shape == (2, 16, 8, 8) and torch.isfinite(z).all()


def test_full_size_encode_against_the_reference_on_this_gpu(golden_dir):
    """Flux's VAE encoder at 1024 x 1024 (img2img, flux_pipeline.py:489-500): the Gaussian's moments against the reference's
    under CUDA autocast and in fp32 (stored by oracle/reference_golden.py), with its own bf16-vs-fp32 distance as the
    floor; the sampled latent's shape."""
    ours, state_sum = _ours(G.VAE_ENCODE_SEEDS[0], prefixes=("decoder.", "encoder."))
    img = G.vae_encode_image(G.VAE_ENCODE_SEEDS[1])
    with torch.inference_mode():
        m_ours, ms_ours = _timed(lambda: ours.encoder(img))
        torch.manual_seed(11)
        with torch.autocast(device_type="cuda", dtype=BF16, cache_enabled=False):
            z_ours = ours.encode(img)
    assert m_ours.shape == (1, 32, 128, 128) and z_ours.shape == (1, 16, 128, 128)
    floor, d32, _, rep = _against_the_stored_reference(golden_dir, "encode-1024", state_sum, {"img": img}, m_ours, "moments",
                                                       "m_ref", "m32")
    rep["ms_ours"] = ms_ours
    print(json.dumps(rep))
    assert torch.isfinite(z_ours).all()
    assert d32.mean().item() <= 1.25 * floor.mean().item() and d32.max().item() <= 1.5 * floor.max().item()
