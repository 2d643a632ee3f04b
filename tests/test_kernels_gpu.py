"""-m gpu: every CUDA kernel, called through the C ABI, against an fp32 torch restatement of the same op.

Tolerances (written per test): outputs are stored in fp16 (rel. rounding 4.9e-4) and MMA operands are fp16, so the
reference uses fp16-rounded operands with fp32 accumulation; the bound covers fp16 output rounding plus rare
1-ulp operand flips caused by the fast GELU (2.5e-5 abs error) in the prologue.
"""
import ctypes as C

import pytest
import torch

import gpu_utils as G
from wav2sleep_b200 import _lib

pytestmark = pytest.mark.gpu


def rel_err(a, b):
    return ((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-6)).item()


def test_pack_conv_weight_layout(cuda_device):
    w = torch.randn(32, 16, 3, device=cuda_device)
    p = G.pack_conv(w, split=1).view(2, 3, 2, 32, 8)  # [hi|lo][tap][cin/8][cout][8]
    torch.cuda.synchronize()
    ref = w.permute(2, 1, 0).reshape(3, 2, 8, 32).permute(0, 1, 3, 2)
    assert torch.equal(p[0], ref.half())
    assert torch.equal(p[1], (ref - ref.half().float()).half())
    assert (p[0].float() + p[1].float() - ref).abs().max().item() < 1e-6
    # Linear(4C -> F) viewed as taps=4 (input index = tap*C + c)
    wl = torch.randn(128, 4 * 64, device=cuda_device)
    pl = G.pack_conv(wl, taps_major=1, taps=4).view(4, 8, 128, 8)
    ref = wl.view(128, 4, 8, 8).permute(1, 2, 0, 3).half()
    assert torch.equal(pl, ref)


@pytest.mark.parametrize("B,T", [(2, 4096), (3, 1024 + 256), (1, 2048)])
def test_first_conv(cuda_device, B, T):
    """first_conv_kernel vs conv1d(k3,pad1) + 1x1 stride-2 branch + sums + -inf row detection."""
    from wav2sleep_b200 import build_default
    torch.manual_seed(1)
    model = build_default({"ABD": "ABD"}, 4, seed=3).to(cuda_device).eval()
    enc = model.signal_encoders.encoders["ABD"]
    x = torch.randn(B, T, device=cuda_device)
    if B > 1:
        x[1] = float("-inf")
    # run the whole encoder in keep mode and look at block 0's first tensors in the workspace
    from wav2sleep_b200.engine import PackPlan, _PackedEncoder
    lib = _lib.load()
    plan = PackPlan(lib, cuda_device)
    pe = _PackedEncoder(lib, enc, cuda_device, plan)
    plan.run()
    ws_bytes = lib.w2s_encoder_workspace_bytes(C.byref(pe.desc), B, T, 1)
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=cuda_device)
    z = torch.zeros(B, T // 256, 128, dtype=torch.float16, device=cuda_device)
    mask = torch.zeros(B, dtype=torch.uint8, device=cuda_device)
    _lib.check(lib.w2s_encoder_fwd(C.byref(pe.desc), x.data_ptr(), B, T, ws.data_ptr(), ws_bytes, 1, z.data_ptr(),
                                   mask.data_ptr(), G.stream()))
    torch.cuda.synchronize()
    assert mask.tolist() == [0] + ([1] if B > 1 else []) + [0] * max(0, B - 2)
    offs = (C.c_int64 * (7 * len(enc.channels)))()
    _lib.check(lib.w2s_encoder_layout(C.byref(pe.desc), B, T, offs))
    s1 = ws[offs[0]: offs[0] + B * 16 * 2 * 8].view(torch.float64).view(B, 16, 2).float()
    y1 = ws[offs[3]: offs[3] + B * T * 16 * 2].view(torch.float16).view(B, T, 16)
    r0 = ws[offs[4]: offs[4] + B * (T // 2) * 16 * 2].view(torch.float16).view(B, T // 2, 16)
    w1 = enc.cnn[0].conv1.conv.weight
    wd = enc.cnn[0].downsample.weight
    live = [b for b in range(B) if not (B > 1 and b == 1)]
    xr = x[live]
    ref = torch.nn.functional.conv1d(xr[:, None], w1, padding=1).transpose(1, 2)
    refr = torch.nn.functional.conv1d(xr[:, None], wd, stride=2).transpose(1, 2)
    assert (y1[live].float() - ref).abs().max().item() < 2e-3 * ref.abs().max().item()  # fp16 storage
    assert (r0[live].float() - refr).abs().max().item() < 2e-3 * refr.abs().max().item()
    assert torch.allclose(s1[live][..., 0], ref.sum(1), rtol=1e-4, atol=1e-2)
    assert torch.allclose(s1[live][..., 1], (ref * ref).sum(1), rtol=1e-4, atol=1e-2)


@pytest.mark.parametrize("cin,S", [(64, 37), (128, 130), (128, 16)])
def test_encoder_linear(cuda_device, cin, S):
    """Linear(4C -> 128) + bias + GELU as a 4-tap stride-4 conv (reference models/wav2sleep.py:261-265)."""
    torch.manual_seed(cin + S)
    dev, B, L = cuda_device, 2, 4 * S
    y = torch.randn(B, L, cin, device=dev).half()
    r = torch.randn(B, L, cin, device=dev).half()
    w = torch.randn(128, 4 * cin, device=dev) / (4 * cin) ** 0.5
    bias = torch.randn(128, device=dev)
    out = torch.full((B, S, 128), float("nan"), dtype=torch.float16, device=dev)
    G.run_conv(cin=cin, cout=128, taps=4, stride=4, dilation=1, pad=0, prologue=_lib.PRO_NORM_RES,
               epilogue=_lib.EPI_BIAS_GELU, has_ds=0, B=B, L_in=L, L_out=S, **{"in": y}, in_res=r,
               in_stats=G.sums(y), w=G.pack_conv(w, taps_major=1, taps=4), bias=bias, out=out, in_eps=1e-2)
    a = G.prologue_ref(y, r).half().float().reshape(B, S, 4 * cin)
    ref = G.gelu(a @ w.half().float().t() + bias)
    assert rel_err(out, ref) < 4e-3


@pytest.mark.parametrize("dil,S,res", [(1, 200, 0), (4, 130, 0), (32, 300, 0), (32, 1200, 1), (2, 50, 1)])
def test_seq_conv_layer(cuda_device, dil, S, res):
    """Dilated k7 conv + ConvLayerNorm + GELU (+ residual + GELU + classifier head)."""
    torch.manual_seed(dil + S)
    dev, B = cuda_device, 2
    x = torch.randn(B, S, 128, device=dev).half()
    w = torch.randn(128, 128, 7, device=dev) / (7 * 128) ** 0.5
    g, b = torch.randn(128, device=dev) * 0.2 + 1, torch.randn(128, device=dev) * 0.1
    xin = torch.randn(B, S, 128, device=dev).half() if res else None
    hw, hb = torch.randn(5, 128, device=dev) / 11, torch.randn(5, device=dev)
    out = torch.full((B, S, 128), float("nan"), dtype=torch.float16, device=dev)
    logits = torch.full((B, S, 5), float("nan"), device=dev)
    G.run_conv(cin=128, cout=128, taps=7, stride=1, dilation=dil, pad=3 * dil, prologue=_lib.PRO_NONE,
               epilogue=_lib.EPI_LN_GELU_RES if res else _lib.EPI_LN_GELU, has_ds=0, B=B, L_in=S, L_out=S,
               **{"in": x}, w=G.pack_conv(w), ln_w=g, ln_b=b, res=xin, head_w=hw if res else None,
               head_b=hb if res else None, logits=logits if res else None, n_classes=5 if res else 0, out=out,
               ln_eps=1e-5)
    c = G.conv_ref(x, w, stride=1, pad=3 * dil, dil=dil)
    mu = c.mean(-1, keepdim=True)
    var = (c - mu).pow(2).mean(-1, keepdim=True)
    ref = G.gelu((c - mu) / torch.sqrt(var + 1e-5) * g + b)
    if res:
        ref = G.gelu(ref + xin.float())
    assert (out.float() - ref).abs().max().item() < 5e-3
    if res:
        assert (logits - (ref @ hw.t() + hb)).abs().max().item() < 5e-3


def _seqmixer_fwd(lib, d, x, B, S, ncls, keep):
    """One w2s_seqmixer_head_fwd call on a workspace of NaN patterns (padding rows must be written), run twice so that
    the second call re-uses the dirty workspace.  Returns (features, logits)."""
    nbytes = lib.w2s_seqmixer_workspace_bytes(C.byref(d), B, S, keep)
    work = torch.full((nbytes,), 0x7F, dtype=torch.uint8, device=x.device)
    feat = torch.full((B, S, 128), float("nan"), dtype=torch.float16, device=x.device)
    logits = torch.full((B, S, ncls), float("nan"), device=x.device)
    for rep in range(2):
        _lib.check(lib.w2s_seqmixer_head_fwd(C.byref(d), x.data_ptr(), B, S, work.data_ptr(), nbytes, keep, feat.data_ptr(),
                                             logits.data_ptr(), G.stream()))
    torch.cuda.synchronize()
    return feat, logits


# Largest night the cluster-per-night kernel takes at 7 dilations: 2 tiles of 128 rows on each of 8 CTAs, because the
# 2 x 192 padding rows leave no room for a third tile in 232,448 B (seq_geometry_for).
SEQ_FUSED_MAX_S7 = 2048


@pytest.mark.parametrize("B,S,n_blocks,n_dil,ncls", [
    (1, 1, 2, 6, 4), (3, 40, 2, 6, 5), (2, 129, 1, 2, 4), (2, 300, 2, 6, 4), (3, 1200, 2, 6, 4), (2, 1680, 2, 6, 5),
    (1, 2048, 2, 3, 4), (1, 2100, 2, 6, 4),
    (2, 300, 3, 6, 4), (2, 260, 4, 6, 5),           # 3 and 4 blocks (24 layers in one launch)
    (2, 150, 2, 1, 4), (1, 70, 4, 1, 8),            # one dilation: never fused, layer-per-launch kernels
    (2, 500, 2, 7, 4),                              # 7 dilations fused: padding 3 * 64 = 192 rows
    (3, 40, 2, 6, 1), (2, 130, 1, 3, 8),            # 1 and 8 classes
    (2, 5, 2, 6, 4), (3, 2, 1, 7, 5),               # nights shorter than the largest dilation
    (1, 2048, 1, 6, 4), (1, 2049, 1, 6, 4),         # around 2048 epochs at 6 dilations ...
    (1, 2048, 1, 7, 4), (1, 2049, 1, 7, 4),         # ... and on both sides of the fused limit at 7 dilations
    (160, 100, 2, 6, 4),                            # more nights than clusters can be resident (148 SMs)
    (2, 64, 1, 8, 4),                               # 8 dilations: layer-per-launch only, which cannot stage dilation 128
])
def test_seqmixer_stage(cuda_device, B, S, n_blocks, n_dil, ncls):
    """w2s_seqmixer_head_fwd (SequenceCNN + classifier, models/wav2sleep.py:379-390, 66) against an fp64 torch
    restatement on the fp16-rounded operands and inter-layer activations.  keep = 0 runs the cluster-per-night kernel
    where it fits (seq_mixer.cuh: 2..7 dilations, 1 CTA for S <= 128 ... 8 CTAs x 4 tiles), the layer-per-launch kernels
    otherwise; keep = 1 (the training layout, every layer output kept) always runs the layer-per-launch kernels.  Both
    must give the same numbers.  The tile-per-CTA conv cannot stage dilation 64 or more in shared memory: those calls
    must fail with the layer's shape and byte count."""
    lib = _lib.load()
    torch.manual_seed(S + n_dil)
    dev = cuda_device
    x = torch.randn(B, S, 128, device=dev).half()
    d = _lib.SeqDesc()
    d.n_blocks, d.n_dilations, d.kernel_size, d.feature_dim, d.n_classes, d.ln_eps = n_blocks, n_dil, 7, 128, ncls, 1e-5
    keep, ws, gs, bs = [], [], [], []
    for bl in range(n_blocks):
        for k in range(n_dil):
            w = torch.randn(128, 128, 7, device=dev) / (7 * 128) ** 0.5 * 1.5
            g, b = torch.randn(128, device=dev) * 0.2 + 1, torch.randn(128, device=dev) * 0.1
            pw = G.pack_conv(w)
            keep += [pw, g, b]
            ws.append(w), gs.append(g), bs.append(b)
            d.w[bl][k], d.ln_w[bl][k], d.ln_b[bl][k] = pw.data_ptr(), g.data_ptr(), b.data_ptr()
    hw, hb = torch.randn(ncls, 128, device=dev) / 11, torch.randn(ncls, device=dev)
    d.head_w, d.head_b = hw.data_ptr(), hb.data_ptr()
    cur = x.double()
    i = 0
    for bl in range(n_blocks):
        blk_in = cur
        for k in range(n_dil):
            c = torch.nn.functional.conv1d(cur.transpose(1, 2), ws[i].half().double(), padding=3 * 2 ** k,
                                           dilation=2 ** k).transpose(1, 2)
            mu = c.mean(-1, keepdim=True)
            var = (c - mu).pow(2).mean(-1, keepdim=True)
            a = G.gelu((c - mu) / torch.sqrt(var + 1e-5) * gs[i].double() + bs[i].double())
            if k == n_dil - 1:
                a = G.gelu(a + blk_in)
            last = (bl == n_blocks - 1 and k == n_dil - 1)
            final = a
            cur = a if last else a.half().double()  # every layer but the last stores fp16
            i += 1
    ref_logits = final @ hw.double().t() + hb.double()
    # the per-layer conv stages (128 - 1) + 6 * dilation + 1 rows: dilation 64 and up exceed the shared memory of a block
    per_layer_fits = n_dil <= 6
    fused = 2 <= n_dil <= 7 and (n_dil < 7 or S <= SEQ_FUSED_MAX_S7)
    out = {}
    for kp in (0, 1):
        if not (per_layer_fits or (kp == 0 and fused)):
            with pytest.raises(RuntimeError, match=r"c128->128 k7 stride 1 dilation 64 needs 269328 B of shared memory"):
                _seqmixer_fwd(lib, d, x, B, S, ncls, kp)
            print(f"seq mixer B={B} S={S} {n_blocks}x{n_dil} keep={kp}: refused ({_lib.load().w2s_last_error().decode()})")
            continue
        feat, logits = _seqmixer_fwd(lib, d, x, B, S, ncls, kp)
        assert torch.isfinite(logits).all() and torch.isfinite(feat.float()).all()
        e_feat = (feat.double() - final).abs().max().item()
        e_log = (logits.double() - ref_logits).abs().max().item()
        print(f"seq mixer B={B} S={S} {n_blocks}x{n_dil} C={ncls} keep={kp}: feature max-abs {e_feat:.3e}, "
              f"logits max-abs {e_log:.3e}")
        # fp16 re-rounding of 1-ulp-different intermediates over n_blocks * n_dil layers
        assert e_feat < 1.5e-2 and e_log < 1.5e-2
        out[kp] = logits
    if len(out) == 2:
        e_keep = (out[1] - out[0]).abs().max().item()
        print(f"seq mixer B={B} S={S}: keep=1 vs keep=0 logits max-abs {e_keep:.3e}")
        assert e_keep < 1.5e-2


@pytest.mark.parametrize("c", [32, 64, 128])
def test_bf16_operands_on_hardware(cuda_device, c):
    """The north star names bf16; this path multiplies fp16 operands.  Hardware evidence at the kernel level: the same
    encoder conv (InstanceNorm + GELU prologue, k3, fp32 accumulate in TMEM) with the MMA operand type flipped to bf16
    (w2s_set_conv_impl(3): bf16 rounding in the prologue, bf16-packed weights, bf16 instruction descriptor), both
    against fp32 torch on UNROUNDED operands.  bf16 keeps 8 mantissa bits instead of 11: its operand error is ~8x the
    fp16 one, on top of the common fp16 output rounding (the model-level consequence - 7.6e-2 / 99.4 % against
    1.05e-2 / 100 % on two cardio nights - is tools/emulate_16bit.py, profiles/r02_emulation_16bit.txt)."""
    lib = _lib.load()
    torch.manual_seed(c)
    dev, B, L = cuda_device, 2, 4096
    y = torch.randn(B, L, c, device=dev).half()
    w = torch.randn(c, c, 3, device=dev) / (3 * c) ** 0.5
    ref = G.conv_ref(G.prologue_ref(y), w, split=1)  # fp32, operands not rounded
    err = {}
    try:
        for name, impl, split in (("fp16", 1, 0), ("bf16", 3, 2)):
            _lib.check(lib.w2s_set_conv_impl(impl))
            out = torch.full((B, L, c), float("nan"), dtype=torch.float16, device=dev)
            stats = torch.zeros(B, c, 2, dtype=torch.float64, device=dev)
            G.run_conv(cin=c, cout=c, taps=3, stride=1, dilation=1, pad=1, prologue=_lib.PRO_NORM, epilogue=_lib.EPI_STATS,
                       has_ds=0, B=B, L_in=L, L_out=L, **{"in": y}, in_stats=G.sums(y), w=G.pack_conv(w, split=split),
                       out=out, out_stats=stats, in_eps=1e-2)
            assert torch.isfinite(out.float()).all()
            err[name] = ((out.float() - ref).abs().mean() / ref.abs().mean()).item()
    finally:
        _lib.check(lib.w2s_set_conv_impl(0))
    print(f"conv {c}->{c}: mean relative error with fp16 operands {err['fp16']:.3e}, with bf16 operands {err['bf16']:.3e} "
          f"({err['bf16'] / err['fp16']:.1f}x)")
    assert err["fp16"] < 1e-3 and err["bf16"] < 1e-2   # both compute the same convolution ...
    assert err["bf16"] > 2.5 * err["fp16"]              # ... bf16 operands are markedly less accurate


def test_pack_batch_matches_single_packs(cuda_device):
    """w2s_pack_batch (strided sources, one launch) against w2s_pack_conv_weight / w2s_pack_linear_frag, incl. the
    flipped + transposed view used for data-gradient weights and the taps-major view of a Linear."""
    from wav2sleep_b200.engine import PackPlan
    lib = _lib.load()
    torch.manual_seed(3)
    w = torch.randn(32, 16, 3, device=cuda_device)
    lin = torch.randn(128, 256, device=cuda_device)  # Linear(4 * 64 -> 128)
    fr = torch.randn(384, 128, device=cuda_device)
    plan = PackPlan(lib, cuda_device)
    jobs = [(plan.conv(w, split=1), w, 0, 1), (plan.conv(w.permute(1, 0, 2), flip=True), w.flip(2).permute(1, 0, 2).contiguous(), 0, 0),
            (plan.conv(lin.view(128, 4, 64).permute(0, 2, 1)), lin, 1, 0)]
    p_frag = plan.frag(fr)
    plan.run()
    torch.cuda.synchronize()
    bufs = {t.data_ptr(): t for t in plan.keep}
    for ptr, src, taps_major, split in jobs:
        if taps_major:
            cout, cin, taps = src.shape[0], src.shape[1] // 4, 4
        else:
            cout, cin, taps = src.shape
        ref = torch.empty(cout * cin * taps * (2 if split else 1), dtype=torch.float16, device=cuda_device)
        _lib.check(lib.w2s_pack_conv_weight(src.data_ptr(), cout, cin, taps, taps_major, split, ref.data_ptr(), G.stream()))
        torch.cuda.synchronize()
        assert torch.equal(bufs[ptr], ref)
    ref = torch.empty(fr.numel(), dtype=torch.float16, device=cuda_device)
    _lib.check(lib.w2s_pack_linear_frag(fr.data_ptr(), 384, 128, ref.data_ptr(), G.stream()))
    torch.cuda.synchronize()
    assert torch.equal(bufs[p_frag], ref)
    # values change in place -> run() again picks them up without rebuilding
    w.mul_(2.0)
    plan.run()
    ref = torch.empty(32 * 16 * 3 * 2, dtype=torch.float16, device=cuda_device)
    _lib.check(lib.w2s_pack_conv_weight(w.data_ptr(), 32, 16, 3, 0, 1, ref.data_ptr(), G.stream()))
    torch.cuda.synchronize()
    assert torch.equal(bufs[jobs[0][0]], ref)
