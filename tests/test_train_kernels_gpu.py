"""-m gpu: every backward kernel of the fast training path, one C-ABI call at a time, against an fp64 torch reference of
the same operation computed from the same fp16-rounded inputs.

The whole-model gradient tests (test_training_gpu.py) bound these kernels only through relative L2 8e-2 / cosine 0.997
over sums of a million terms; a kernel wrong on a tile tail, a masked night, the zero-stuffed rows of a stride-2
gradient or past its grid cap can stay inside those bounds.  Here each kernel is held to the precision of its own
arithmetic:

* ``w2s_conv1d_fwd`` with ``W2S_EPI_ACT_BWD`` (the encoder data-gradient convs fused with the activation backward), in
  the three forms ``TrainEngine._encoder_backward`` uses, with and without ``W2S_PRO_DNORM`` (the InstanceNorm backward
  of the incoming gradient in the prologue);
* ``w2s_conv1d_fwd`` with ``W2S_EPI_PLAIN`` at every instance, in the output indexing each is used with;
* ``w2s_enc_act_fwd/bwd``, ``w2s_enc_norm_bwd``, ``w2s_first_conv_wgrad``, ``w2s_row_ln_fwd/bwd``, ``w2s_gelu_fwd/bwd``,
  ``w2s_colsum`` and ``w2s_dropout``;
* the argument checks of those entry points (calls the kernels cannot run must fail with a message).

References use the exact erf GELU (the reference model's ``nn.GELU()``) and ``torch.autograd`` of the forward formula.
Bounds:
* element-wise outputs: max-abs error over the largest |reference|;
* reductions (statistics, weight and bias gradients, column sums): every element within tol x the fp64 sum of the
  absolute values of its terms, since these sums cancel.
Each bound's source is written next to it, every test prints its measured errors, and every test asserts that a
plausible wrong reference misses by at least 10x its bound.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

import gpu_utils as G
from wav2sleep_b200 import _lib
from wav2sleep_b200._lib import EPI_ACT_BWD, EPI_PLAIN, PRO_DNORM, PRO_NONE

pytestmark = pytest.mark.gpu
F64, F16 = torch.float64, torch.float16
EPS = 1e-2                 # InstanceNorm1d eps of the encoders
SENT, SENT64 = 1000.0, 3.25  # fp16 / fp64 sentinels of rows a call must not write
ECG_NIGHT = 1200 * 1024    # block-0 length of a full ECG night


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _h(shape, g, scale=1.0, shift=0.0):
    return (torch.randn(*shape, generator=g, device="cuda") * scale + shift).half()


def _full(shape, v=SENT, dtype=F16):
    return torch.full(shape, v, dtype=dtype, device="cuda")


def _mask(B=3):
    m = torch.zeros(B, dtype=torch.uint8, device="cuda")
    m[1] = 1  # the middle night has no such signal
    return m


def _rel(out, ref):
    """max-abs error over the largest |reference| value."""
    return ((out.to(F64) - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()


def _red(out, ref, absref):
    """Worst error of a reduction, per element, over the fp64 sum of the absolute values of its terms."""
    return ((out.to(F64) - ref).abs() / absref.clamp_min(1e-300)).max().item()


def _untouched(t, v=SENT):
    return torch.equal(t, torch.full_like(t, v))


def _ulps(a, b):
    """Distance in fp16 units in the last place (0 and -0 are equal)."""
    def ordered(t):
        i = t.contiguous().view(torch.int16).to(torch.int32)
        return torch.where(i < 0, -(i & 0x7FFF), i)
    return (ordered(a) - ordered(b)).abs()


def _in_hat(y):
    """InstanceNorm1d over L (biased variance, eps 1e-2) of a [B, L, C] fp64 tensor, as the kernels' fp64 sums define it."""
    mu = y.mean(1, keepdim=True)
    var = (y * y).mean(1, keepdim=True) - mu * mu
    return (y - mu) / torch.sqrt(var.clamp_min(0) + EPS)


def _act_ref(y, r, loss_of_a):
    """Backward through a = GELU(IN(y)) [-> GELU(a + r)] by fp64 autograd: d(x_hat), a, d(r) and the two reductions
    sum d(x_hat), sum d(x_hat) x_hat over L.  Their error scale is sum |d(a)|, sum |d(a) x_hat|: the kernels' GELU'
    has an absolute error, so each term's error follows the gradient d(a) that reaches the activation, not the term
    itself, which vanishes where GELU' crosses zero (x = -0.75)."""
    xh = _in_hat(y.to(F64)).detach().requires_grad_(True)
    rr = None if r is None else r.to(F64).requires_grad_(True)
    a = F.gelu(xh)
    if rr is not None:
        a = F.gelu(a + rr)
    a.retain_grad()
    loss_of_a(a).backward()
    d, x, da = xh.grad, xh.detach(), a.grad
    return {"dxh": d, "a": a.detach(), "dr": None if rr is None else rr.grad,
            "s": torch.stack([d.sum(1), (d * x).sum(1)], -1),
            "s_abs": torch.stack([da.abs().sum(1), (da * x).abs().sum(1)], -1)}


def _in_bwd_ref(y, dxh, keep_m2=True):
    """dy of InstanceNorm1d given d(x_hat), by fp64 autograd; keep_m2=False: a wrong formula without the
    x_hat mean(d x_hat . x_hat) term."""
    if not keep_m2:
        mu = y.to(F64).mean(1, keepdim=True)
        rstd = 1.0 / torch.sqrt(((y.to(F64) - mu) ** 2).mean(1, keepdim=True) + EPS)
        d = dxh.to(F64)
        return rstd * (d - d.mean(1, keepdim=True))
    yy = y.to(F64).requires_grad_(True)
    (_in_hat(yy) * dxh.to(F64)).sum().backward()
    return yy.grad


def _dxh_like(y, g):
    """A d(x_hat) with a mean and a component along x_hat, as real gradients have: both terms of the InstanceNorm
    backward matter at every length."""
    return (torch.randn(y.shape, generator=g, device="cuda") + 0.5 * _in_hat(y.to(F64)).float() + 0.3).half()


def _in_sums(y, dxh):
    """fp64 (sum d(x_hat), sum d(x_hat) x_hat) over L: what the producing kernel accumulates for the norm backward."""
    x, d = _in_hat(y.to(F64)), dxh.to(F64)
    return torch.stack([d.sum(1), (d * x).sum(1)], -1).contiguous()


def _conv_rc(**kw):
    """w2s_conv1d_fwd with keyword fields; int values are raw device pointers.  -> (return code, last error)."""
    lib = _lib.load()
    c = _lib.ConvCall()
    for k, v in kw.items():
        if v is not None:
            setattr(c, "in_" if k == "in" else k, v.data_ptr() if isinstance(v, torch.Tensor) else v)
    rc = lib.w2s_conv1d_fwd(C.byref(c), G.stream())
    torch.cuda.synchronize()
    return rc, lib.w2s_last_error().decode()


def _dgrad_weights(cin, cout, taps, g):
    """Forward weights [cin, cout, taps] (the layer maps cout -> cin channels; fp16-rounded, fp64) and the packed
    data-gradient weights: w.permute(1, 0, 2) with the taps flipped, as TrainEngine packs them."""
    w = (torch.randn(cin, cout, taps, generator=g, device="cuda") / math.sqrt(taps * cout)).half().to(F64)
    return w, G.pack_conv(w.permute(1, 0, 2).flip(-1).float())


# ---------------------------------------------------------------------------------------------------------------------
# a. data-gradient convs fused with the activation backward (W2S_EPI_ACT_BWD)
# ---------------------------------------------------------------------------------------------------------------------
# (cin, cout) of the data-gradient conv: gradient of a layer with cin output channels back to its cout input channels
ACT_INSTANCES = [(16, 16), (32, 16), (32, 32), (64, 32), (64, 64), (128, 64), (128, 128)]
# Element-wise bound (out = d(x_hat), act_a, act_dr).  The conv itself is exact fp16 x fp16 products in fp32; the
# activation backward evaluates GELU and GELU' in the fitted tanh form with tanh.approx.f32.  Sources: fp16 output
# rounding 2^-11 = 4.9e-4 relative; the tanh fit against erf (measured in fp64 with an exact tanh) 2.5e-5 on the value and
# 1.1e-4 on the derivative; tanh.approx.f32's documented relative error 2^-11 on tanh, which enters GELU' as up to
# 0.5 |th| 2^-11 = 2.4e-4.  Set from the first B200 run (NVIDIA B200, 1000 W): worst 5.6e-4 over ACT_CASES and the
# conv of DN_CASES, so 1.5e-3 keeps a 2.7x margin.
ACT_TOL = 1.5e-3
# Reductions sum d(x_hat) and sum d(x_hat) x_hat (fp32 within a tile, fp64 atomics across tiles), per element over
# sum |d(a)| and sum |d(a) x_hat| (see _act_ref): each term carries the absolute GELU' error above times |d(a)|.
# Set from the B200 runs: worst 2.2e-4, so 6e-4 (2.7x).
ACT_RED_TOL = 6e-4
ACT_FORMS = ["conv2", "conv3", "conv1"]  # plain / after the stride-2 upsampled gradient / with res + act_r, act_dr
ACT_CASES = [(ci, co, form, L) for ci, co in ACT_INSTANCES for form in ACT_FORMS for L in (1, 2, 127, 128, 129, 383)]
ACT_CASES += [(16, 16, form, ECG_NIGHT) for form in ACT_FORMS]


def _act_inputs(cin, cout, form, L, seed):
    g = _gen(seed)
    B = 3
    w, wpk = _dgrad_weights(cin, cout, 3, g)
    y = _h((B, L, cout), g, 2.0, 0.5)
    Lo = (L + 1) // 2 if form == "conv3" else L
    dY = _h((B, Lo, cin), g)
    r = _h((B, L, cout), g) if form == "conv1" else None
    res = None
    if form == "conv1":  # gradient of the 1x1 stride-2 residual branch, scattered to the even rows
        res = _h((B, L, cout), g, 0.5)
        res[:, 1::2] = 0
    return B, w, wpk, y, dY, r, res


def _conv_loss(w, dY, stride, res, odd_rows=False):
    """Scalar whose gradient with respect to the activated conv input a is the conv's data gradient (+ res)."""
    def loss(a):
        at = a.transpose(1, 2)
        if odd_rows:  # wrong: the stride-2 gradient placed on the odd rows of the zero-stuffed tensor
            at = F.pad(at, (0, 1))[:, :, 1:]
        Y = F.conv1d(at, w, stride=stride, padding=1).transpose(1, 2)
        out = (Y * dY.to(F64)).sum()
        return out + (a * res.to(F64)).sum() if res is not None else out
    return loss


def _act_bwd_call(cin, cout, B, L, dy, wpk, y, stats, r, res, mask, with_a, dnorm=None):
    out, sums = _full((B, L, cout)), torch.zeros(B, cout, 2, dtype=F64, device="cuda")
    sums[1] = SENT64
    a = _full((B, L, cout)) if with_a else None
    dr = _full((B, L, cout)) if r is not None else None
    kw = dict(cin=cin, cout=cout, taps=3, stride=1, dilation=1, pad=1, prologue=PRO_NONE, epilogue=EPI_ACT_BWD, has_ds=0,
              B=B, L_in=L, L_out=L, w=wpk, out=out, out_stats=sums, row_mask=mask, act_y=y, act_stats=stats,
              act_eps=EPS, act_a=a, act_r=r, act_dr=dr, res=res)
    kw["in"] = dy
    if dnorm is not None:
        kw.update(dnorm)
        kw["prologue"] = PRO_DNORM
    G.run_conv(**kw)
    return out, a, dr, sums


def _check_act(tag, ref, out, a, dr, sums, live):
    errs = {"out": _rel(out[live], ref["dxh"][live]), "sums": _red(sums[live], ref["s"][live], ref["s_abs"][live])}
    if a is not None:
        errs["act_a"] = _rel(a[live], ref["a"][live])
    if dr is not None:
        errs["act_dr"] = _rel(dr[live], ref["dr"][live])
    print(f"{tag}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()) + f" (bounds {ACT_TOL:.0e} / red {ACT_RED_TOL:.0e})")
    for k, v in errs.items():
        assert v < (ACT_RED_TOL if k == "sums" else ACT_TOL), (tag, k, v)
    for t in (out, a, dr):  # the masked night is skipped
        assert t is None or _untouched(t[1]), tag
    assert _untouched(sums[1], SENT64), tag


@pytest.mark.parametrize("cin,cout,form,L", ACT_CASES)
def test_conv_act_bwd(cuda_device, cin, cout, form, L):
    B, w, wpk, y, dY, r, res = _act_inputs(cin, cout, form, L, seed=cin * 7 + cout + L + ACT_FORMS.index(form))
    mask, live = _mask(B), [0, 2]
    stats = G.sums(y)
    dy = dY
    if form == "conv3":  # the stride-2 layer's gradient enters zero-stuffed: row 2j = dY[j], odd rows 0
        dy = torch.zeros(B, L, cin, dtype=F16, device="cuda")
        dy[:, 0::2] = dY
    stride = 2 if form == "conv3" else 1
    ref = _act_ref(y, r, _conv_loss(w, dY, stride, res))
    tag = f"act_bwd {cin}->{cout} {form} L={L}"
    outs = {}
    for with_a in (False, True):
        out, a, dr, sums = _act_bwd_call(cin, cout, B, L, dy.contiguous(), wpk, y, stats, r, res, mask, with_a)
        _check_act(f"{tag} act_a={'set' if with_a else 'NULL'}", ref, out, a, dr, sums, live)
        outs[with_a] = out
    assert torch.equal(outs[False], outs[True]), "act_a changes d(x_hat)"
    # plausible wrong references
    if form == "conv2":  # a backward that treats GELU as the identity: d(x_hat) = d(a)
        xh = _in_hat(y.to(F64)).requires_grad_(True)
        _conv_loss(w, dY, 1, None)(xh).backward()
        wrong, what = xh.grad, "GELU' dropped"
    elif form == "conv3":
        wrong, what = _act_ref(y, r, _conv_loss(w, dY, 2, res, odd_rows=True))["dxh"], "upsampled gradient on odd rows"
    else:
        wrong, what = _act_ref(y, r, _conv_loss(w, dY, stride, None))["dxh"], "res contribution dropped"
    werr = _rel(outs[True][live], wrong[live])
    print(f"  wrong reference ({what}): {werr:.2e} ({werr / ACT_TOL:.0f}x the bound)")
    assert werr >= 10 * ACT_TOL


# ---------------------------------------------------------------------------------------------------------------------
# b. the same instances with the InstanceNorm backward in the prologue (W2S_PRO_DNORM)
# ---------------------------------------------------------------------------------------------------------------------
# dn_out = rstd (d - mean d - x_hat mean(d x_hat)) from fp32 constants of fp64 sums, stored fp16: the fp16 rounding
# (4.9e-4 relative) plus the fp32 cancellation of the three terms.  Set from the first B200 run: worst 4.3e-4 over
# DN_CASES and test_enc_norm_bwd, so 1.2e-3 (2.8x).  The fused prologue and enc_norm_bwd were bitwise equal there.
DN_TOL = 1.2e-3


def _dn_lengths(cout, up):
    pos = 128 * (128 // cout)  # output positions of one tile: halo rows sit at multiples of it
    base = [10, 130, 258, pos + 2] if up else [5, 129, 257, pos + 1]
    return sorted(set(base))


DN_CASES = [(ci, co, up, L) for ci, co in ACT_INSTANCES for up in (0, 1) for L in _dn_lengths(co, up)]


@pytest.mark.parametrize("cin,cout,up,L", DN_CASES)
def test_conv_act_bwd_dnorm(cuda_device, cin, cout, up, L):
    lib = _lib.load()
    g = _gen(cin * 3 + cout + L + up)
    B, mask, live = 3, _mask(), [0, 2]
    Ls = L // 2 if up else L
    w, wpk = _dgrad_weights(cin, cout, 3, g)
    y = _h((B, L, cout), g, 2.0, 0.5)  # the producing layer (EPI_ACT_BWD side)
    stats = G.sums(y)
    y_in = _h((B, Ls, cin), g, 1.5, -0.3)  # the consuming layer (PRO_DNORM side)
    dxh_in = _dxh_like(y_in, g)
    stats_in, dn_sums = G.sums(y_in), _in_sums(y_in, dxh_in)
    dn_out = _full((B, L, cin))
    dnorm = {"in": dxh_in, "in_res": y_in, "in_stats": stats_in, "dn_sums": dn_sums, "dn_out": dn_out,
             "dn_upsample": up, "in_eps": EPS}
    out, a, _, sums = _act_bwd_call(cin, cout, B, L, None, wpk, y, stats, None, None, mask, True, dnorm=dnorm)
    dy_ref = torch.zeros(B, L, cin, dtype=F64, device="cuda")
    dy_core = _in_bwd_ref(y_in, dxh_in)
    dy_ref[:, ::2 if up else 1] = dy_core
    tag = f"dnorm {cin}->{cout} up={up} L={L}"
    e_dn = _rel(dn_out[live], dy_ref[live])
    print(f"{tag}: dn_out {e_dn:.2e} (bound {DN_TOL:.0e})")
    assert e_dn < DN_TOL
    if up:
        assert (dn_out[live][:, 1::2].view(torch.int16) == 0).all(), "odd rows of the zero-stuffed gradient must be +0"
    assert _untouched(dn_out[1])
    # the conv + activation backward fed with the dy the prologue computed
    ref = _act_ref(y, None, _conv_loss(w, dn_out.to(F64), 1, None))
    _check_act(f"{tag} conv", ref, out, a, None, sums, live)
    # the separate kernel: the same formula, so at most one fp16 ulp apart
    dy_sep = _full((B, L, cin))
    _lib.check(lib.w2s_enc_norm_bwd(dxh_in.data_ptr(), y_in.data_ptr(), stats_in.data_ptr(), dn_sums.data_ptr(),
                                    dy_sep.data_ptr(), mask.data_ptr(), B, Ls, cin, up, EPS, G.stream()))
    torch.cuda.synchronize()
    u = _ulps(dn_out[live], dy_sep[live])
    print(f"  vs w2s_enc_norm_bwd: {(u != 0).sum().item()} of {u.numel()} elements not bitwise equal, max {u.max().item()} ulp")
    assert u.max().item() <= 1
    wrong = torch.zeros_like(dy_ref)
    wrong[:, ::2 if up else 1] = _in_bwd_ref(y_in, dxh_in, keep_m2=False)
    werr = _rel(dn_out[live], wrong[live])
    print(f"  wrong reference (no x_hat mean(d x_hat) term): {werr:.2e} ({werr / DN_TOL:.0f}x the bound)")
    assert werr >= 10 * DN_TOL


# ---------------------------------------------------------------------------------------------------------------------
# c. plain GEMMs and data-gradient convs (W2S_EPI_PLAIN), each instance in the output indexing training uses it with
# ---------------------------------------------------------------------------------------------------------------------
# fp16 x fp16 products accumulated in fp32 over <= 7 * 128 terms, (+ bias, + residual) and one fp16 rounding of the
# result (4.9e-4 relative).  Set from the first B200 run: worst 4.5e-4 over PLAIN_CASES, so 1.2e-3 (2.7x).
PLAIN_TOL = 1.2e-3
PLAIN_CASES = (
    # mode, cin, cout, taps, L_out, dilation
    [("lin_dgrad", 128, co, 1, S, 1) for co in (64, 128) for S in (1, 37)]       # encoder Linear dgrad: rows 4s + t
    + [("ds_dgrad", ci, co, 1, L, 1) for ci, co in ACT_INSTANCES for L in (1, 300)]  # 1x1 stride-2 branch: even rows
    + [("mix", 128, 128, 1, L, 1) for L in (5, 1000)]                             # mixer GEMM + bias + residual
    + [("k4", ci, 128, 4, S, 1) for ci in (64, 128) for S in (1, 37, 300)]        # Linear fwd / FFN as 4-tap stride-4
    + [("k7", 128, 128, 7, S, d) for d in (1, 2, 4, 8, 16, 32) for S in (1, 5, 129)]  # sequence-mixer dgrad
    + [("k3", ci, co, 3, L, 1) for ci, co in ACT_INSTANCES for L in (129, 1000)]  # dense k3 data-gradient conv
)


@pytest.mark.parametrize("mode,cin,cout,taps,L,d", PLAIN_CASES)
def test_conv_plain(cuda_device, mode, cin, cout, taps, L, d):
    g = _gen(cin + cout * 3 + taps + L * 5 + d)
    B = 2 if mode in ("mix", "k7") else 3
    mask = _mask(B) if B == 3 else None
    live = [0, 2] if B == 3 else [0, 1]
    w = (torch.randn(cout, cin, taps, generator=g, device="cuda") / math.sqrt(taps * cin)).half()
    stride, pad = (4, 0) if mode == "k4" else (1, (taps // 2) * d)
    L_in = L * stride
    x = _h((B, L_in, cin), g)
    # bias: the mixer GEMMs, the encoder Linear (64 -> 128) and linear2 of the FFN; linear1's data gradient (128 -> 128
    # k4, here at L = 37) has none
    bias = (torch.randn(cout, generator=g, device="cuda") * 0.5) if mode in ("mix", "k4") and (cin == 64 or L != 37) else None
    use_res = mode == "mix" or (mode == "k7" and (d % 2 == 0 or L == 1))
    offsets, o_stride = ([0, 1, 2, 3], 4) if mode == "lin_dgrad" else ([0], 2 if mode == "ds_dgrad" else 1)
    rows = L * o_stride
    ref_dense = F.conv1d(x.to(F64).transpose(1, 2), w.to(F64), stride=stride, padding=pad, dilation=d).transpose(1, 2)
    if bias is not None:
        ref_dense = ref_dense + bias.to(F64)
    pk = G.pack_conv(w.float())
    for off in offsets:
        out = _full((B, rows, cout))
        res = None
        if use_res:
            res = _h((B, rows, cout), g)
        kw = dict(cin=cin, cout=cout, taps=taps, stride=stride, dilation=d, pad=pad, prologue=PRO_NONE,
                  epilogue=EPI_PLAIN, has_ds=0, B=B, L_in=L_in, L_out=L, w=pk, out=out, bias=bias, res=res,
                  row_mask=mask, out_stride=o_stride if o_stride > 1 else 0, out_offset=off,
                  out_rows=rows if o_stride > 1 else 0)
        kw["in"] = x
        G.run_conv(**kw)
        ref = ref_dense + (res[:, off::o_stride].to(F64) if res is not None else 0)
        got = out[:, off::o_stride]
        err = _rel(got[live], ref[live])
        tag = f"plain {mode} {cin}->{cout} k{taps} d{d} L={L} offset {off}/{o_stride}"
        print(f"{tag}: {err:.2e} (bound {PLAIN_TOL:.0e})")
        assert err < PLAIN_TOL
        others = torch.ones(rows, dtype=torch.bool, device="cuda")
        others[off::o_stride] = False  # rows this call does not own keep their contents bit for bit
        assert _untouched(out[:, others]), tag
        if mask is not None:
            assert _untouched(out[1]), tag
        if res is not None:
            wrong, what = ref - res[:, off::o_stride].to(F64), "residual dropped"
        elif bias is not None:
            wrong, what = ref - bias.to(F64), "bias dropped"
        else:
            wrong, what = torch.roll(ref, 1, dims=1), "rows one position off"
            if L == 1:  # one row: the scatter lands one sample off instead
                wrong = torch.roll(ref, 1, dims=0)
        werr = _rel(got[live], wrong[live])
        print(f"  wrong reference ({what}): {werr:.2e} ({werr / PLAIN_TOL:.0f}x the bound)")
        assert werr >= 10 * PLAIN_TOL


# ---------------------------------------------------------------------------------------------------------------------
# d. element-wise and row kernels
# ---------------------------------------------------------------------------------------------------------------------
# enc_act_fwd / enc_act_bwd evaluate GELU and GELU' in the fitted tanh form (sources as ACT_TOL, without a conv);
# enc_norm_bwd is the formula of DN_TOL.  Set from the first B200 run: worst 5.5e-4 element-wise, so 1.5e-3 (2.7x);
# the sums as ACT_RED_TOL, worst 3.6e-5, so 1e-4 (2.8x).
ENC_TOL = 1.5e-3
ENC_RED_TOL = 1e-4
ENC_CHANNELS = [8, 16, 32, 64, 128]


def _enc_big_L(C):
    """A length past the grid caps, so that every grid-stride loop runs more than once: enc_act_bwd caps at 4 x SMs
    blocks of 256 / (C / 8) x 8 rows, the ew_grid launches (enc_act_fwd, enc_norm_bwd) at 8 x SMs x 256 chunks of 8."""
    return max(4 * _sms() * (256 // (C // 8)) * 8, 8 * _sms() * 256 // (C // 8)) + 37


@pytest.mark.parametrize("C", ENC_CHANNELS)
@pytest.mark.parametrize("big", [False, True])
def test_enc_act_fwd_bwd(cuda_device, C, big):
    lib = _lib.load()
    L = _enc_big_L(C) if big else 129
    g = _gen(C * 11 + L)
    B, mask, live = 3, _mask(), [0, 2]
    y, r, dout = _h((B, L, C), g, 2.0, 0.5), _h((B, L, C), g), _h((B, L, C), g)
    stats = G.sums(y)
    for rr in (None, r):
        tag = f"enc_act C={C} L={L} r={'set' if rr is not None else 'NULL'}"
        a = _full((B, L, C))
        _lib.check(lib.w2s_enc_act_fwd(y.data_ptr(), None if rr is None else rr.data_ptr(), stats.data_ptr(), a.data_ptr(),
                                       mask.data_ptr(), B, L, C, EPS, G.stream()))
        for with_a in (False, True):
            dxh, sums = _full((B, L, C)), torch.zeros(B, C, 2, dtype=F64, device="cuda")
            sums[1] = SENT64
            dr = _full((B, L, C)) if rr is not None else None
            a_out = _full((B, L, C)) if with_a else None
            p = lambda t: None if t is None else t.data_ptr()
            _lib.check(lib.w2s_enc_act_bwd(dout.data_ptr(), y.data_ptr(), p(rr), stats.data_ptr(), dxh.data_ptr(), p(dr),
                                           sums.data_ptr(), p(a_out), mask.data_ptr(), B, L, C, EPS, G.stream()))
            torch.cuda.synchronize()
            ref = _act_ref(y, rr, lambda t: (t * dout.to(F64)).sum())
            errs = {"fwd a": _rel(a[live], ref["a"][live]), "dxh": _rel(dxh[live], ref["dxh"][live]),
                    "sums": _red(sums[live], ref["s"][live], ref["s_abs"][live])}
            if dr is not None:
                errs["dr"] = _rel(dr[live], ref["dr"][live])
            if a_out is not None:
                errs["a_out"] = _rel(a_out[live], ref["a"][live])
                assert torch.equal(a_out, a), "enc_act_bwd's a_out differs from enc_act_fwd"
            print(f"{tag} a_out={'set' if with_a else 'NULL'}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items())
                  + f" (bounds {ENC_TOL:.0e} / red {ENC_RED_TOL:.0e})")
            for k, v in errs.items():
                assert v < (ENC_RED_TOL if k == "sums" else ENC_TOL), (tag, k, v)
            for t in (a, dxh, dr, a_out):
                assert t is None or _untouched(t[1]), tag
            assert _untouched(sums[1], SENT64)
        if rr is not None:  # wrong: the block output's outer GELU' dropped (dr = dout)
            werr, what = _rel(dr[live], dout[live].to(F64)), "outer GELU' dropped"
        else:  # wrong: the backward through GELU as the identity
            werr, what = _rel(dxh[live], dout[live].to(F64)), "GELU' dropped"
        print(f"  wrong reference ({what}): {werr:.2e} ({werr / ENC_TOL:.0f}x the bound)")
        assert werr >= 10 * ENC_TOL


@pytest.mark.parametrize("C", ENC_CHANNELS)
@pytest.mark.parametrize("up", [0, 1])
@pytest.mark.parametrize("big", [False, True])
def test_enc_norm_bwd(cuda_device, C, up, big):
    lib = _lib.load()
    L = _enc_big_L(C) if big else 129
    g = _gen(C * 13 + L + up)
    B, mask, live = 3, _mask(), [0, 2]
    y = _h((B, L, C), g, 1.5, -0.3)
    dxh = _dxh_like(y, g)
    stats, sums = G.sums(y), _in_sums(y, dxh)
    dy = _full((B, 2 * L if up else L, C))
    _lib.check(lib.w2s_enc_norm_bwd(dxh.data_ptr(), y.data_ptr(), stats.data_ptr(), sums.data_ptr(), dy.data_ptr(),
                                    mask.data_ptr(), B, L, C, up, EPS, G.stream()))
    torch.cuda.synchronize()
    ref = _in_bwd_ref(y, dxh)
    got = dy[:, ::2] if up else dy
    err = _rel(got[live], ref[live])
    print(f"enc_norm_bwd C={C} L={L} up={up}: {err:.2e} (bound {DN_TOL:.0e})")
    assert err < DN_TOL
    if up:
        assert (dy[live][:, 1::2].view(torch.int16) == 0).all(), "odd rows of the zero-stuffed gradient must be +0"
        werr, what = _rel(dy[live][:, 1::2], ref[live]), "gradient on the odd rows"
    else:
        werr, what = _rel(got[live], _in_bwd_ref(y, dxh, keep_m2=False)[live]), "no x_hat mean(d x_hat) term"
    assert _untouched(dy[1])
    print(f"  wrong reference ({what}): {werr:.2e} ({werr / DN_TOL:.0f}x the bound)")
    assert werr >= 10 * DN_TOL


# first_conv_wgrad accumulates fp16 x fp32 products in fp32: per thread over ~16 rows, then warp shuffles, a shared and
# a global fp32 atomic per block.  Each of the ~log2(T) + 16 additions rounds to 2^-24 of a partial sum bounded by the
# sum of |terms|.  Set from the first B200 run: worst 2.2e-8 (T = 256), so 6e-8 (2.7x).
WG_TOL = 6e-8


@pytest.mark.parametrize("T", [256, 4096 + 256, ECG_NIGHT])
def test_first_conv_wgrad(cuda_device, T):
    lib = _lib.load()
    g = _gen(T)
    B, mask, live = 3, _mask(), [0, 2]
    x = torch.randn(B, T, generator=g, device="cuda")
    x[0, 5:9] = float("-inf")  # missing samples inside a live night count as 0
    x[2, T - 3:] = float("-inf")
    x[1] = float("-inf")       # the masked night
    dy1, dr = _h((B, T, 16), g), _h((B, T // 2, 16), g)
    scale = 0.375
    dw1 = torch.zeros(48, device="cuda")
    dwds = torch.zeros(16, device="cuda")
    _lib.check(lib.w2s_first_conv_wgrad(x.data_ptr(), dy1.data_ptr(), dr.data_ptr(), dw1.data_ptr(), dwds.data_ptr(),
                                        mask.data_ptr(), B, T, scale, G.stream()))
    torch.cuda.synchronize()
    xc = torch.where(torch.isinf(x), torch.zeros_like(x), x).to(F64)[live]

    def grads(xs, d1, d2):
        W1 = torch.zeros(16, 1, 3, dtype=F64, device="cuda", requires_grad=True)
        Wd = torch.zeros(16, 1, 1, dtype=F64, device="cuda", requires_grad=True)
        y1 = F.conv1d(xs[:, None], W1, padding=1)
        yd = F.conv1d(xs[:, None], Wd, stride=2)
        ((y1 * d1.to(F64)[live].transpose(1, 2)).sum() + (yd * d2.to(F64)[live].transpose(1, 2)).sum()).backward()
        return W1.grad.reshape(48) * scale, Wd.grad.reshape(16) * scale

    r1, rd = grads(xc, dy1, dr)
    a1, ad = grads(xc.abs(), dy1.abs(), dr.abs())
    e1, ed = _red(dw1, r1, a1), _red(dwds, rd, ad)
    print(f"first_conv_wgrad T={T}: dw1 {e1:.2e}, dwds {ed:.2e} (bound {WG_TOL:.0e})")
    assert e1 < WG_TOL and ed < WG_TOL
    w1, _ = grads(F.pad(xc, (1, 0))[:, :-1], dy1, dr)  # wrong: taps shifted by one sample
    werr = _red(dw1, w1, a1)
    print(f"  wrong reference (taps shifted by one): {werr:.2e} ({werr / WG_TOL:.0f}x the bound)")
    assert werr >= 10 * WG_TOL


# row_ln_fwd / row_ln_bwd: fp32 LayerNorm over 128 features with the exact erf GELU (erff, __expf in GELU'): the fp16
# rounding of the outputs (4.9e-4 relative) and fp32 sums over 128 features.  dg / db are fp32 sums over the rows of a
# warp, the 8 warps of a block and one fp32 atomic per block, bounded over sum |dout x_hat| and sum |dout| (GELU' has an
# absolute error, see _act_ref).  Set from the first B200 run: worst 4.1e-4 element-wise, so 1.2e-3 (2.9x); dg / db
# worst 5.4e-7, so 1.5e-6 (2.8x).
LN_TOL = 1.2e-3
LN_RED_TOL = 1.5e-6


def _ln_big_rows():
    """Past both grid caps: row_ln_bwd runs 2 x SMs blocks of 8 rows, row_ln_fwd 8 x SMs blocks of 8 rows."""
    return 64 * _sms() + 5


@pytest.mark.parametrize("gelu,res", [(0, False), (1, False), (0, True), (1, True)])
@pytest.mark.parametrize("rows", [1, 7, "big"])
@pytest.mark.parametrize("extras", [False, True])
def test_row_ln_fwd_bwd(cuda_device, gelu, res, rows, extras):
    lib = _lib.load()
    rows = _ln_big_rows() if rows == "big" else rows
    g = _gen(rows * 4 + gelu * 2 + res + extras * 8)
    x = _h((rows, 128), g, 2.0, 0.5)
    gw = 1.0 + 0.2 * torch.randn(128, generator=g, device="cuda")
    gb = 0.1 * torch.randn(128, generator=g, device="cuda")
    r = _h((rows, 128), g) if res else None
    dout = (torch.randn(rows, 128, generator=g, device="cuda") + 0.3 * x.float()).half()  # correlated with x_hat
    dadd = _h((rows, 128), g) if extras else None
    eps, gscale = 1e-5, 0.375
    p = lambda t: None if t is None else t.data_ptr()
    out = _full((rows, 128))
    _lib.check(lib.w2s_row_ln_fwd(x.data_ptr(), p(r), gw.data_ptr(), gb.data_ptr(), out.data_ptr(), rows, gelu, eps,
                                  G.stream()))
    dx = _full((rows, 128))
    ds = _full((rows, 128)) if (res and extras) else None
    dg, db = torch.zeros(128, device="cuda"), torch.zeros(128, device="cuda")
    _lib.check(lib.w2s_row_ln_bwd(x.data_ptr(), p(r), gw.data_ptr(), gb.data_ptr(), dout.data_ptr(), p(dadd), dx.data_ptr(),
                                  p(ds), dg.data_ptr(), db.data_ptr(), rows, gelu, eps, gscale, G.stream()))
    torch.cuda.synchronize()
    # fp64 autograd of o = LN(x) g + b ; [GELU] ; [GELU(. + r)]
    xx = x.to(F64).requires_grad_(True)
    rr = None if r is None else r.to(F64).requires_grad_(True)
    mu = xx.mean(1, keepdim=True)
    xh = (xx - mu) / torch.sqrt(((xx - mu) ** 2).mean(1, keepdim=True) + eps)
    u = xh * gw.to(F64) + gb.to(F64)
    u.retain_grad()
    o = F.gelu(u) if gelu else u
    if rr is not None:
        o = F.gelu(o + rr)
    (o * dout.to(F64)).sum().backward()
    ref_dx = xx.grad + (dadd.to(F64) if dadd is not None else 0)
    du, xh = u.grad, xh.detach()
    ref_dg, ref_db = (du * xh).sum(0) * gscale, du.sum(0) * gscale
    # error scale of dg / db: sum |dout x_hat|, sum |dout| (GELU' has an absolute error, as in _act_ref)
    abs_dg, abs_db = (dout.to(F64) * xh).abs().sum(0) * gscale, dout.to(F64).abs().sum(0) * gscale
    errs = {"fwd": _rel(out, o.detach()), "dx": _rel(dx, ref_dx), "dg": _red(dg, ref_dg, abs_dg),
            "db": _red(db, ref_db, abs_db)}
    if ds is not None:
        errs["ds"] = _rel(ds, rr.grad)
    tag = f"row_ln gelu={gelu} res={int(res)} rows={rows} dadd/ds={'set' if extras else 'NULL'}"
    print(f"{tag}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()) + f" (bounds {LN_TOL:.1e} / red {LN_RED_TOL:.0e})")
    for k, v in errs.items():
        assert v < (LN_RED_TOL if k in ("dg", "db") else LN_TOL), (tag, k, v)
    if dadd is not None:
        wrong, what = ref_dx - dadd.to(F64), "dadd dropped"
    else:  # the LayerNorm backward without its x_hat mean(d x_hat . x_hat) term
        dxh = du * gw.to(F64)
        rstd = 1.0 / torch.sqrt(((x.to(F64) - x.to(F64).mean(1, keepdim=True)) ** 2).mean(1, keepdim=True) + eps)
        wrong, what = rstd * (dxh - dxh.mean(1, keepdim=True)), "no x_hat mean(d x_hat . x_hat) term"
    werr = _rel(dx, wrong)
    print(f"  wrong reference ({what}): {werr:.2e} ({werr / LN_TOL:.0f}x the bound)")
    assert werr >= 10 * LN_TOL


# gelu_fwd / gelu_bwd: exact-erf GELU in fp32 (erff, __expf), one fp16 rounding of the result.  Set from the first B200
# run: worst 9.8e-5 (forward) and 3.5e-4 (backward), so 1e-3 (2.9x).
GELU_TOL = 1e-3


@pytest.mark.parametrize("n8", [1, "big"])
def test_gelu_fwd_bwd(cuda_device, n8):
    lib = _lib.load()
    n = 8 * ((8 * _sms() * 256 + 77) if n8 == "big" else n8)  # past the 8 x SMs x 256 grid cap, not a multiple of 256
    g = _gen(n)
    x = ((torch.rand(n, generator=g, device="cuda") * 2 - 1) * 10).half()
    x[:2] = torch.tensor([10.0, -10.0], dtype=F16)
    dout = _h((n,), g, 2.0)
    out, din = _full((n,)), _full((n,))
    _lib.check(lib.w2s_gelu_fwd(x.data_ptr(), out.data_ptr(), n, G.stream()))
    _lib.check(lib.w2s_gelu_bwd(x.data_ptr(), dout.data_ptr(), din.data_ptr(), n, G.stream()))
    torch.cuda.synchronize()
    xx = x.to(F64).requires_grad_(True)
    ref = F.gelu(xx)
    (ref * dout.to(F64)).sum().backward()
    ef, eb = _rel(out, ref.detach()), _rel(din, xx.grad)
    print(f"gelu n={n}: fwd {ef:.2e}, bwd {eb:.2e} (bound {GELU_TOL:.0e})")
    assert ef < GELU_TOL and eb < GELU_TOL
    x64 = x.to(F64)
    wf = _rel(out, torch.relu(x64))
    wb = _rel(din, dout.to(F64) * 0.5 * (1 + torch.erf(x64 / math.sqrt(2))))
    print(f"  wrong references: ReLU {wf:.2e}, GELU' without x phi(x) {wb:.2e} ({min(wf, wb) / GELU_TOL:.0f}x the bound)")
    assert min(wf, wb) >= 10 * GELU_TOL


# colsum: fp32 sums per thread, per block through shared memory, one fp32 atomic per block and column.  Set from the
# first B200 run: worst 2.1e-7 of the sum of |terms|, so 6e-7 (2.8x).
COLSUM_TOL = 6e-7


@pytest.mark.parametrize("Cc", [8, 64, 128])
@pytest.mark.parametrize("mode", ["plain", "ffn", "mask"])
@pytest.mark.parametrize("rows", [7, 100003])
def test_colsum(cuda_device, Cc, mode, rows):
    lib = _lib.load()
    g = _gen(Cc + rows + len(mode))
    scale = 0.375
    stride = 4 if mode == "ffn" else 1
    x = _h((rows * stride, Cc), g, 1.0, 0.2)
    mask, rps = None, 0
    if mode == "mask":  # rows of 3 samples, the middle one masked
        rps = (rows + 2) // 3
        mask = _mask()
    offsets = range(4) if mode == "ffn" else [0]
    for off in offsets:
        out = torch.zeros(Cc, device="cuda")
        _lib.check(lib.w2s_colsum(x.data_ptr(), out.data_ptr(), rows, Cc, stride, off,
                                  None if mask is None else mask.data_ptr(), rps, scale, G.stream()))
        torch.cuda.synchronize()
        sel = x.to(F64)[off::stride][:rows]
        keep = torch.ones(rows, dtype=torch.bool, device="cuda")
        if mask is not None:
            keep = mask[torch.arange(rows, device="cuda") // rps] == 0
        ref, absref = sel[keep].sum(0) * scale, sel[keep].abs().sum(0) * scale
        err = _red(out, ref, absref)
        print(f"colsum C={Cc} {mode} rows={rows} offset {off}: {err:.2e} (bound {COLSUM_TOL:.0e})")
        assert err < COLSUM_TOL
        if mode == "ffn":
            wrong, what = x.to(F64)[(off + 1) % 4::stride][:rows].sum(0) * scale, "next row offset"
        elif mode == "mask":
            wrong, what = sel.sum(0) * scale, "row mask ignored"
        else:
            wrong, what = ref / scale, "scale dropped"
        werr = _red(out, wrong, absref)
        print(f"  wrong reference ({what}): {werr:.2e} ({werr / COLSUM_TOL:.0f}x the bound)")
        assert werr >= 10 * COLSUM_TOL


# dropout: x / (1 - p) (+ res) in fp32, one fp16 rounding (4.9e-4 relative, and a second rounding of the fp32 sum with
# res).  Set from the first B200 run: worst 3.8e-4, so 1.1e-3 (2.9x).
DROP_TOL = 1.1e-3


def _keep_mask(lib, n, p, seed, site):
    m = torch.empty(n, dtype=torch.uint8, device="cuda")
    _lib.check(lib.w2s_dropout(None, None, None, m.data_ptr(), n, p, seed, site, G.stream()))
    return m


@pytest.mark.parametrize("p", [0.0, 0.1, 0.5])
@pytest.mark.parametrize("with_res", [False, True])
@pytest.mark.parametrize("n", [8, 8 * 250_001])
def test_dropout(cuda_device, p, with_res, n):
    lib = _lib.load()
    seed, site = 1234 + n, 8 * 2 + 2
    g = _gen(n + int(p * 10) + with_res)
    x = _h((n,), g, 2.0)
    res = _h((n,), g) if with_res else None
    out = _full((n,))
    _lib.check(lib.w2s_dropout(x.data_ptr(), None if res is None else res.data_ptr(), out.data_ptr(), None, n, p, seed,
                               site, G.stream()))
    keep = _keep_mask(lib, n, p, seed, site)
    torch.cuda.synchronize()
    kf = keep.to(F64)
    ref = x.to(F64) * kf / (1 - p) + (res.to(F64) if res is not None else 0)
    err = _rel(out, ref)
    print(f"dropout n={n} p={p} res={with_res}: {err:.2e} (bound {DROP_TOL:.0e}), keep rate {kf.mean().item():.5f}")
    assert err < DROP_TOL
    if p == 0.0:
        assert keep.all()
        if res is None:
            assert torch.equal(out, x), "p = 0 must pass x through unchanged"
    if n > 1000:  # keep rate within 5 standard deviations of Binomial(n, 1 - p)
        assert abs(kf.mean().item() - (1 - p)) <= 5 * math.sqrt(max(p * (1 - p), 1e-12) / n)
    if p > 0:
        wrong, what = x.to(F64) * kf + (res.to(F64) if res is not None else 0), "kept values not scaled by 1 / (1 - p)"
    elif res is not None:
        wrong, what = x.to(F64), "res dropped"
    else:
        return  # checked bit for bit above
    werr = _rel(out, wrong)
    print(f"  wrong reference ({what}): {werr:.2e} ({werr / DROP_TOL:.0f}x the bound)")
    assert werr >= 10 * DROP_TOL


# ---------------------------------------------------------------------------------------------------------------------
# argument checks.  Every buffer is large enough that, had the library accepted the call, its launch would have stayed
# inside its allocations.
# ---------------------------------------------------------------------------------------------------------------------
def _plain_call(out_ptr, B, L, cin, cout, x, pk, **kw):
    args = dict(cin=cin, cout=cout, taps=1, stride=1, dilation=1, pad=0, prologue=PRO_NONE, epilogue=EPI_PLAIN, has_ds=0,
                B=B, L_in=L, L_out=L, w=pk, out=out_ptr)
    args["in"] = x
    args.update(kw)
    return _conv_rc(**args)


@pytest.mark.parametrize("case", ["offset_negative", "offset_ge_stride", "last_row_past_out_rows", "out_rows_unset"])
def test_plain_output_rows_refused(cuda_device, case):
    B, L, cin, cout = 2, 37, 32, 16
    g = _gen(5)
    x = _h((B, L, cin), g)
    pk = G.pack_conv(torch.randn(cout, cin, 1, device="cuda"))
    pad_rows = 8  # rows before the pointer handed to the call: room for a row index of -1
    if case == "offset_negative":
        stride, off, rows = 2, -1, 2 * L
    elif case == "offset_ge_stride":
        stride, off, rows = 2, 2, 2 * L + 1
    elif case == "last_row_past_out_rows":
        stride, off, rows = 4, 3, 4 * L - 1
    else:  # out_rows = 0 means L_out: a stride-2 scatter would run past each sample into the next one
        stride, off, rows = 2, 0, 0
    buf = _full((pad_rows + (B + 1) * max(rows, 2 * L) * 2 + 8, cout))
    rc, msg = _plain_call(buf.data_ptr() + pad_rows * cout * 2, B, L, cin, cout, x, pk, out_stride=stride, out_offset=off,
                          out_rows=rows)
    print(f"{case}: rc {rc}, {msg}")
    assert rc != 0 and "W2S_EPI_PLAIN output rows out of range" in msg
    assert f"out_offset={off}" in msg and f"out_rows={rows if rows > 0 else L}" in msg
    assert _untouched(buf), "a refused call must not launch"
    # the same shape with a valid row layout runs
    rc, msg = _plain_call(buf.data_ptr() + pad_rows * cout * 2, B, L, cin, cout, x, pk, out_stride=stride, out_offset=0,
                          out_rows=stride * L)
    assert rc == 0, msg


@pytest.mark.parametrize("C", [24, 256])
def test_enc_kernels_refuse_channel_counts(cuda_device, C):
    lib = _lib.load()
    B, L = 2, 64
    n = (B + 1) * L * max(C, 128) * 2
    big = torch.zeros(n, dtype=F16, device="cuda")  # every tensor argument, oversized: a launch would stay inside
    sums = torch.zeros(n, dtype=F64, device="cuda")
    rc = lib.w2s_enc_act_fwd(big.data_ptr(), None, sums.data_ptr(), big.data_ptr(), None, B, L, C, EPS, G.stream())
    msgs = [("enc_act_fwd", rc, lib.w2s_last_error().decode())]
    rc = lib.w2s_enc_act_bwd(big.data_ptr(), big.data_ptr(), None, sums.data_ptr(), big.data_ptr(), None, sums.data_ptr(),
                             None, None, B, L, C, EPS, G.stream())
    msgs.append(("enc_act_bwd", rc, lib.w2s_last_error().decode()))
    if C == 24:  # (256 channels would overrun the kernel's 512-entry shared-memory constants)
        rc = lib.w2s_enc_norm_bwd(big.data_ptr(), big.data_ptr(), sums.data_ptr(), sums.data_ptr(), big.data_ptr(), None,
                                  B, L, C, 0, EPS, G.stream())
        msgs.append(("enc_norm_bwd", rc, lib.w2s_last_error().decode()))
    torch.cuda.synchronize()
    for name, rc, msg in msgs:
        print(f"{name} C={C}: rc {rc}, {msg}")
        assert rc != 0 and msg.startswith(f"{name}: C={C} (built for 8, 16, 32, 64 or 128 channels)"), (name, msg)


@pytest.mark.parametrize("B,T", [(0, 256), (2, 0), (2, 255)])
def test_first_conv_wgrad_refuses_shapes(cuda_device, B, T):
    lib = _lib.load()
    Tb = max(T, 2) + 2
    x = torch.zeros(3 * Tb, device="cuda")
    d = torch.zeros(3 * Tb * 16, dtype=F16, device="cuda")
    dw1, dwds = torch.zeros(48, device="cuda"), torch.zeros(16, device="cuda")
    rc = lib.w2s_first_conv_wgrad(x.data_ptr(), d.data_ptr(), d.data_ptr(), dw1.data_ptr(), dwds.data_ptr(), None, B, T,
                                  1.0, G.stream())
    torch.cuda.synchronize()
    msg = lib.w2s_last_error().decode()
    print(f"first_conv_wgrad B={B} T={T}: rc {rc}, {msg}")
    assert rc != 0 and msg == f"first_conv_wgrad: B={B} T={T} (needs B > 0 and an even T > 0)"
