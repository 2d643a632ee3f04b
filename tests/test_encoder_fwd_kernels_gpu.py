"""-m gpu: every forward launch form of the signal encoders against an fp64 reference, element by element.

``FORMS`` has one row per kernel instantiation the forward dispatch (``conv_dispatch`` in capi.cu) can reach: the 32
stream-kernel rows (fp16, wide and forced-split storage; ``PRO_NORM``, ``PRO_NORM_RES`` and the block-0 fusion prologues
``PRO_FIR`` / ``PRO_NORM_RES_X``), the paired form of every pairable stream row, the encoder Linear (64 -> 128 and
128 -> 128, single and paired), the ``EPI_STATS`` tile kernels of ``w2s_set_conv_impl(1)`` and ``first_conv`` (the
``keep = 1`` training forward).  ``test_forms_match_dispatcher`` holds the table to the dispatcher's source, and
``test_forward_launches_are_tested_forms`` replays real forwards and requires every launch to be a row, so a form added
later fails until it is tested here.

The reference is computed in fp64 from exactly the bytes a kernel reads: the stored fp16 / fp32 input and residual,
the fp64 ``in_stats`` handed to it (each night with its own offset and scale), the raw fp32 signal with -inf read as 0,
the fp32 block-0 taps and the packed fp16 weights (hi + lo for split operands).  Every output element has a bound of
its own (``_bound``); each test prints its worst ratio error / bound, which must be <= 1.
"""
import ctypes as C
import math
import re
from collections import namedtuple
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

import gpu_utils as G
from wav2sleep_b200 import _lib
from wav2sleep_b200._lib import EPI_BIAS_GELU, EPI_STATS, PRO_FIR, PRO_NORM, PRO_NORM_RES, PRO_NORM_RES_X

F64, F32, F16 = torch.float64, torch.float32, torch.float16
EPS = 1e-2                      # InstanceNorm1d eps of the encoders
ROOT = Path(__file__).resolve().parent.parent
NAN16, NAN32 = 0x7E5B, 0x7FC0A5A5  # NaN bit patterns of memory a call must not write

# Accumulation: the tensor core sums exact fp16 x fp16 products in fp32.  Its error is bounded as
# ACC_C * 2^-23 * sum |A| |w| over the products of the element.  On the first B200 run (NVIDIA B200, 1000 W power
# limit) no element of any form needed this term: every error was already inside the operand and output-rounding
# terms (test_form prints the measured need, which was <= 0 throughout), so ACC_C cannot be fitted from these kernels.
# It is kept at 1, one fp32 rounding of the sum of |terms|.
ACC_C = 1.0

# form: kind stream | tile | linear | first_conv; mt = output rows per tile / 128; ntw = transform warps (stream)
Form = namedtuple("Form", "kind cin cout stride pro ds win wout split mt ntw paired")


def _stream(cin, cout, s, pro, ds, mt, ntw, win=False, wout=False, split=None):
    return Form("stream", cin, cout, s, pro, ds, win, wout, (cin <= 16 and cout <= 16) if split is None else split, mt,
                ntw, False)


N, R, FIR, RX = PRO_NORM, PRO_NORM_RES, PRO_FIR, PRO_NORM_RES_X
STREAM_FORMS = [
    _stream(16, 16, 1, FIR, False, 8, 18), _stream(16, 16, 1, RX, True, 8, 14), _stream(16, 16, 1, N, False, 8, 18),
    _stream(16, 16, 2, N, False, 4, 18), _stream(16, 16, 1, R, True, 4, 14), _stream(16, 32, 1, R, True, 4, 10),
    _stream(32, 32, 1, N, False, 4, 14), _stream(32, 32, 2, N, False, 2, 14), _stream(32, 32, 1, R, True, 2, 10),
    _stream(32, 64, 1, R, True, 2, 14), _stream(64, 64, 1, N, False, 2, 14), _stream(64, 64, 2, N, False, 1, 14),
    _stream(64, 64, 1, R, True, 1, 14), _stream(64, 128, 1, R, True, 1, 14), _stream(128, 128, 1, N, False, 1, 14),
    _stream(128, 128, 2, N, False, 1, 14), _stream(128, 128, 1, R, True, 1, 14),
    # wide (fp32) storage of the leading blocks
    _stream(16, 16, 1, FIR, False, 8, 18, False, True), _stream(16, 16, 1, RX, True, 4, 14, True, True),
    _stream(16, 16, 1, N, False, 6, 18, True, True), _stream(16, 16, 2, N, False, 3, 18, True, True),
    _stream(16, 32, 1, R, True, 4, 10, True, False, False), _stream(16, 32, 1, R, True, 4, 10, True, True, True),
    _stream(32, 32, 1, N, False, 3, 14, True, True, True), _stream(32, 32, 2, N, False, 1, 14, True, True, True),
    _stream(32, 32, 1, R, True, 2, 10, True, True, True), _stream(32, 64, 1, R, True, 2, 14, True, False, False),
    # wide storage + split operands of the 64-channel blocks (wide_blocks = 6)
    _stream(32, 64, 1, R, True, 2, 14, True, True, True), _stream(64, 64, 1, N, False, 1, 14, True, True, True),
    _stream(64, 64, 2, N, False, 1, 14, True, True, True), _stream(64, 64, 1, R, True, 1, 14, True, True, True),
    _stream(64, 128, 1, R, True, 1, 14, True, False, False),
]
PAIRED_FORMS = [f._replace(paired=True) for f in STREAM_FORMS if not (f.cout == 128 and f.ds)]  # stream_pairable
LINEAR_FORMS = [Form("linear", cin, 128, 4, R, False, False, False, False, 1, 0, p) for cin in (64, 128) for p in (False, True)]
TILE_FORMS = ([Form("tile", ci, co, s, R, True, False, False, ci <= 16 and co <= 16, 0, 0, False)
               for ci, co in ((16, 16), (16, 32), (32, 32), (32, 64), (64, 64), (64, 128), (128, 128)) for s in (1,)]
              + [Form("tile", c, c, s, N, False, False, False, c <= 16, 0, 0, False) for c in (16, 32, 64, 128) for s in (1, 2)])
FIRST_CONV_FORM = Form("first_conv", 1, 16, 1, 0, True, False, False, False, 0, 0, False)
FORMS = STREAM_FORMS + PAIRED_FORMS + LINEAR_FORMS + TILE_FORMS + [FIRST_CONV_FORM]


def _form_id(f):
    pro = {N: "norm", R: "res", FIR: "fir", RX: "resx"}.get(f.pro, "-")
    st = ("w" + ("32" if f.win else "16") + ("32" if f.wout else "16")) if (f.win or f.wout) else "h"
    return (f"{f.kind}{'x2' if f.paired else ''}-c{f.cin}-{f.cout}-s{f.stride}-{pro}{'-ds' if f.ds else ''}-{st}"
            + ("-split" if f.split else ""))


def _launch_key(f):
    """What a profile label says about a launch of the form: (cin, cout, taps, stride, prologue, epilogue, ds, wide, x2)."""
    if f.kind == "first_conv":
        return ("first_conv",)
    wide = (" w32/32" if f.wout else " w32/16") if f.win else (" w16/32" if f.wout else "")
    taps, epi = (4, EPI_BIAS_GELU) if f.kind == "linear" else (3, EPI_STATS)
    return (f.cin, f.cout, taps, f.stride, f.pro, epi, f.ds, wide, f.paired)


LABEL = re.compile(r"conv c(\d+)->(\d+) k(\d+) s(\d+) d\d+ pro(\d+) epi(\d+)( \+ds)?( w\d+/\d+)?( x2)? B\d+ L\d+")


def _label_key(label):
    if label.startswith("first_conv"):
        return ("first_conv",)
    m = LABEL.fullmatch(label)
    assert m, label
    ci, co, k, s, pro, epi = (int(v) for v in m.groups()[:6])
    return (ci, co, k, s, pro, epi, bool(m.group(7)), m.group(8) or "", bool(m.group(9)))


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the table against the dispatcher's source
# ----------------------------------------------------------------------------------------------------------------------
def _dispatch_source():
    src = (ROOT / "wav2sleep_b200" / "csrc" / "capi.cu").read_text()
    body = src[src.index("int conv_dispatch("):]
    return body[:body.index("\n}\n")]


def test_forms_match_dispatcher():
    body = _dispatch_source()
    pro = {"PRO_NORM": N, "PRO_NORM_RES": R, "PRO_FIR": FIR, "PRO_NORM_RES_X": RX}
    tf = {"true": True, "false": False}
    rows = set()
    for macro, args in re.findall(r"^\s*(W2S_STREAM[WX]?)\((\d[^)]*)\)", body, flags=re.M):
        a = [v.strip() for v in args.split(",")]
        cin, cout, s, mt, ntw = int(a[0]), int(a[1]), int(a[2]), int(a[5]), int(a[8])
        win, wout = (tf[a[9]], tf[a[10]]) if macro != "W2S_STREAM" else (False, False)
        split = tf[a[11]] if macro == "W2S_STREAMX" else (cin <= 16 and cout <= 16)
        rows.add(Form("stream", cin, cout, s, pro[a[3]], tf[a[4]], win, wout, split, mt, ntw, False))
    assert len(rows) == 32
    assert rows == set(STREAM_FORMS), (rows ^ set(STREAM_FORMS))
    assert len(STREAM_FORMS) == 32
    # stream_pairable(cout, has_ds) = !(cout == 128 && has_ds)
    hdr = (ROOT / "wav2sleep_b200" / "csrc" / "conv_igemm.cuh").read_text()
    assert "stream_pairable(int cout, bool has_ds) { return !(cout == 128 && has_ds); }" in hdr
    cases = re.findall(r"W2S_CASE\((\d+), (\d+), (\d+), \d+, (PRO_\w+), (EPI_\w+), (true|false)\)", body)
    lin = {(int(ci), int(co)) for ci, co, k, p, e, ds in cases if e == "EPI_BIAS_GELU"}
    assert lin == {(f.cin, f.cout) for f in LINEAR_FORMS} and len(LINEAR_FORMS) == 2 * len(lin)
    assert "launch_conv_igemm_pair<64, 128, 4, 4, PRO_NORM_RES, EPI_BIAS_GELU" in body
    assert "launch_conv_igemm_pair<128, 128, 4, 2, PRO_NORM_RES, EPI_BIAS_GELU" in body
    tile = {(int(ci), int(co), pro[p], tf[ds]) for ci, co, k, p, e, ds in cases if e == "EPI_STATS"}
    assert tile == {(f.cin, f.cout, f.pro, f.ds) for f in TILE_FORMS}
    assert len({_form_id(f) for f in FORMS}) == len(FORMS)


def test_dispatch_refusals_and_split_policy_on_cpu():
    """Calls the kernels cannot run fail with their shape in the message, before any device work (no GPU needed), and
    the encoder's split-operand policy is the one the wide rows of FORMS are built with."""
    lib = _lib.load()
    assert lib.w2s_conv1d_fwd_pair(None, None, None) != 0 and b"null" in lib.w2s_last_error()
    # the block-0 fusion prologues copy raw-signal rows in 16-byte pieces: T_raw must be a multiple of 4
    c = _lib.ConvCall()
    c.cin, c.cout, c.taps, c.stride, c.dilation, c.pad = 16, 16, 3, 1, 1, 1
    c.prologue, c.epilogue, c.B, c.L_in, c.L_out, c.T_raw, c.x_raw = PRO_FIR, EPI_STATS, 2, 38, 38, 38, 256
    assert lib.w2s_conv1d_fwd(C.byref(c), None) != 0
    assert "T_raw that is a multiple of 4" in lib.w2s_last_error().decode() and "T_raw=38" in lib.w2s_last_error().decode()
    # ... and need x_raw on both calls of a pair (the pairing rule compares T_raw, not pointers)
    c.L_in = c.L_out = c.T_raw = 40
    c1 = _lib.ConvCall.from_buffer_copy(c)
    c1.x_raw = None
    assert lib.w2s_conv1d_fwd_pair(C.byref(c), C.byref(c1), None) != 0
    assert "need x_raw" in lib.w2s_last_error().decode()
    # split operands: every conv with cin, cout <= 16; in the wide blocks of deep encoders every conv with cin, cout <= 64
    for wb in (0, 2, 4, 6):
        for block in range(10):
            for cin, cout in ((16, 16), (16, 32), (32, 32), (32, 64), (64, 64), (64, 128), (128, 128)):
                want = (cin <= 16 and cout <= 16) or (block < wb and cout <= 64)
                assert lib.w2s_encoder_conv_split(wb, block, cin, cout) == int(want), (wb, block, cin, cout)
    assert all(f.split == (f.cin <= 16 and f.cout <= 16 or (f.wout and f.cout <= 64)) for f in STREAM_FORMS if f.win or f.wout)


# ----------------------------------------------------------------------------------------------------------------------
# fp64 reference and per-element bound
# ----------------------------------------------------------------------------------------------------------------------
# GELU of the prologues against the exact erf form.  Both fitted forms are within 2.53e-5 of it in exact arithmetic
# (evaluated in fp64 on a 3e-5 grid over [-30, 30]); GFIT = 2.6e-5.
#   stream kernels, gelu_fast2: 0.5 x (1 + tanh.approx(u)); tanh.approx has 2^-11 relative error, so + 2^-12 |x|, and
#     fp32 rounding of t, q, u and the final FMA adds < 2^-22 (|x| + 1);
#   tile kernel, gelu_fast: the fp32 exponent argument xc q (|xc q| <= 28, polynomial and product within 3 x 2^-24)
#     is off by up to 5e-6, which changes x / (1 + e) by up to 0.25 |x| 3.5e-6; with ex2.approx (2^-22 relative) and
#     __fdividef (2 ulp): + 2^-19 (|x| + 1).
GFIT = 2.6e-5


def _gelu_err(x, stream):
    return GFIT + (2.0 ** -12 * x.abs() + 2.0 ** -22 * (x.abs() + 1) if stream else 2.0 ** -19 * (x.abs() + 1))


def _gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _unpack(p, cout, cin, taps, split, taps_major=False):
    """Packed weights ([hi|lo][tap][cin/8][cout][8], the layout test_pack_conv_weight_layout pins) -> fp64 [cout, cin, taps]
    (hi + lo).  taps_major (the Linear): input index tap * cin + c, returned as [cout, cin, taps] of the conv view."""
    w = p.view(2 if split else 1, taps, cin // 8, cout, 8).double().sum(0)   # [tap][cin/8][cout][8]
    return w.permute(2, 1, 3, 0).reshape(cout, cin, taps).contiguous()


def _ulp16(a):
    """fp16 unit in the last place at |a| (the larger one across a power of two), subnormals included."""
    m = a.abs().clamp_min(2.0 ** -14)
    return torch.exp2(torch.floor(torch.log2(m * (1 + 2.0 ** -10))) - 10)


def _operand(A, delta, split):
    """The MMA operand the reference uses and u, how far the kernel's operand can be from it, per element.
    fp16: the kernel rounds its own a = A +- delta.  Away from an fp16 rounding midpoint by more than delta it rounds
    to fp16(A) exactly (u = 0); within delta of one it may round to the neighbour (u = the fp16 spacing there), and
    where delta reaches half that spacing it may land anywhere in [A - delta, A + delta] rounded (u = delta + ulp).
    split (hi + lo fp16 pairs): hi + lo represents a to 2^-22 |a| (+ 2^-25 where lo is subnormal), and the dropped
    lo x lo_w product is below 2^-11 |a| x 2^-11 |w|: u = delta + 2^-21 |A| + 2^-25."""
    if split:
        return A, delta + 2.0 ** -21 * A.abs() + 2.0 ** -25
    A16 = A.half().double()
    # spacing between fp16(A) and its neighbour on A's side: below a power of two it is half the spacing above, so it is
    # taken at the smaller of |A|, |fp16(A)| (just under it when they are equal)
    gap = torch.exp2(torch.floor(torch.log2((torch.minimum(A.abs(), A16.abs()) * (1 - 2.0 ** -12)).clamp_min(2.0 ** -14))) - 10)
    near = (gap / 2 - (A - A16).abs()) <= delta
    u = torch.where(near, torch.where(delta < gap / 2, gap, delta + _ulp16(A.abs() + delta)), torch.zeros_like(A))
    return A16, u


def _norm_consts(stats, L):
    mean = stats[..., 0] / L
    var = (stats[..., 1] / L - mean * mean).clamp_min(0)
    return mean[:, None, :], (1.0 / torch.sqrt(var + EPS))[:, None, :]


def _prologue(f, side, L_in, wrong=None):
    """Activated conv input A [B, L_in, cin] (fp64) and delta, the bound on |kernel's fp32 value - A|.

    Affine x_hat = fma(y, rstd, -mean * rstd) in fp32: rstd = 1 / sqrt((float)(var + eps)) is within 2^-21 (fp32 cast,
    sqrt, reciprocal), -mean * rstd within 2^-22 + 2^-21 of |mean| rstd, and the FMA rounds to 2^-24 |x_hat|:
    e_aff = 2^-20 (|y| + |mean|) rstd + 2^-23 |x_hat|.  PRO_FIR: |y| is sum_t |w_t x_t| (three FMAs of taps pre-scaled
    by rstd in fp32).  The first GELU gives delta1 = gelu_err(x_hat) + 1.13 e_aff (|GELU'| <= 1.13); the residual
    prologues add r (PRO_NORM_RES, rounding 2^-24 |s|) or fma(w_ds, x[2i], a) (PRO_NORM_RES_X, 2^-24 |s|) and apply
    the second GELU: delta = gelu_err(s) + 1.13 (delta1 + 2^-23 |s|)."""
    stream = f.kind == "stream"
    st = side["stats"]
    if wrong == "stats":
        st = st.roll(1, 0)
    mean, rstd = _norm_consts(st, L_in)
    if f.pro == FIR:
        x = side["xz"]
        taps = side["w_first"].double()                       # [16, 3]
        xp = F.pad(x, (1, 1))
        cols = torch.stack([xp[:, t:t + L_in] for t in range(3)], -1)           # [B, L, 3]
        if wrong == "tap":
            cols = torch.stack([xp[:, t + 1:t + 1 + L_in] if t < 2 else xp[:, t:t + L_in] for t in range(3)], -1)
        if wrong == "inf":
            xr = F.pad(side["x"].double(), (1, 1))
            cols = torch.stack([xr[:, t:t + L_in] for t in range(3)], -1)
        y = cols @ taps.t()
        yabs = cols.abs() @ taps.abs().t()
    else:
        y = side["y"].double()
        yabs = y.abs()
    xh = (y - mean) * rstd
    e_aff = 2.0 ** -20 * (yabs + mean.abs()) * rstd + 2.0 ** -23 * xh.abs()
    a = _gelu(xh)
    d = _gelu_err(xh, stream) + 1.13 * e_aff
    if f.pro in (R, RX):
        if f.pro == R:
            s = a + side["r"].double()
        else:
            xr = side["xz"][:, 1::2] if wrong == "odd_x" else side["xz"][:, 0::2]
            s = a + xr[:, :L_in, None] * side["w_first_ds"].double()
        d = _gelu_err(s, stream) + 1.13 * (d + 2.0 ** -23 * s.abs())
        a = _gelu(s)
    return a, d


def _conv(A, W, stride, pad):
    return F.conv1d(A.transpose(1, 2), W, stride=stride, padding=pad).transpose(1, 2)


def _reference(f, side, L_in, L_out, wrong=None):
    """Reference outputs and their error bounds E (before output rounding): dict out / ds -> (ref, E, acc)."""
    A, delta = _prologue(f, side, L_in, wrong)
    Aop, u = _operand(A, delta, f.split)
    W, Wa = side["W"], side["W"].abs()
    if wrong == "tap":
        W = W.roll(1, 2)
    taps, stride, pad = (4, 4, 0) if f.kind == "linear" else (3, f.stride, 1)
    res = {}
    ref = _conv(Aop, W, stride, pad)
    if wrong == "rows" and f.stride == 2:
        ref = _conv(F.pad(Aop, (0, 0, 0, 1))[:, 1:], W, stride, pad)
    acc = _conv(Aop.abs(), Wa, stride, pad)
    E = _conv(u, Wa, stride, pad) + ACC_C * 2.0 ** -23 * acc
    res["out"] = (ref[:, :L_out], E[:, :L_out], acc[:, :L_out])
    if f.ds and L_out // 2 == 0:  # L_out = 1: out_ds has no rows
        z = Aop.new_zeros(Aop.shape[0], 0, f.cout)
        res["ds"] = (z, z, z)
    elif f.ds:
        Wd, Wda = side["Wd"], side["Wd"].abs()
        sel = slice(1, None, 2) if wrong == "odd_ds" else slice(0, None, 2)
        Ad, ud = Aop[:, sel][:, :L_out // 2], u[:, sel][:, :L_out // 2]
        if Ad.shape[1] < L_out // 2:
            Ad, ud = F.pad(Ad, (0, 0, 0, 1)), F.pad(ud, (0, 0, 0, 1))
        accd = _conv(Ad.abs(), Wda, 1, 0)
        res["ds"] = (_conv(Ad, Wd, 1, 0), _conv(ud, Wda, 1, 0) + ACC_C * 2.0 ** -23 * accd, accd)
    return res


def _out_bound(ref, E, wide):
    """Stored output: the value is within E of ref, then rounded once to fp16 (2^-11 relative, 2^-25 below the normal
    range) or fp32 (2^-24 relative)."""
    if wide:
        return E * (1 + 2.0 ** -24) + 2.0 ** -24 * ref.abs() + 1e-44
    return E * (1 + 2.0 ** -11) + 2.0 ** -11 * ref.abs() + 2.0 ** -25


def _linear_bound(pre, E):
    """Linear epilogue: gelu_erf(acc + bias) in fp32 (erff within 2 ulp, the bias add 2^-24), stored fp16:
    1.13 (E + 2^-24 |pre|) + 2^-21 (|pre| + 1), then the fp16 rounding of the result."""
    g = _gelu(pre)
    e = 1.13 * (E + 2.0 ** -24 * pre.abs()) + 2.0 ** -21 * (pre.abs() + 1)
    return g, e * (1 + 2.0 ** -11) + 2.0 ** -11 * g.abs() + 2.0 ** -25


# ----------------------------------------------------------------------------------------------------------------------
# one launch: inputs, prefilled outputs, call, checks
# ----------------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _lengths(f, L_out, odd_in=False):
    """(L_in, L_out).  Stride 2 with odd_in: L_in = 2 L_out - 1, so the last output row reads the right zero-padding row."""
    if f.kind == "linear":
        return 4 * L_out, L_out
    return (2 * L_out - (1 if odd_in else 0), L_out) if f.stride == 2 else (L_out, L_out)


def _side(f, B, L_in, seed, inf_at=()):
    """Inputs of one call.  Each night has its own offset and scale (so another night's norm constants show up)."""
    g = _gen(seed)
    dev = "cuda"
    store = F32 if f.win else F16
    side = {}
    off = torch.randn(B, 1, 1, generator=g, device=dev) * 2.0
    sc = torch.rand(B, 1, 1, generator=g, device=dev) * 2.5 + 0.5
    if f.pro == FIR:
        T = L_in
        x = torch.randn(B, T, generator=g, device=dev) * sc[:, :, 0] + off[:, :, 0] * 0.2
        for p in inf_at:
            if 0 < p < T:
                x[:, p] = float("-inf")
        side["x"] = x
        side["xz"] = torch.where(torch.isinf(x), torch.zeros_like(x), x).double()
        side["w_first"] = torch.randn(16, 3, generator=g, device=dev) * 0.5
        xp = F.pad(side["xz"], (1, 1))
        h = torch.stack([xp[:, t:t + T] for t in range(3)], -1) @ side["w_first"].double().t()
        side["stats"] = torch.stack([h.sum(1), (h * h).sum(1)], -1).contiguous()
    else:
        y = (torch.randn(B, L_in, f.cin, generator=g, device=dev) * sc + off).to(store)
        side["y"] = y
        yd = y.double()
        side["stats"] = torch.stack([yd.sum(1), (yd * yd).sum(1)], -1).contiguous()
        if f.pro == R:
            side["r"] = torch.randn(B, L_in, f.cin, generator=g, device=dev).to(store)
        if f.pro == RX:
            T = 2 * L_in
            x = torch.randn(B, T, generator=g, device=dev)
            for p in inf_at:
                if 0 < p < T:
                    x[:, p] = float("-inf")
            side["x"] = x
            side["xz"] = torch.where(torch.isinf(x), torch.zeros_like(x), x).double()
            side["w_first_ds"] = torch.randn(16, generator=g, device=dev)
    if f.kind == "linear":
        w = torch.randn(128, 4 * f.cin, generator=g, device=dev) / (4 * f.cin) ** 0.5
        side["pw"] = G.pack_conv(w, taps_major=1, taps=4)
        side["W"] = _unpack(side["pw"], 128, f.cin, 4, False)
        side["bias"] = torch.randn(128, generator=g, device=dev) * 0.3
    else:
        w = torch.randn(f.cout, f.cin, 3, generator=g, device=dev) / (3 * f.cin) ** 0.5
        side["pw"] = G.pack_conv(w, split=int(f.split))
        side["W"] = _unpack(side["pw"], f.cout, f.cin, 3, f.split)
        if f.ds:
            wd = torch.randn(f.cout, f.cin, 1, generator=g, device=dev) / f.cin ** 0.5
            side["pwd"] = G.pack_conv(wd, split=int(f.split))
            side["Wd"] = _unpack(side["pwd"], f.cout, f.cin, 1, f.split)
    return side


def _guard(cols, wide):
    """Guard rows on each side of an output tensor: 256 bytes, so that the tensor keeps the allocator's alignment."""
    return 256 // (cols * (4 if wide else 2))


def _nan_buf(rows, cols, wide):
    """[rows + 2 g, cols] of a NaN bit pattern: the first and last g rows guard the call's tensor (rows g .. g + rows)."""
    n = rows + 2 * _guard(cols, wide)
    if wide:
        return torch.full((n * cols,), NAN32, dtype=torch.int32, device="cuda").view(F32).view(n, cols)
    return torch.full((n * cols,), NAN16, dtype=torch.int16, device="cuda").view(F16).view(n, cols)


def _inner(f, buf):
    g = _guard(f.cout, f.wout)
    return buf[g:buf.shape[0] - g]


def _bits(t):
    return t.view(torch.int32 if t.dtype == F32 else torch.int16).clone()


def _call(f, side, B, L_in, L_out, mask, seed):
    """Output buffers (prefilled) and the w2s_conv_call of one side."""
    g = _gen(seed + 99)
    wide = f.wout
    o = {"out": _nan_buf(B * L_out, f.cout, wide)}
    if f.ds:
        o["ds"] = _nan_buf(B * (L_out // 2), f.cout, wide)
    if f.kind != "linear":
        o["stats"] = torch.randn(B, f.cout, 2, generator=g, device="cuda", dtype=F64) * 100
    o["before"] = {k: (_bits(v) if k != "stats" else v.clone()) for k, v in o.items()}
    c = _lib.ConvCall()
    taps, stride, pad = (4, 4, 0) if f.kind == "linear" else (3, f.stride, 1)
    c.cin, c.cout, c.taps, c.stride, c.dilation, c.pad = f.cin, f.cout, taps, stride, 1, pad
    c.prologue, c.epilogue, c.has_ds = f.pro, EPI_BIAS_GELU if f.kind == "linear" else EPI_STATS, int(f.ds)
    c.B, c.L_in, c.L_out, c.in_eps = B, L_in, L_out, EPS
    c.in_stats = side["stats"].data_ptr()
    if "y" in side:
        c.in_ = side["y"].data_ptr()
    if "r" in side:
        c.in_res = side["r"].data_ptr()
    if "x" in side:
        c.x_raw, c.T_raw = side["x"].data_ptr(), side["x"].shape[1]
    if "w_first" in side:
        c.w_first = side["w_first"].data_ptr()
    if "w_first_ds" in side:
        c.w_first_ds = side["w_first_ds"].data_ptr()
    c.w = side["pw"].data_ptr()
    if f.ds:
        c.w_ds = side["pwd"].data_ptr()
        c.out_ds = _inner(f, o["ds"]).data_ptr()
    if "bias" in side:
        c.bias = side["bias"].data_ptr()
    c.out = _inner(f, o["out"]).data_ptr()
    if "stats" in o:
        c.out_stats = o["stats"].data_ptr()
    if mask is not None:
        c.row_mask = mask.data_ptr()
    c.in_wide, c.out_wide = int(f.win), int(f.wout)
    c.force_split = int(f.split and not (f.cin <= 16 and f.cout <= 16))
    o["mask"] = mask
    return c, o


def _launch(f, calls):
    lib = _lib.load()
    if f.kind == "tile":
        _lib.check(lib.w2s_set_conv_impl(1))
    try:
        if len(calls) == 2:
            rc = lib.w2s_conv1d_fwd_pair(C.byref(calls[0]), C.byref(calls[1]), G.stream())
        else:
            rc = lib.w2s_conv1d_fwd(C.byref(calls[0]), G.stream())
        torch.cuda.synchronize()
    finally:
        lib.w2s_set_conv_impl(0)
    assert rc == 0, lib.w2s_last_error().decode()


def _lanes_rows(f, B, L_out, mask, pair=None):
    """Rows one epilogue lane sums in fp32 for one night, plus the 5 butterfly levels and the fp32 adds across tiles.
    Stream kernels: a lane takes MT rows per tile, over at most ceil(live tiles / CTAs of its group) tiles, with the
    grid and the split of a paired launch between its groups computed as launch_conv_stream / conv_stream_kernel do
    (pair = (group, row_mask of group 0, row_mask of group 1)).  Tile kernel: one tile."""
    if f.kind == "tile":  # squares rounded, 5 butterfly levels, then MT x 4 <= 32 slots summed in fp32
        return 1 + 5 + 32
    pos = 128 * f.mt
    tps = (L_out + pos - 1) // pos
    total = tps * B
    ctas = torch.cuda.get_device_properties(0).multi_processor_count * (2 if 32 * (6 + f.ntw) <= 384 else 1)
    compact = mask is not None and B <= 120  # live-night list (kMaxLive = 120)
    n_live = lambda m: B if m is None else int((m == 0).sum())
    if pair is None:
        nctas, live = min(total, ctas), n_live(mask)
    else:
        group, m0, m1 = pair
        grid = 2 * min(total, ctas // 2)
        ctas0 = grid >> 1
        n0, n1 = n_live(m0), n_live(m1)
        if compact and n0 != n1:
            ctas0 = (grid * n0 + ((n0 + n1) >> 1)) // (n0 + n1)
            if n0 > 0 and ctas0 < 1:
                ctas0 = 1
            if n1 > 0 and ctas0 > grid - 1:
                ctas0 = grid - 1
        nctas, live = (ctas0, n0) if group == 0 else (grid - ctas0, n1)
    live_tiles = (live if compact else B) * tps
    if live_tiles == 0 or nctas <= 0:
        return 8
    return 2 * f.mt * (-(-live_tiles // nctas)) + 8


def _check(tag, f, side, o, B, L_in, L_out, wrong=None, pair=None):
    """Per-element check of one side; returns the worst ratio error / bound (over outputs and statistics)."""
    mask = o["mask"]
    live = [b for b in range(B) if mask is None or not bool(mask[b])]
    dead = [b for b in range(B) if b not in live]
    refs = _reference(f, side, L_in, L_out, wrong)
    worst = 0.0
    for key in ("out", "ds"):
        if key not in o:
            continue
        buf, rows = o[key], (L_out if key == "out" else L_out // 2)
        got = _inner(f, buf).view(B, rows, f.cout)
        # memory the call does not address: guard rows, masked nights
        bb, gr = o["before"][key], _guard(f.cout, f.wout)
        assert torch.equal(_bits(buf[:gr]), bb[:gr]) and torch.equal(_bits(buf[-gr:]), bb[-gr:]), f"{tag} {key}: guard row written"
        if dead:
            assert torch.equal(_bits(got[dead]), _inner(f, bb).view(B, rows, f.cout)[dead]), f"{tag} {key}: masked night written"
        if not live or rows == 0:
            continue
        ref, E, _ = refs[key]
        ref, E = ref[live], E[live]
        if f.kind == "linear":
            ref, bound = _linear_bound(ref + side["bias"].double(), E)
        else:
            bound = _out_bound(ref, E, f.wout)
        v = got[live].double()
        ratio = ((v - ref).abs() / bound).nan_to_num(nan=float("inf"))
        if ratio.max().item() > 1 and wrong is None:
            i = int(ratio.argmax())
            print(f"{tag} {key}: ratio {ratio.max().item():.3f} at {list(torch.unravel_index(torch.tensor(i), ratio.shape))} "
                  f"got {v.flatten()[i].item():.6g} ref {ref.flatten()[i].item():.6g} bound {bound.flatten()[i].item():.3g}")
        worst = max(worst, ratio.max().item())
    if "stats" in o and live:
        ref, E, _ = refs["out"]
        ref, E = ref[live], E[live]
        n = _lanes_rows(f, B, L_out, mask, pair)
        got = o["stats"][live] - o["before"]["stats"][live]
        pre = o["before"]["stats"][live].abs()
        s_ref, q_ref = ref.sum(1), (ref * ref).sum(1)
        s_b = E.sum(1) + n * 2.0 ** -24 * ref.abs().sum(1) + 2.0 ** -50 * (pre[..., 0] + ref.abs().sum(1))
        q_b = (2 * ref.abs() * E + E * E).sum(1) + n * 2.0 ** -23 * q_ref + 2.0 ** -50 * (pre[..., 1] + q_ref)
        rs = ((got[..., 0] - s_ref).abs() / s_b).max().item()
        rq = ((got[..., 1] - q_ref).abs() / q_b).max().item()
        if max(rs, rq) > 1 and wrong is None:
            print(f"{tag} stats: sum {rs:.3f} sumsq {rq:.3f} (n {n})")
        worst = max(worst, rs, rq)
        if dead:
            assert torch.equal(o["stats"][dead], o["before"]["stats"][dead]), f"{tag}: masked night's statistics written"
    return worst


def _acc_need(f, side, o, B, L_in, L_out):
    """Measured accumulation constant: max over elements of (|err| - bound without accumulation) / (2^-23 sum |A||w|)."""
    global ACC_C
    saved, ACC_C = ACC_C, 0.0
    try:
        mask = o["mask"]
        live = [b for b in range(B) if mask is None or not bool(mask[b])]
        if not live:
            return 0.0
        ref, E, acc = _reference(f, side, L_in, L_out)["out"]
        ref, E, acc = ref[live], E[live], acc[live]
        if f.kind == "linear":
            ref, bound = _linear_bound(ref + side["bias"].double(), E)
            acc = acc * 1.13
        else:
            bound = _out_bound(ref, E, f.wout)
        v = _inner(f, o["out"]).view(B, L_out, f.cout)[live].double()
        return (((v - ref).abs() - bound) / (2.0 ** -23 * acc).clamp_min(1e-300)).max().item()
    finally:
        ACC_C = saved


def _pos(f):
    return 128 * f.mt if f.kind == "stream" else 128


def _case_lengths(f):
    """Output lengths: a 1-epoch night at the deepest block (8 rows; 1 for the Linear), below one tile, a tile +-1
    (+-4 / +-2 for the block-0 fusion prologues), several tiles with an edge tile at each end; odd lengths with out_ds."""
    if f.kind == "linear":
        return [1, 37, 127, 128, 129, 300]
    P = _pos(f)
    # raw-signal rows are copied in 16-byte pieces: T_raw = L_in (PRO_FIR) or 2 L_in (PRO_NORM_RES_X) is a multiple of 4
    d = 4 if f.pro == FIR else 2 if f.pro == RX else 1
    e = 36 if f.pro == FIR else 38
    ls = [8 if f.stride == 1 else 4, e, P - d, P, P + d, 3 * P + e]
    return ls + ([2998 if f.pro == RX else 2999] if f.ds else [])


def _inf_positions(f, T):
    P = _pos(f)
    return sorted({1, 2, 3, 4, T - 2, T - 1, P - 1, P, P + 1, 2 * P - 2, 2 * P, 2 * P + 2, 4 * P, T // 2, T // 2 + 1})


def _masks(B, kind):
    m = torch.zeros(B, dtype=torch.uint8, device="cuda")
    if kind == "middle":
        m[B // 2] = 1
    elif kind == "all":
        m[:] = 1
    elif kind == "every3":
        m[1::3] = 1
    elif kind == "one_live":
        m[:] = 1
        m[B // 2] = 0
    elif kind == "null":
        return None
    return m  # "none": a mask with every night live


def _run_single(f, B, L_out, mkind, seed, wrong=None, odd_in=False):
    L_in, L_out = _lengths(f, L_out, odd_in)
    side = _side(f, B, L_in, seed, _inf_positions(f, L_in if f.pro == FIR else 2 * L_in))
    c, o = _call(f, side, B, L_in, L_out, _masks(B, mkind), seed)
    _launch(f, [c])
    tag = f"{_form_id(f)} B={B} L_in={L_in} L_out={L_out} mask={mkind}"
    return _check(tag, f, side, o, B, L_in, L_out, wrong), _acc_need(f, side, o, B, L_in, L_out)


def _run_pair(f, B, L_out, mk0, mk1, seed, wrong_side1=False, odd_in=False):
    """Paired launch of two sides with different inputs, weights, raw signals, taps and masks: outputs bitwise equal to
    two single launches, each side within its fp64 bound."""
    L_in, L_out = _lengths(f, L_out, odd_in)
    T = L_in if f.pro == FIR else 2 * L_in
    sides = [_side(f, B, L_in, seed, _inf_positions(f, T)), _side(f, B, L_in, seed + 1, _inf_positions(f, T)[::2])]
    masks = [_masks(B, mk0), _masks(B, mk1)]
    single = [_call(f, s, B, L_in, L_out, m, seed + 10 * i) for i, (s, m) in enumerate(zip(sides, masks))]
    for c, _ in single:
        _launch(f, [c])
    pair = [_call(f, s, B, L_in, L_out, m, seed + 10 * i) for i, (s, m) in enumerate(zip(sides, masks))]
    _launch(f, [pair[0][0], pair[1][0]])
    tag = f"{_form_id(f)} B={B} L_in={L_in} L_out={L_out} masks={mk0}/{mk1}"
    worst, need = 0.0, 0.0
    for i in range(2):
        so, po = single[i][1], pair[i][1]
        for k in ("out", "ds"):
            if k in so:
                # per-tile arithmetic does not depend on which CTA owns the tile
                assert torch.equal(_bits(so[k]), _bits(po[k])), f"{tag} side {i} {k}: paired != single"
        # out_stats: each lane's fp32 partial sums cover the tiles of its CTA, and a paired launch splits the grid
        # differently from a single one, so the two agree within the fp32 partial-sum term, not to fp64 reordering;
        # each side is held to the statistics bound in _check
        worst = max(worst, _check(f"{tag} side {i} paired", f, sides[i], po, B, L_in, L_out, pair=(i, *masks)))
        need = max(need, _acc_need(f, sides[i], po, B, L_in, L_out))
    wrong = None
    if wrong_side1:  # group 1 computed with group 0's raw signal and block-0 taps
        s1 = dict(sides[1])
        for k in ("x", "xz", "w_first", "w_first_ds"):
            if k in sides[0]:
                s1[k] = sides[0][k]
        wrong = _check(f"{tag} side 1 with side 0's raw inputs", f, s1, pair[1][1], B, L_in, L_out, pair=(1, *masks))
    return worst, need, wrong


@pytest.mark.gpu
@pytest.mark.parametrize("f", [f for f in FORMS if f.kind != "first_conv"], ids=_form_id)
def test_form(cuda_device, f):
    """Every length of _case_lengths over 3 nights with the middle one masked, then row_mask NULL, all nights masked,
    and 120 / 121 nights (the stream kernels compact up to 120 live nights and skip masked tiles one by one above).
    Stride 2 also with an odd L_in (L_out = (L_in + 1) / 2), whose last output row reads the right padding row."""
    worst, need = 0.0, 0.0
    seed = f.cin * 31 + f.cout * 7 + f.stride + f.pro * 1000 + int(f.win) * 10 + int(f.wout) * 20 + int(f.split) * 40
    if f.paired:
        cases = [(3, L, "middle", "middle") for L in _case_lengths(f)]
        P = _pos(f)
        cases += [(5, P + 36, "one_live", "none"), (3, 2 * P + 36, "all", "middle"), (3, 40, "null", "null"),
                  (121, 2 * P + 36, "every3", "middle"), (120, 40, "every3", "one_live")]
        odd = [(3, L, "middle", "none") for L in (4, P - 1, P, P + 1, 3 * P + 38)] + [(121, 2 * P + 36, "every3", "middle")]
        for B, L, m0, m1, odd_in in [c + (False,) for c in cases] + [c + (True,) for c in (odd if f.stride == 2 else [])]:
            w, n, _ = _run_pair(f, B, L, m0, m1, seed + B + L, odd_in=odd_in)
            worst, need = max(worst, w), max(need, n)
    else:
        cases = [(3, L, "middle") for L in _case_lengths(f)]
        # 121 nights of 3 tiles: more tiles than CTAs, so CTA tile ranges cross from one night into the next
        cases += [(2, _pos(f) + 36, "null"), (2, 40, "all"), (120, 40, "every3"), (121, 2 * _pos(f) + 36, "every3")]
        P = _pos(f)
        odd = [(3, L, "middle") for L in (4, P - 1, P, P + 1, 3 * P + 38)] + [(121, 2 * P + 36, "every3"), (2, P + 1, "null")]
        for B, L, m, odd_in in [c + (False,) for c in cases] + [c + (True,) for c in (odd if f.stride == 2 else [])]:
            w, n = _run_single(f, B, L, m, seed + B + L, odd_in=odd_in)
            worst, need = max(worst, w), max(need, n)
    print(f"{_form_id(f)}: worst error / bound {worst:.3f}, accumulation constant needed {need:.4f} (ACC_C {ACC_C})")
    assert worst <= 1.0


def _find(kind, **kw):
    return next(f for f in FORMS if f.kind == kind and all(getattr(f, k) == v for k, v in kw.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("defect", ["tap", "inf", "odd_x", "stats", "rows", "odd_ds", "pair_raw"])
def test_wrong_references_miss(cuda_device, defect):
    """A plausible defect must exceed 10x the bound on the case built to show it: a tap shifted by one row, a -inf not
    zeroed in PRO_FIR, the residual read from x[2i+1], a neighbouring night's in_stats, stride-2 output rows off by one,
    out_ds taken from odd rows, and group 1 of a pair using group 0's raw signal and block-0 weights."""
    fir = _find("stream", pro=FIR, win=False, wout=False)
    rx = _find("stream", pro=RX, win=False, wout=False)
    if defect == "pair_raw":
        for f in (fir._replace(paired=True), rx._replace(paired=True)):
            worst, _, wrong = _run_pair(f, 3, 3 * _pos(f) + 36, "middle", "none", 7, wrong_side1=True)
            print(f"{_form_id(f)}: right {worst:.3f}, {defect} {wrong:.3g}")
            assert worst <= 1.0 and wrong > 10
        return
    f = {"tap": _find("stream", cin=32, cout=32, stride=1, pro=N, win=False), "inf": fir, "odd_x": rx,
         "stats": _find("stream", cin=64, cout=64, stride=1, pro=N, win=False),
         "rows": _find("stream", cin=32, cout=32, stride=2, pro=N, win=False),
         "odd_ds": _find("stream", cin=16, cout=32, pro=R, win=False)}[defect]
    L = 2 * _pos(f) + 36
    right, _ = _run_single(f, 3, L, "middle", 5)
    wrong, _ = _run_single(f, 3, L, "middle", 5, wrong=defect)
    print(f"{_form_id(f)}: right {right:.3f}, {defect} {wrong:.3g}")
    assert right <= 1.0 and wrong > 10


@pytest.mark.gpu
@pytest.mark.parametrize("f", [_find("stream", cin=32, cout=32, pro=R, win=False), _find("tile", cin=32, cout=32, pro=R),
                               _find("stream", cin=16, cout=32, pro=R, win=True, wout=True)._replace(paired=True)],
                         ids=_form_id)
def test_odd_downsample_length_stays_in_bounds(cuda_device, f):
    """With an odd L_out, out_ds is [B, L_out / 2 rounded down, cout]: row L_out / 2 is not stored, neither into the next
    night's row 0 nor past the end of the tensor (the guard rows after the last night)."""
    for L in (2999, 2998, 1):
        if f.paired:
            worst, _, _ = _run_pair(f, 5, L, "null", "null", 3)
        else:
            worst, _ = _run_single(f, 5, L, "null", 3)
        print(f"{_form_id(f)} L_out={L}: worst error / bound {worst:.3f}")
        assert worst <= 1.0


@pytest.mark.gpu
def test_full_night_statistics(cuda_device):
    """One full ECG night (1,228,800 rows, 16 channels, paired) whose output mean is far above its spread: out_stats within
    the bound, and the relative error the fp32 partial sums put into the next layer's rstd."""
    f = _find("stream", cin=16, cout=16, pro=R, win=False)._replace(paired=True)
    B, L = 1, 1200 * 1024
    sides = []
    for i in range(2):
        s = _side(f, B, L, 50 + i)
        s["r"] = (s["r"].float() * 0.1 + 8.0).half()   # large residual: GELU(a + r) ~ 8, conv output mean >> std
        w = torch.full((16, 16, 3), 0.3, device="cuda") + 0.01 * torch.randn(16, 16, 3, generator=_gen(60 + i), device="cuda")
        s["pw"] = G.pack_conv(w, split=1)
        s["W"] = _unpack(s["pw"], 16, 16, 3, True)
        sides.append(s)
    calls = [_call(f, s, B, L, L, None, 70 + i) for i, s in enumerate(sides)]
    for _, o in calls:
        o["stats"].zero_()
        o["before"]["stats"].zero_()
    _launch(f, [calls[0][0], calls[1][0]])
    for i, (s, (_, o)) in enumerate(zip(sides, calls)):
        worst = _check(f"full night side {i}", f, s, o, B, L, L, pair=(i, None, None))
        ref = _reference(f, s, L, L)["out"][0]
        mean_r, rstd_r = _norm_consts(torch.stack([ref.sum(1), (ref * ref).sum(1)], -1), L)
        mean_k, rstd_k = _norm_consts(o["stats"], L)
        rel = ((rstd_k - rstd_r).abs() / rstd_r).max().item()
        print(f"full night side {i}: |mean| / std {(mean_r * rstd_r).abs().min().item():.0f}, worst error / bound "
              f"{worst:.3f}, next layer's rstd relative error {rel:.2e}")
        assert worst <= 1.0


# ----------------------------------------------------------------------------------------------------------------------
# block 0: x_stats + finalize (keep = 0) and first_conv (keep = 1), through the encoder entry points
# ----------------------------------------------------------------------------------------------------------------------
def _encoders(names, dev):
    from wav2sleep_b200 import build_default
    from wav2sleep_b200.engine import PackPlan, _PackedEncoder
    lib = _lib.load()
    model = build_default({n: n for n in names}, 4, seed=3).to(dev).eval()
    plan = PackPlan(lib, dev)
    pes = [_PackedEncoder(lib, model.signal_encoders.encoders[n], dev, plan) for n in names]
    plan.run()
    return model, pes


def _raw_sums_bound(x):
    """S0 = sum x in 4-sample fp32 groups (x0 + x1) + (x2 + x3): 2 roundings, 2^-23 sum |x|; R_k: chains of 4 fp32 FMAs,
    2^-22 sum |x_p x_p+k|; the fp64 sums of the groups add 2^-50 of the same."""
    z = F.pad(x, (0, 2))
    T = x.shape[1]
    prods = [(x * z[:, k:k + T]) for k in range(3)]
    exact = torch.stack([x.sum(1)] + [p.sum(1) for p in prods], -1)
    bound = torch.stack([2.0 ** -23 * x.abs().sum(1)] + [2.0 ** -22 * p.abs().sum(1) for p in prods], -1) * (1 + 2.0 ** -20)
    return exact, bound


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True], ids=["single", "paired"])
def test_block0_statistics(cuda_device, paired):
    """Inference (keep = 0): S0, R0, R1, R2 and block-0 conv1 statistics (x_stats_kernel / x_stats_finalize_kernel,
    closed form with the first and last sample corrected) against fp64 sums with -inf read as 0; row_mask set exactly
    for nights whose first sample is -inf.  Training (keep = 1): first_conv's y1, residual branch and statistics.  Each
    x_stats thread takes an odd number (3) of 4-sample groups; live nights have -inf at samples 1, 2 and T - 1."""
    lib = _lib.load()
    dev = cuda_device
    names = ["ECG", "PPG"] if paired else ["ECG"]
    model, pes = _encoders(names, dev)
    B = 3
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cap = (4 * sms + len(names) * B - 1) // (len(names) * B)
    T = 4 * 256 * cap * 3                        # 3 groups per thread; a multiple of 1024 samples (one ECG epoch)
    g = _gen(11)
    xs = []
    for i in range(len(names)):
        x = torch.randn(B, T, generator=g, device=dev) * (1 + i) + 0.5
        x[:, [1, 2, T - 1, T // 2]] = float("-inf")
        x[i + 1 if i + 1 < B else 0, 0] = float("-inf")  # a night without this signal
        xs.append(x)
    n_blocks = len(model.signal_encoders.encoders[names[0]].channels)
    for keep in (0, 1):
        ws_bytes = lib.w2s_encoder_workspace_bytes(C.byref(pes[0].desc), B, T, keep)
        wss = [torch.zeros(ws_bytes, dtype=torch.uint8, device=dev) for _ in names]
        zs = [torch.zeros(B, T // 1024, 128, dtype=F16, device=dev) for _ in names]
        ms = [torch.full((B,), 7, dtype=torch.uint8, device=dev) for _ in names]
        if paired:
            _lib.check(lib.w2s_encoder_fwd_pair(C.byref(pes[0].desc), xs[0].data_ptr(), wss[0].data_ptr(), zs[0].data_ptr(),
                                                ms[0].data_ptr(), C.byref(pes[1].desc), xs[1].data_ptr(), wss[1].data_ptr(),
                                                zs[1].data_ptr(), ms[1].data_ptr(), B, T, ws_bytes, keep, G.stream()))
        else:
            _lib.check(lib.w2s_encoder_fwd(C.byref(pes[0].desc), xs[0].data_ptr(), B, T, wss[0].data_ptr(), ws_bytes, keep,
                                           zs[0].data_ptr(), ms[0].data_ptr(), G.stream()))
        torch.cuda.synchronize()
        offs = (C.c_int64 * (7 * n_blocks))()
        _lib.check(lib.w2s_encoder_layout(C.byref(pes[0].desc), B, T, offs))
        chans = list(model.signal_encoders.encoders[names[0]].channels)
        n_layer = sum(3 * B * c * 2 for c in chans)
        for i, n in enumerate(names):
            x, ws = xs[i], wss[i]
            dead = torch.isinf(x[:, 0])
            assert ms[i].tolist() == dead.to(torch.uint8).tolist()
            live = (~dead).nonzero().flatten().tolist()
            enc = model.signal_encoders.encoders[n]
            w = enc.cnn[0].conv1.conv.weight[:, 0, :].double()
            xz = torch.where(torch.isinf(x), torch.zeros_like(x), x).double()[live]
            xp = F.pad(xz, (1, 1))
            cols = torch.stack([xp[:, t:t + T] for t in range(3)], -1)
            h = cols @ w.t()                                              # conv1 of block 0 in fp64
            stats1 = ws[:B * 16 * 2 * 8].view(F64).view(B, 16, 2)[live]
            exact1 = torch.stack([h.sum(1), (h * h).sum(1)], -1)
            if keep == 0:
                raw = ws[n_layer * 8:(n_layer + 4 * B) * 8].view(F64).view(B, 4)[live]
                exact, bound = _raw_sums_bound(xz)
                r_raw = ((raw - exact).abs() / bound).max().item()
                # stats1 = linear / quadratic forms of S0, R0, R1, R2 in the taps (edge terms exact in fp64)
                wa = w.abs()
                b1 = torch.stack([wa.sum(1)[None] * bound[:, :1],
                                  (wa.sum(1) ** 2)[None] * bound[:, 1:].max(1, keepdim=True).values], -1)
                b1 = b1 + 2.0 ** -48 * torch.stack([cols.abs() @ wa.t(), (cols.abs() @ wa.t()) ** 2], -1).sum(1)
                r_s1 = ((stats1 - exact1).abs() / b1).max().item()
                print(f"x_stats {n} {'x2' if paired else ''}: S0/R0/R1/R2 worst error / bound {r_raw:.3f}, "
                      f"stats1 {r_s1:.3f}")
                assert r_raw <= 1.0 and r_s1 <= 1.0
                assert not ws[:B * 16 * 2 * 8].view(F64).view(B, 16, 2)[dead].any()  # masked nights: no statistics
            else:
                # first_conv: y1 = fmaf chain of 3 taps (2^-23 sum |w x|), stored fp16; r0 = w_ds x[2i] (2^-24), fp16
                y1 = ws[offs[3]: offs[3] + B * T * 16 * 2].view(F16).view(B, T, 16)[live].double()
                e1 = 2.0 ** -22 * (cols.abs() @ w.abs().t())
                ry1 = ((y1 - h).abs() / (e1 * (1 + 2.0 ** -11) + 2.0 ** -11 * h.abs() + 2.0 ** -25)).max().item()
                wd = enc.cnn[0].downsample.weight[:, 0, 0].double()
                r0 = ws[offs[4]: offs[4] + B * (T // 2) * 16 * 2].view(F16).view(B, T // 2, 16)[live].double()
                rr = xz[:, 0::2, None] * wd
                rr0 = ((r0 - rr).abs() / (2.0 ** -23 * rr.abs() * (1 + 2.0 ** -11) + 2.0 ** -11 * rr.abs() + 2.0 ** -25)).max().item()
                # statistics: fp32 per-thread sums of 4 rows, 5 butterfly levels, 8 warps: n = 4 + 5 + 8
                n_add = 17
                sb = torch.stack([(e1.sum(1) + n_add * 2.0 ** -24 * h.abs().sum(1)),
                                  ((2 * h.abs() * e1 + e1 * e1).sum(1) + n_add * 2.0 ** -23 * (h * h).sum(1))], -1)
                rs = ((stats1 - exact1).abs() / sb).max().item()
                print(f"first_conv {n}: y1 {ry1:.3f}, r0 {rr0:.3f}, stats1 {rs:.3f} (worst error / bound)")
                assert ry1 <= 1.0 and rr0 <= 1.0 and rs <= 1.0


# ----------------------------------------------------------------------------------------------------------------------
# replay: every forward launch of real models is a tested form
# ----------------------------------------------------------------------------------------------------------------------
def _labels(fn):
    lib = _lib.load()
    torch.cuda.synchronize()
    lib.w2s_profile_enable(1)
    try:
        fn()
        torch.cuda.synchronize()
        buf, ms = C.create_string_buffer(128), C.c_float()
        out = []
        for i in range(lib.w2s_profile_count()):
            _lib.check(lib.w2s_profile_get(i, buf, 128, C.byref(ms), None, None))
            out.append(buf.value.decode())
        return out
    finally:
        lib.w2s_profile_enable(0)


@pytest.mark.gpu
def test_forward_launches_are_tested_forms(cuda_device):
    """Default cardio (paired), cardio with PPG missing on every night, ECG only, the 10-block EOG model
    (wide_blocks = 6), the corner models of test_fast_path_envelope_gpu.py, predict_async and one training forward:
    every encoder forward launch must be a row of FORMS.  The training-only EPI_PLAIN / EPI_ACT_BWD launches are
    test_train_kernels_gpu.py's."""
    from conftest import SPE
    from test_fast_path_envelope_gpu import EDGE, build_model
    from wav2sleep_b200 import build_default
    dev = cuda_device
    cardio = {"ABD": "ABD", "THX": "THX", "ECG": "ECG", "PPG": "PPG"}

    def inputs(smap, B=2, S=3, seed=0):
        g = torch.Generator().manual_seed(seed)
        return {k: torch.randn(B, S * SPE[k], generator=g).to(dev) for k in smap}

    runs = []
    m = build_default(cardio, 4, seed=0).to(dev).eval()
    x = inputs(cardio)
    runs.append(("cardio", lambda: m(x)))
    x_noppg = dict(x)
    x_noppg["PPG"] = torch.full_like(x["PPG"], float("-inf"))
    runs.append(("cardio without PPG", lambda: m(x_noppg)))
    runs.append(("predict_async", lambda: m.predict_async(x)))
    ecg = build_default({"ECG": "ECG"}, 4, seed=1).to(dev).eval()
    runs.append(("ECG only", lambda: ecg(inputs({"ECG": "ECG"}))))
    eog = build_default({"EOG-L": "EOG-L", "EOG-R": "EOG-R"}, 4, seed=2).to(dev).eval()
    assert eog.signal_encoders.encoders["EOG-L"].wide_blocks == 6
    runs.append(("EOG", lambda: eog(inputs({"EOG-L": "EOG-L", "EOG-R": "EOG-R"}))))
    edge_models = []
    for name, (smap, ncls, ml, sb, sd, _) in EDGE.items():
        em = build_model(smap, ncls, ml, sb, sd).to(dev).eval()
        edge_models.append(em)
        runs.append((name, lambda em=em, smap=smap: em(inputs(smap))))
    tm = build_default(cardio, 4, seed=4).to(dev).train()
    runs.append(("training forward", lambda: tm(x)))
    for model in [m, ecg, eog, tm] + edge_models:
        model._get_engine().use_graph = False  # graph replays launch nothing the profiler sees
    # the tile kernels share their keys with fp16 stream rows but are not launched by a forward: only the forms a
    # forward can launch count, so removing any of them from FORMS fails here
    tested = {_launch_key(f) for f in FORMS if f.kind != "tile"}
    seen = set()
    for name, fn in runs:
        with torch.inference_mode(mode=name != "training forward"):
            labels = _labels(fn)
        for lab in labels:
            if lab.startswith("x_stats"):
                seen.add(lab)
                continue
            if not (lab.startswith("conv ") or lab.startswith("first_conv")):
                continue
            key = _label_key(lab)
            if key[0] != "first_conv" and key[5] not in (EPI_STATS, EPI_BIAS_GELU):
                continue  # training-only EPI_PLAIN / EPI_ACT_BWD
            assert key in tested, f"{name}: launch '{lab}' is not a tested form"
            seen.add(key)
    assert {"x_stats", "x_stats x2", ("first_conv",)} <= seen
    print(f"replay: {len(seen)} distinct encoder forward launch forms, all in FORMS")
