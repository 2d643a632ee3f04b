"""Epoch-by-epoch inference of causal models (wav2sleep_b200/streaming.py, csrc/stream.cuh).

Chain of evidence: the full-night forward of the general CUDA path matches the real reference's golden logits
(tests/test_general.py); a StreamingSession fed the same nights in chunks must give the same logits as that forward (and
as the golden files), with any chunking, any number of streams and any reset pattern.  The sequence-mixer step kernel
is also checked on its own against an fp64 CPU restatement of the causal SequenceCNN (oracle/general_oracle.py).
"""
import ctypes
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from oracle import general_oracle as O
from oracle import make_golden_general as G
from wav2sleep_b200 import StreamingSession, _lib, build_default
from wav2sleep_b200 import model as M

CAUSAL_CASES = ["general_causal_batch_relu", "general_causalconv_layer_silu"]


def _model(enc=None, seq=None, smap=None, F=16):
    enc = {**dict(feature_dim=F, activation="relu", norm="batch", causal=True), **(enc or {})}
    seq = {**dict(feature_dim=F, causal=True, norm="batch"), **(seq or {})}
    encoders = M.SignalEncoders(signal_map=smap or {"ECG": "ECG"}, **enc)
    return M.Wav2Sleep(encoders, M.MultiModalAttentionEmbedder(feature_dim=F), M.SequenceCNN(**seq), 4)


def _golden_model(name, dev):
    case = G.CASES[name]
    model = G.build(M, case)
    G.perturb(model, case["seed"])
    return case, model.to(dev).eval()


def _spe(model, name):
    return model.signal_encoders.get_encoder(name).samples_per_epoch


def _stream(sess, model, x, chunks, dev):
    """Feed x {signal: [N, S * spe]} through sess in calls of `chunks` epochs; stacked logits [N, S, C]."""
    out, e = [], 0
    for r in chunks:
        out.append(sess.step({k: v[:, e * _spe(model, k):(e + r) * _spe(model, k)].to(dev) for k, v in x.items()}))
        e += r
    return torch.cat(out, dim=1)


# ---------------------------------------------------------------------------------------------------------- CPU
def test_only_causal_models_stream():
    with pytest.raises(ValueError, match="signal_encoders"):
        StreamingSession(build_default({"ECG": "ECG"}, 4, seed=0), 1)
    with pytest.raises(ValueError, match="signal_encoders"):
        StreamingSession(_model(enc=dict(causal=False), seq=dict()), 1)
    for norm in ("instance", "auto"):
        with pytest.raises(ValueError, match=r"encoders\['ECG'\].*norm 'instance'"):
            StreamingSession(_model(enc=dict(chunk_causal=False, norm=norm)), 1)
    with pytest.raises(ValueError, match="sequence_mixer.*'group'"):
        StreamingSession(_model(seq=dict(norm="group")), 1)
    with pytest.raises(ValueError, match="sequence_mixer is not causal"):
        StreamingSession(_model(seq=dict(causal=False)), 1)
    with pytest.raises(ValueError, match="feature_dim"):
        StreamingSession(_model(F=264), 1)
    from wav2sleep_b200.ppgnet import SleepPPGNet
    with pytest.raises(ValueError, match="SleepPPGNet"):
        StreamingSession(SleepPPGNet(n_classes=4, feature_dim=16), 1)
    # chunk-causal encoders stream with any norm; causal convolutions with a per-position one
    for enc in (dict(norm="instance"), dict(norm="group"), dict(chunk_causal=False, norm="layer"),
                dict(chunk_causal=False, norm="batch")):
        with pytest.raises(RuntimeError, match="CUDA"):  # eligible, but on the CPU: no fallback
            StreamingSession(_model(enc=enc, seq=dict(norm="rms")), 2)
    with pytest.raises(ValueError):
        StreamingSession(_model(), 0)


def test_stream_descriptor_sizes_match_header():
    src = ('#include <stdio.h>\n#include "w2s_b200.h"\nint main(){printf("%zu %zu\\n", sizeof(w2s_gen_seq_stream_layer), '
           'sizeof(w2s_gen_seq_stream_desc));return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "p.c").write_text(src)
        subprocess.run(["gcc", "-I", str(ROOT / "include"), "-o", f"{d}/p", f"{d}/p.c"], check=True)
        out = subprocess.run([f"{d}/p"], capture_output=True, text=True, check=True).stdout.split()
    assert [ctypes.sizeof(_lib.SeqStreamLayer), ctypes.sizeof(_lib.SeqStreamDesc)] == [int(v) for v in out]


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", CAUSAL_CASES)
def test_streaming_matches_golden_and_full_forward(cuda_device, name):
    case, model = _golden_model(name, cuda_device)
    x = G.make_inputs(case)
    with torch.no_grad():
        full = model({k: v.to(cuda_device) for k, v in x.items()}).cpu()
    sess = StreamingSession(model, case["B"])
    got = _stream(sess, model, x, [1] * case["S"], cuda_device).cpu()
    gold = torch.from_numpy(np.load(GOLDEN / f"{name}.npz")["logits"])
    e_gold, e_full = (got - gold).abs().max().item(), (got - full).abs().max().item()
    print(f"{name}: streamed logits vs golden {e_gold:.2e}, vs the CUDA full forward {e_full:.2e}")
    assert got.shape == gold.shape and e_gold <= 2e-4 and e_full <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("name", CAUSAL_CASES)
def test_chunking_is_bitwise_invariant(cuda_device, name):
    case, model = _golden_model(name, cuda_device)
    x, S = G.make_inputs(case), case["S"]
    mixed = [2, 3, 1, 2, 3, 1]
    while sum(mixed) > S:
        mixed[-1] -= sum(mixed) - S
        mixed = [r for r in mixed if r > 0]
    runs = []
    for chunks in ([S], [1] * S, mixed):
        runs.append(_stream(StreamingSession(model, case["B"]), model, x, chunks, cuda_device))
    model.train()  # sessions have eval semantics whatever the module mode says
    runs.append(_stream(StreamingSession(model, case["B"]), model, x, mixed, cuda_device))
    assert all(torch.equal(runs[0], r) for r in runs[1:])
    preds = StreamingSession(model, case["B"]).predict_step({k: v.to(cuda_device) for k, v in x.items()})
    assert preds.dtype == torch.int64 and torch.equal(preds, runs[0].argmax(-1))


def _causality_test_model(dev):
    """The configuration of the reference's tests/model/test_causality.py (chunk-causal, BatchNorm, ReLU, F = 16)."""
    torch.manual_seed(0)
    encoders = M.SignalEncoders(signal_map={"ECG": "ECG", "PPG": "PPG"}, feature_dim=16, activation="relu", norm="batch",
                                causal=True)
    model = M.Wav2Sleep(signal_encoders=encoders, epoch_mixer=M.MultiModalAttentionEmbedder(feature_dim=16),
                        sequence_mixer=M.SequenceCNN(feature_dim=16, causal=True, norm="batch"), num_classes=4)
    return model.to(dev).eval()


@pytest.mark.gpu
def test_full_night_one_epoch_per_call(cuda_device):
    model = _causality_test_model(cuda_device)
    g = torch.Generator().manual_seed(5)
    x = {"ECG": torch.randn(2, 1200 * 1024, generator=g), "PPG": torch.randn(2, 1200 * 1024, generator=g)}
    x["PPG"][1] = float("-inf")  # PPG missing for the whole night of stream 1
    with torch.no_grad():
        full = model({k: v.to(cuda_device) for k, v in x.items()})
    got = _stream(StreamingSession(model, 2), model, x, [1] * 1200, cuda_device)
    err = (got - full).abs().max().item()
    print(f"causality-test model, 1200 epochs one per call: max-abs {err:.2e} vs the full forward")
    assert got.shape == (2, 1200, 4) and err <= 1e-4


@pytest.mark.gpu
def test_full_night_carried_conv_context(cuda_device):
    case, model = _golden_model("general_causalconv_layer_silu", cuda_device)
    x = G.make_inputs({**case, "B": 2, "S": 1200})
    with torch.no_grad():
        full = model({k: v.to(cuda_device) for k, v in x.items()})
    got = _stream(StreamingSession(model, 2), model, x, [50] * 24, cuda_device)
    err = (got - full).abs().max().item()
    print(f"causal-conv encoders, 1200 epochs in chunks of 50 (1.2 M ECG samples of context): max-abs {err:.2e}")
    assert err <= 1e-4


@pytest.mark.gpu
def test_streams_and_staggered_resets_equal_single_stream_sessions(cuda_device):
    case, model = _golden_model("general_causalconv_layer_silu", cuda_device)
    T, resets = 8, {1: 3, 2: 5}  # stream -> call before which it is reset
    nights = [G.make_inputs({**case, "B": 1, "S": T}, seed=s) for s in range(5)]
    # stream 0: night 0 throughout; stream 1: night 1 then night 3; stream 2: night 2 then night 4
    after = {1: 3, 2: 4}
    sess, out = StreamingSession(model, 3), []
    for t in range(T):
        reset_now = [s for s, at in resets.items() if at == t]
        if reset_now:
            sess.reset(reset_now)
        xs = {}
        for k in nights[0]:
            spe = _spe(model, k)
            rows = []
            for s in range(3):
                night, e = (nights[after[s]], t - resets[s]) if s in resets and t >= resets[s] else (nights[s], t)
                rows.append(night[k][:, e * spe:(e + 1) * spe])
            xs[k] = torch.cat(rows).to(cuda_device)
        out.append(sess.step(xs))
    got = torch.cat(out, dim=1)

    def single(night, n):
        return _stream(StreamingSession(model, 1), model, night, [1] * n, cuda_device)[0]

    assert torch.equal(got[0], single(nights[0], T))
    for s, at in resets.items():
        assert torch.equal(got[s, :at], single(nights[s], at))
        assert torch.equal(got[s, at:], single(nights[after[s]], T - at))


# kernel cases: (F, norm, activation, kernel_size, num_dilations, num_layers); dilations up to 32 with T = 200 > 192
KERNEL_CASES = [
    (16, "batch", "relu", 3, 6, 2),
    (40, "layer", "gelu", 7, 6, 1),
    (128, "rms", "silu", 7, 6, 2),
    (256, None, "leaky", 3, 6, 1),
    (128, "layer", "gelu", 7, 6, 2),
    (40, "batch", "gelu", 7, 3, 3),
]


def _seq_oracle(h_NTF, sd, F, norm, act, k, n_dil, n_layers):
    """Causal SequenceCNN + classifier of oracle/general_oracle.py on [n, T, F] features (fp64 parameters)."""
    h = h_NTF.transpose(1, 2)
    for bi in range(n_layers):
        out = h
        for j in range(n_dil):
            dil = 2 ** j
            out = O.conv_layer(out, sd, f"sequence_mixer.dilated_convs.{bi}.conv_layers.{j}", k, 1, dil,
                               (k + (k - 1) * (dil - 1)) // 2, True, norm, act)
        h = O.act(out + h, act)
    return h.transpose(1, 2) @ sd["classifier.weight"].t() + sd["classifier.bias"]


def _kernel_model(dev, F, norm, act, k, n_dil, n_layers):
    torch.manual_seed(F + k)
    model = _model(seq=dict(norm=norm, activation=act, kernel_size=k, num_dilations=n_dil, num_layers=n_layers), F=F)
    model.classifier = torch.nn.Linear(F, 5)
    model.num_classes = 5
    G.perturb(model, F)
    return model.to(dev).eval()


CHUNKS = [1, 7, 32, 3, 64, 50, 43]  # T = 200 epochs in uneven calls
T_KERNEL = sum(CHUNKS)


def _run_sequence_steps(sess, feat, reset_at, dev):
    """sess.sequence_step over feat [N, T, F] in CHUNKS, resetting reset_at[call] (stream indices) before a call ->
    (logits [N, T, C], the epoch each stream last started at).  Asserts one launch per call."""
    lib = _lib.load()
    out, e, starts = [], 0, [0] * feat.shape[0]
    for i, r in enumerate(CHUNKS):
        if reset_at.get(i):
            for s in reset_at[i]:
                starts[s] = e
            sess.reset(reset_at[i])
        n0 = lib.w2s_launch_count()
        out.append(sess.sequence_step(feat[:, e:e + r].to(dev)).cpu())
        assert lib.w2s_launch_count() - n0 == 1
        e += r
    return torch.cat(out, dim=1), starts


def _oracle_rel_err(model, got, feat, starts, rows, cfg):
    """Relative L2 error of got[rows] against the fp64 oracle over each stream's segments since its resets."""
    sd = {kk: v.detach().cpu().double() for kk, v in model.state_dict().items()}
    got, want = got[rows].double(), torch.empty(len(rows), *got.shape[1:], dtype=torch.float64)
    st = [starts[s] for s in rows]
    for start in sorted(set(st)):  # streams restarted at the same epoch share one oracle run per segment
        sel = [i for i, v in enumerate(st) if v == start]
        src = [rows[i] for i in sel]
        for a, b in ((0, start), (start, feat.shape[1])) if start else ((0, feat.shape[1]),):
            if b > a:
                want[sel, a:b] = _seq_oracle(feat[src, a:b].double(), sd, *cfg)
    return ((got - want).norm() / want.norm()).item()


@pytest.mark.gpu
@pytest.mark.parametrize("F,norm,act,k,n_dil,n_layers", KERNEL_CASES)
def test_sequence_step_kernel_matches_oracle(cuda_device, F, norm, act, k, n_dil, n_layers):
    model = _kernel_model(cuda_device, F, norm, act, k, n_dil, n_layers)
    N = 37  # not a multiple of any stream tile
    feat = torch.randn(N, T_KERNEL, F, generator=torch.Generator().manual_seed(k))
    got, starts = _run_sequence_steps(StreamingSession(model, N), feat, {3: [4, 17, 36], 5: [0, 20]}, cuda_device)
    rel = _oracle_rel_err(model, got, feat, starts, list(range(N)), (F, norm, act, k, n_dil, n_layers))
    print(f"F={F} norm={norm} act={act} k={k} dilations={n_dil} blocks={n_layers}: relative L2 {rel:.2e}")
    assert rel <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("F,norm,act,k,n_dil,n_layers", [KERNEL_CASES[0], KERNEL_CASES[4], KERNEL_CASES[3]])
def test_sequence_step_multi_stream_tiles(cuda_device, F, norm, act, k, n_dil, n_layers):
    """Enough streams that every thread carries several (the launch takes ceil(N / (G * SMs)) streams per thread,
    G = 256 / F thread groups) and the last tile is partial.  Logits must be bitwise those of sessions small enough
    for one stream per thread, and match the oracle on the first streams and the partial last tile."""
    sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    Gt = 256 // F
    N = 2 * Gt * sms + 1  # 3 streams per thread
    while N % (3 * Gt) == 0:
        N += 1
    model = _kernel_model(cuda_device, F, norm, act, k, n_dil, n_layers)
    feat = torch.randn(N, T_KERNEL, F, generator=torch.Generator().manual_seed(F))
    resets = {3: [1, N // 2, N - 1], 5: [0, N - 2]}
    got, starts = _run_sequence_steps(StreamingSession(model, N), feat, resets, cuda_device)
    step = Gt * sms  # one stream per thread
    for a in range(0, N, step):
        b = min(a + step, N)
        part = {i: [s - a for s in v if a <= s < b] for i, v in resets.items()}
        ref, _ = _run_sequence_steps(StreamingSession(model, b - a), feat[a:b], part, cuda_device)
        assert torch.equal(got[a:b], ref), f"streams {a}..{b - 1} differ from a session of one stream per thread"
    rows = list(range(8)) + list(range(N - 3 * Gt - 2, N))
    rel = _oracle_rel_err(model, got, feat, starts, rows, (F, norm, act, k, n_dil, n_layers))
    print(f"F={F}, N={N} streams (3 per thread, last tile partial): relative L2 {rel:.2e} vs the oracle")
    assert rel <= 1e-5


@pytest.mark.gpu
def test_shared_causal_conv_encoder_with_signal_embeddings(cuda_device):
    """One causal-conv encoder serving ECG and PPG (separate contexts per signal name) plus signal embeddings, streamed
    in uneven chunks with a whole-night missing PPG row, against the full-night forward."""
    torch.manual_seed(11)
    enc = M.SignalEncoders(signal_map={"ECG": "UNI", "PPG": "UNI"}, feature_dim=16, activation="silu", norm="layer",
                           causal=True, chunk_causal=False, embed_signals=True)
    model = M.Wav2Sleep(enc, M.MultiModalAttentionEmbedder(feature_dim=16, layers=2),
                        M.SequenceCNN(feature_dim=16, causal=True, norm="layer", num_dilations=4), 4)
    G.perturb(model, 11)
    model = model.to(cuda_device).eval()
    assert list(model.signal_encoders.encoders) == ["UNI"]
    g = torch.Generator().manual_seed(3)
    S = 12
    x = {k: torch.randn(3, S * 1024, generator=g) for k in ("ECG", "PPG")}
    x["PPG"][2] = float("-inf")
    with torch.no_grad():
        full = model({k: v.to(cuda_device) for k, v in x.items()})
    got = _stream(StreamingSession(model, 3), model, x, [2, 3, 1, 4, 2], cuda_device)
    err = (got - full).abs().max().item()
    print(f"shared causal-conv encoder + signal embeddings: max-abs {err:.2e} vs the full forward")
    assert err <= 1e-4


@pytest.mark.gpu
def test_masked_chunk_equals_absent_key(cuda_device):
    case, model = _golden_model("general_causal_batch_relu", cuda_device)
    x = G.make_inputs(case)
    calls = [{k: v[:, e * _spe(model, k):(e + 1) * _spe(model, k)].to(cuda_device) for k, v in x.items()}
             for e in range(case["S"])]
    a, b = StreamingSession(model, case["B"]), StreamingSession(model, case["B"])
    for e, c in enumerate(calls):
        if e == 2:
            la = a.step({**c, "PPG": torch.full_like(c["PPG"], float("-inf"))})
            lb = b.step({"ECG": c["ECG"]})
        else:
            la, lb = a.step(c), b.step(c)
        assert torch.equal(la, lb)


@pytest.mark.gpu
def test_causal_conv_encoder_restarts_after_a_masked_chunk(cuda_device):
    case, model = _golden_model("general_causalconv_layer_silu", cuda_device)
    S, gap = 8, 3
    x = G.make_inputs({**case, "B": 2, "S": S})["ECG"].to(cuda_device)
    spe = _spe(model, "ECG")
    sess = StreamingSession(model, 2)
    zs = []
    for e in range(S):
        c = x[:, e * spe:(e + 1) * spe].clone()
        if e == gap:
            c[0] = float("-inf")  # stream 0's ECG is missing for this call
        with torch.no_grad():
            z, mask = sess.encode("ECG", c)
        assert mask.tolist() == [int(e == gap), 0]
        zs.append(z)
    z = torch.cat(zs, dim=1)
    enc = model.signal_encoders.get_encoder("ECG")
    with torch.no_grad():
        suffix, _ = sess.eng.encode(enc, x[0:1, (gap + 1) * spe:].contiguous())
        whole, _ = sess.eng.encode(enc, x[1:2])
    torch.testing.assert_close(z[0, gap + 1:], suffix[0], rtol=0, atol=1e-6)
    torch.testing.assert_close(z[1], whole[0], rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_input_errors_raise_before_any_launch(cuda_device):
    case, model = _golden_model("general_causal_batch_relu", cuda_device)
    sess = StreamingSession(model, 2)
    lib = _lib.load()
    ok = torch.zeros(2, 1024, device=cuda_device)
    n0 = lib.w2s_launch_count()
    for bad in ({"EEG": ok}, {"ECG": ok[:, :1000]}, {"ECG": ok, "PPG": torch.zeros(2, 2048, device=cuda_device)},
                {"ECG": ok[:1]}, {}):
        with pytest.raises(ValueError):
            sess.step(bad)
    with pytest.raises(RuntimeError):
        sess.step({"ECG": torch.zeros(2, 1024)})
    assert lib.w2s_launch_count() == n0 and sess.pos == 0


@pytest.mark.gpu
def test_step_that_raises_leaves_the_session_unchanged(cuda_device, monkeypatch):
    case, model = _golden_model("general_causalconv_layer_silu", cuda_device)
    x = G.make_inputs({**case, "S": 4})
    ref = _stream(StreamingSession(model, case["B"]), model, x, [1, 1, 1, 1], cuda_device)
    sess = StreamingSession(model, case["B"])
    first = _stream(sess, model, {k: v[:, :_spe(model, k)] for k, v in x.items()}, [1], cuda_device)

    def fail(feat):
        raise RuntimeError("sequence step failed")

    monkeypatch.setattr(sess, "sequence_step", fail)
    with pytest.raises(RuntimeError, match="sequence step failed"):
        _stream(sess, model, {k: v[:, _spe(model, k):2 * _spe(model, k)] for k, v in x.items()}, [1], cuda_device)
    monkeypatch.undo()
    rest = _stream(sess, model, {k: v[:, _spe(model, k):] for k, v in x.items()}, [1, 1, 1], cuda_device)
    assert torch.equal(torch.cat([first, rest], dim=1), ref)
