"""Timing of epoch-by-epoch streaming (wav2sleep_b200/streaming.py) against re-running the whole prefix.

Two causal models, N in {1, 64, 1024} streams, R = 1 new epoch per call:
  * causality: the configuration of the reference's tests/model/test_causality.py (ECG + PPG, chunk-causal encoders,
    BatchNorm, ReLU, feature_dim 16);
  * f128: ECG + PPG chunk-causal encoders with layer norm and GELU, feature_dim 128, the reference's default mixer
    (MultiModalAttentionEmbedder(feature_dim=128)) and SequenceCNN(feature_dim=128, causal=True, norm="layer").
For each: wall time per ``step`` (CUDA events around warmed-up calls, host launch time included, as a caller sees it),
split into encoders / epoch mixer / sequence step (events between the stages of the same calls), the device time of the
``w2s_gen_seq_stream_step`` kernel alone (the library's per-launch event profile), and one full forward
over a 1200-epoch prefix for the same N - what a caller without a session runs to get the newest epoch.  N = 1024
nights do not fit one general-path forward (at most 65535 epoch rows), so N > 32 runs as consecutive forwards of 32
nights, timed together.

    python tools/time_streaming.py [--iters 50]
"""
import argparse
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from wav2sleep_b200 import StreamingSession, _lib  # noqa: E402
from wav2sleep_b200 import model as M  # noqa: E402

SIGNALS = {"ECG": "ECG", "PPG": "PPG"}
SPE = 1024
PREFIX = 1200
PREFIX_BATCH = 32  # nights per prefix forward: the general encoder kernels take at most 65535 epoch rows


def build(name):
    torch.manual_seed(0)
    if name == "causality":
        enc = M.SignalEncoders(signal_map=SIGNALS, feature_dim=16, activation="relu", norm="batch", causal=True)
        return M.Wav2Sleep(enc, M.MultiModalAttentionEmbedder(feature_dim=16),
                           M.SequenceCNN(feature_dim=16, causal=True, norm="batch"), 4)
    enc = M.SignalEncoders(signal_map=SIGNALS, feature_dim=128, activation="gelu", norm="layer", causal=True)
    return M.Wav2Sleep(enc, M.MultiModalAttentionEmbedder(feature_dim=128),
                       M.SequenceCNN(feature_dim=128, causal=True, norm="layer"), 4)


def time_steps(sess, x, iters):
    """(encoders, mixer, sequence) ms per step: the body of StreamingSession.step with events between its stages."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    acc = [0.0, 0.0, 0.0]
    for _ in range(iters):
        with torch.no_grad():
            ev[0].record()
            zs, masks = [], []
            for name in sorted(x):
                z, mask = sess.encode(name, x[name])
                zs.append(z)
                masks.append(mask)
            ev[1].record()
            feat = sess.eng.epoch_mixer(zs, masks, sess.n_streams, 1)
            ev[2].record()
            sess.sequence_step(feat)
            ev[3].record()
        ev[3].synchronize()
        for i in range(3):
            acc[i] += ev[i].elapsed_time(ev[i + 1])
    return [acc[0] / iters, acc[1] / iters, acc[2] / iters]


def time_seq_kernel(sess, x, iters):
    """Mean device time of one w2s_gen_seq_stream_step launch (ms), from the library's per-launch events."""
    with torch.no_grad():
        enc = [sess.encode(n, x[n]) for n in sorted(x)]
        feat = sess.eng.epoch_mixer([z for z, _ in enc], [m for _, m in enc], sess.n_streams, 1)
    lib = _lib.load()
    torch.cuda.synchronize()
    lib.w2s_profile_enable(1)
    for _ in range(iters):
        sess.sequence_step(feat)
    torch.cuda.synchronize()
    recs = [t for label, t, _, _ in bench.collect_profile(lib) if label == "gen_seq_stream_step"]
    lib.w2s_profile_enable(0)
    return sum(recs) / len(recs)


def time_step_calls(sess, x, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        sess.step(x)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def time_prefix(model, N, dev):
    g = torch.Generator(device=dev).manual_seed(1)
    nb = min(N, PREFIX_BATCH)
    x = {k: torch.randn(nb, PREFIX * SPE, generator=g, device=dev) for k in SIGNALS}
    with torch.no_grad():
        model(x)  # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(N // nb):
            model(x)
        e1.record()
        torch.cuda.synchronize()
    del x
    torch.cuda.empty_cache()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--streams", type=int, nargs="+", default=[1, 64, 1024])
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    print(f"device: {torch.cuda.get_device_name(dev)}; nvidia-smi: {smi.stdout.strip() or smi.stderr.strip()}", flush=True)
    print("model      N    step ms  (encoders  mixer  sequence)  seq kernel ms  per stream-epoch us   prefix-1200 forward ms  "
          "ratio")
    for name in ("causality", "f128"):
        model = build(name).to(dev).eval()
        for N in args.streams:
            sess = StreamingSession(model, N)
            g = torch.Generator(device=dev).manual_seed(N)
            x = {k: torch.randn(N, SPE, generator=g, device=dev) for k in SIGNALS}
            for _ in range(10):
                sess.step(x)
            torch.cuda.synchronize()
            step_ms = time_step_calls(sess, x, args.iters)
            enc_ms, mix_ms, seq_ms = time_steps(sess, x, args.iters)
            kern_ms = time_seq_kernel(sess, x, args.iters)
            prefix_ms = time_prefix(model, N, dev)
            print(f"{name:9s} {N:5d} {step_ms:9.3f}  ({enc_ms:8.3f} {mix_ms:6.3f} {seq_ms:9.3f})  {kern_ms:13.3f}  "
                  f"{1e3 * step_ms / N:18.2f}"
                  f"   {prefix_ms:22.1f}  {prefix_ms / step_ms:6.0f}x", flush=True)
            del sess
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
