"""Forward time of the cardio model when signals are missing on some nights (rows of -inf, data/dataset.py:170-173):
16 synthetic 10-h nights, PPG missing on 12 of them, THX on 8.  Compares the engine's launch policies, set through
its ``enc_pairs`` attribute: 0 (one launch chain per signal) against the default 1 (paired launches, the grid split
in proportion to the live samples of the two encoders)."""
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from wav2sleep_b200 import build_default  # noqa: E402

dev = torch.device("cuda:0")
model = build_default(bench.CARDIO, 4, seed=0).to(dev).eval()
xs = []
for seed in (42, 43):
    x = {k: v.to(dev) for k, v in bench.make_night_batch(16, seed=seed).items()}
    x["PPG"][:12] = float("-inf")
    x["THX"][:8] = float("-inf")
    xs.append(x)
eng = model._get_engine()


def time_forward(enc_pairs):
    eng.enc_pairs = enc_pairs
    with torch.inference_mode():
        for i in range(4):
            model.predict(xs[i % 2])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pend = []
        for i in range(30):
            pend.append(model.predict_async(xs[i % 2]))
            if len(pend) > 1:
                pend.pop(0).wait()
        for q in pend:
            q.wait()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 30


for enc_pairs in (0, 1):
    ms = time_forward(enc_pairs)
    print(f"masked forward (PPG 4/16, THX 8/16 nights live), enc_pairs={enc_pairs}: {ms:.3f} ms/step")
