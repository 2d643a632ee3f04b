"""Every CUDA entry point that takes a Wav2Sleep input {signal: [B, T]} rejects the same bad inputs with the same
exception types (wav2sleep_b200.engine.check_inputs), and before it launches any kernel."""
import pytest
import torch

from wav2sleep_b200 import StreamingSession, _lib, build_default, integrated_gradients
from wav2sleep_b200 import model as M
from wav2sleep_b200.engine import NotASignalDict, UnknownSignal

SMAP = {"ECG": "ECG", "THX": "THX"}


def _pair(dev, ecg, thx, dev_thx=None):
    """ECG [B, T] and THX [B, T] zeros; shapes as (B, epochs)."""
    return {"ECG": torch.zeros(ecg[0], ecg[1] * 1024, device=dev),
            "THX": torch.zeros(thx[0], thx[1] * 256, device=dev_thx or dev)}


def _second_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    return torch.device("cuda:1")


# name -> (input builder, expected exception, rejected by the stand-alone SignalEncoders call as well)
CASES = {
    "not_a_dict": (lambda d: torch.zeros(2, 1024, device=d), NotASignalDict, True),
    "empty_dict": (lambda d: {}, NotASignalDict, False),
    "unknown_signal": (lambda d: {"ECG": torch.zeros(2, 1024, device=d), "PPG": torch.zeros(2, 1024, device=d)},
                       UnknownSignal, True),
    "not_a_tensor": (lambda d: {"ECG": [0.0] * 1024}, ValueError, True),
    "not_2d": (lambda d: {"ECG": torch.zeros(2, 1, 1024, device=d)}, ValueError, True),
    "cpu_tensor": (lambda d: {"ECG": torch.zeros(2, 1024)}, RuntimeError, True),
    "length_not_a_multiple": (lambda d: {"ECG": torch.zeros(2, 1000, device=d)}, ValueError, True),
    "empty_batch": (lambda d: _pair(d, (0, 1), (0, 1)), ValueError, True),
    "no_epochs": (lambda d: _pair(d, (2, 0), (2, 0)), ValueError, True),
    "batch_mismatch": (lambda d: _pair(d, (2, 1), (1, 1)), ValueError, False),
    "epoch_mismatch": (lambda d: _pair(d, (2, 2), (2, 1)), ValueError, False),
    "mixed_devices": (lambda d: _pair(d, (2, 1), (2, 1), _second_gpu()), ValueError, False),
}


@pytest.fixture(scope="module")
def models(cuda_device):
    fast = build_default(SMAP, 4, seed=0).to(cuda_device)
    # a causal general-path model without BatchNorm: it infers, trains and streams
    enc = M.SignalEncoders(signal_map=SMAP, feature_dim=16, activation="relu", norm="layer", causal=True)
    general = M.Wav2Sleep(enc, M.MultiModalAttentionEmbedder(feature_dim=16),
                          M.SequenceCNN(feature_dim=16, norm="layer", causal=True), 4).to(cuda_device)
    assert fast.fast_path and not general.fast_path
    return fast, general, StreamingSession(general.eval(), 2)


def _requiring_grad(x):
    if isinstance(x, dict):
        return {k: v.clone().requires_grad_() if isinstance(v, torch.Tensor) else v for k, v in x.items()}
    return x


def _entry_points(fast, general, sess):
    def mode(m, train, fn):
        m.train(train)
        return fn()

    return {
        "fast forward": lambda x: mode(fast, False, lambda: fast(x)),
        "fast predict": lambda x: mode(fast, False, lambda: fast.predict(x)),
        "fast predict_async": lambda x: mode(fast, False, lambda: fast.predict_async(x)),
        "fast training forward": lambda x: mode(fast, True, lambda: fast(x)),
        "general eval": lambda x: mode(general, False, lambda: general(x)),
        "general train": lambda x: mode(general, True, lambda: general(x)),
        "general input grad": lambda x: mode(general, False, lambda: general(_requiring_grad(x))),
        "SignalEncoders.forward": lambda x: general.signal_encoders(x),
        "StreamingSession.step": lambda x: sess.step(x),
        "integrated_gradients": lambda x: integrated_gradients(general, x, 0),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_bad_input_raises_before_any_launch(models, cuda_device, case):
    fast, general, sess = models
    build, exc, per_signal = CASES[case]
    lib = _lib.load()
    for name, call in _entry_points(fast, general, sess).items():
        if name == "SignalEncoders.forward" and not per_signal:
            continue  # encodes each signal on its own: B, S and the device may differ between signals
        n0 = lib.w2s_launch_count()
        try:
            call(build(cuda_device))
        except exc:
            pass
        except Exception as e:
            raise AssertionError(f"{name}: {case} raised {type(e).__name__}, expected {exc.__name__}") from e
        else:
            pytest.fail(f"{name}: {case} was accepted")
        assert lib.w2s_launch_count() == n0, f"{name}: launched before rejecting {case}"
    assert sess.pos == 0
