"""CPU tests of the host-side API: reference artefact loading and the N>1 sharding path (gloo, world_size 2)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import yaml

from wav2sleep_b200 import api, build_default

CARDIO = {"ABD": "ABD", "THX": "THX", "ECG": "ECG", "PPG": "PPG"}


def test_instantiate_reference_targets_matches_build_default():
    torch.manual_seed(0)
    a = api.instantiate(api.default_config(CARDIO, 4))
    b = build_default(CARDIO, 4, seed=0)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb)
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    with pytest.raises(ValueError):
        api.instantiate({"_target_": "os.system", "command": "true"})


def test_load_model_reads_reference_artefacts(tmp_path):
    ref = build_default(CARDIO, 4, seed=3)
    (tmp_path / "config.yaml").write_text(yaml.safe_dump(api.default_config(CARDIO, 4), sort_keys=False))
    torch.save(ref.state_dict(), tmp_path / "state_dict.pth")
    m = api.load_model(str(tmp_path), device="cpu")
    assert not m.training and m.valid_signals == list(CARDIO) and m.num_classes == 4
    assert all(torch.equal(v, ref.state_dict()[k]) for k, v in m.state_dict().items())
    with pytest.raises(FileNotFoundError):
        api.load_model(str(tmp_path / "missing"))


@pytest.mark.parametrize("n,world", [(10, 3), (2, 4), (16, 8), (0, 2)])
def test_shard_range_partitions(n, world):
    parts = [list(api.shard_range(n, r, world)) for r in range(world)]
    assert sum(parts, []) == list(range(n))
    assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


def _worker(rank, world, port, n_items, epochs, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    calls = []

    def fake_predict(indices):  # stands in for model.predict on this rank's GPU
        calls.append(list(indices))
        return torch.tensor([[i * 100 + e for e in range(epochs)] for i in indices], dtype=torch.int64).reshape(-1, epochs)

    out = api.predict_sharded(fake_predict, n_items, epochs)
    q.put((rank, calls, out))
    dist.destroy_process_group()


def test_predict_sharded_gloo_world2():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    n_items, epochs, world = 5, 7, 2
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_items, epochs, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=120) for _ in range(world)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    expect = torch.tensor([[i * 100 + e for e in range(epochs)] for i in range(n_items)])
    assert res[0][1] == [[0, 1, 2]] and res[1][1] == [[3, 4]]  # disjoint contiguous shards
    for _, _, out in res:
        assert torch.equal(out, expect)  # every rank sees all predictions, in recording order


def test_top_level_functions_mirror_the_reference_package():
    """`from wav2sleep import load_model, predict, save_predictions, predict_on_folder` (reference __init__.py:3-19)."""
    import inspect
    import wav2sleep_b200 as pkg
    for name in ("load_model", "predict", "save_predictions", "predict_on_folder"):
        assert callable(getattr(pkg, name)), name
    params = list(inspect.signature(pkg.load_model).parameters)
    assert params == ["folder", "device", "compile", "revision", "cache_dir"]  # api.py:53-59
    import pytest
    with pytest.raises(NotImplementedError):
        pkg.load_model("hf://joncarter/wav2sleep")


def test_hostmem_binding_is_placement_only():
    """hostmem.bind_to_gpu_numa narrows the process's CPU affinity to the GPU-local CPUs and never widens or empties it;
    without NVML / a GPU it is a silent no-op (multi-rank bench.py calls it before allocating pinned batches)."""
    import os
    from wav2sleep_b200 import hostmem
    before = os.sched_getaffinity(0)
    cpus = hostmem.gpu_local_cpus(0)
    assert isinstance(cpus, list) and all(isinstance(c, int) and 0 <= c < (os.cpu_count() or 1) for c in cpus)
    n = hostmem.bind_to_gpu_numa(0)
    after = os.sched_getaffinity(0)
    try:
        assert after <= before and len(after) > 0
        assert n in (0, len(after))
        if not cpus:
            assert n == 0 and after == before
    finally:
        os.sched_setaffinity(0, before)


def test_encoder_pairing_rules():
    """Host logic of the paired encoder launches (engine._enc_groups): signals are paired when their encoders have the
    same architecture and their inputs the same length; the longest chains come first; in the default mode pairs are
    formed only while at least two launch chains remain (the two-signal EOG model keeps one chain per signal)."""
    import types
    import torch
    from wav2sleep_b200 import _lib
    from wav2sleep_b200.engine import ForwardEngine

    def desc(channels, wide=0):
        d = _lib.EncoderDesc()
        d.n_blocks, d.feature_dim, d.norm_eps, d.wide_blocks = len(channels), 128, 1e-2, wide
        for i, c in enumerate(channels):
            d.channels[i] = c
        return d

    hi, lo = [16, 16, 32, 32, 64, 64, 128, 128], [16, 16, 32, 32, 64, 64]

    def stub(smap, descs, mode):
        model = types.SimpleNamespace(signal_encoders=types.SimpleNamespace(signal_map=smap))
        return types.SimpleNamespace(enc_pairs=mode, model=model,
                                     enc={k: types.SimpleNamespace(desc=d) for k, d in descs.items()})

    groups = ForwardEngine._enc_groups
    smap = {n: n for n in ("ABD", "THX", "ECG", "PPG")}
    descs = {"ABD": desc(lo), "THX": desc(lo), "ECG": desc(hi), "PPG": desc(hi)}
    xs = {"ABD": torch.empty(2, 256 * 8), "THX": torch.empty(2, 256 * 8), "ECG": torch.empty(2, 1024 * 8),
          "PPG": torch.empty(2, 1024 * 8)}
    names = sorted(xs)
    assert groups(stub(smap, descs, 1), names, xs, True) == [("ECG", "PPG"), ("ABD", "THX")]
    assert groups(stub(smap, descs, 0), names, xs, True) == [("ECG",), ("PPG",), ("ABD",), ("THX",)]
    assert groups(stub(smap, descs, 1), names, xs, False) == [("ECG",), ("PPG",), ("ABD",), ("THX",)]
    # a different architecture (wide storage) or input length is never paired
    odd = dict(descs, PPG=desc(hi, wide=2))
    assert groups(stub(smap, odd, 1), names, xs, True) == [("ECG",), ("PPG",), ("ABD", "THX")]
    # three signals: one pair + one single = two chains
    three = {k: xs[k] for k in ("ABD", "ECG", "PPG")}
    assert groups(stub(smap, descs, 1), sorted(three), three, True) == [("ECG", "PPG"), ("ABD",)]
    # two signals of one architecture: default keeps two chains, mode 2 pairs
    eog = {"EOG-L": "EOG-L", "EOG-R": "EOG-R"}
    de = {k: desc(hi + [128, 128], wide=6) for k in eog}
    xe = {k: torch.empty(1, 4096 * 4) for k in eog}
    assert groups(stub(eog, de, 1), sorted(xe), xe, True) == [("EOG-L",), ("EOG-R",)]
    assert groups(stub(eog, de, 2), sorted(xe), xe, True) == [("EOG-L", "EOG-R")]
    # two signals sharing ONE encoder (same weights) may be paired too
    shared = {"EOG-L": "EOG", "EOG-R": "EOG"}
    assert groups(stub(shared, {"EOG": de["EOG-L"]}, 2), sorted(xe), xe, True) == [("EOG-L", "EOG-R")]


@pytest.mark.parametrize("mixer_layers,seq_blocks,seq_dilations,ncls,fast", [
    (1, 1, 1, 1, True), (8, 4, 6, 8, True), (2, 2, 6, 4, True), (3, 3, 2, 2, True),
    (2, 2, 7, 4, False), (2, 2, 8, 4, False), (1, 1, 7, 1, False),   # dilation 64 / 128: the per-layer conv cannot stage it
    (9, 2, 6, 4, False), (2, 5, 6, 4, False), (2, 2, 6, 9, False),
])
def test_fast_path_routing_corners(mixer_layers, seq_blocks, seq_dilations, ncls, fast):
    """Wav2Sleep.fast_path at the corners of its range; everything outside it runs on the general path."""
    from wav2sleep_b200.model import MultiModalAttentionEmbedder, SequenceCNN, SignalEncoders, Wav2Sleep
    enc = SignalEncoders(signal_map={"ECG": "ECG"}, feature_dim=128, activation="gelu", norm="instance", causal=False,
                         chunk_causal=False)
    mix = MultiModalAttentionEmbedder(feature_dim=128, activation="gelu", layers=mixer_layers, dim_ff=512, nhead=8)
    seq = SequenceCNN(feature_dim=128, activation="gelu", norm="layer", num_layers=seq_blocks, kernel_size=7,
                      num_dilations=seq_dilations)
    assert Wav2Sleep(enc, mix, seq, ncls).fast_path is fast
