"""Log-mel write-out of the fused kernel, on 48 kHz mono f32 batches (the kernel cfg2 runs).  Rows whose base is 16-byte
aligned are written with 16-byte stores, a base 4 bytes off 16 takes the scalar stores: both must give the same bits for
every step shape (last steps with 1 to 32 valid frames, streams shorter than a tile), and neither may write past a
stream's T x n_mels values of its row.  Host batches of several sub-batches, each launched over its own step-balanced
tile order, must give the rows a device batch gives."""
import numpy as np
import pytest

import audioflow as af_mod

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FBADBAD          # a NaN pattern the kernel never produces


def _n_in_for_frames(T: int, extra: int = 0) -> int:
    """Length of a 48 kHz input whose 16 kHz output has exactly T STFT frames (extra: output samples past the last hop)."""
    n_out = 400 + (T - 1) * 160 + extra if T > 0 else 100
    n = 3 * n_out
    while af_mod.resample_output_len(48000, 16000, n) > n_out:
        n -= 1
    while af_mod.resample_output_len(48000, 16000, n) < n_out:
        n += 1
    return n


def _run_device(af, xs, cfg, offset):
    """log-mel rows (uint32, [S, stride]) of a device batch over the 48 kHz mono f32 streams xs, the output base `offset`
    bytes past a 16-byte boundary, every other word pre-filled with SENTINEL; and the frame counts"""
    import torch
    dev = torch.device("cuda")
    arrs = [torch.tensor(x, device=dev) for x in xs]
    pipe = af.Pipeline(cfg)
    b = pipe.batch([(a.data_ptr(), len(x), 48000, 1, af.AF_FMT_F32) for a, x in zip(arrs, xs)], af.AF_MEM_DEVICE)
    S, stride = len(xs), b.logmel_stride
    lm = torch.full((S * stride + 4,), SENTINEL, device=dev, dtype=torch.int32)
    torch.cuda.synchronize()            # torch fills run on the legacy stream; the library uses its own non-blocking stream
    b.run_device(b.outputs_struct(0, 0, lm.data_ptr() + offset, stride))
    torch.cuda.synchronize()
    out = lm.cpu().numpy().view(np.uint32)
    w = offset // 4
    return out[w:w + S * stride].reshape(S, stride), b.n_feat[:S].astype(np.int64)


def _check_pair(af, xs, cfg):
    M = cfg.n_mels
    vec, T = _run_device(af, xs, cfg, 0)
    direct, T2 = _run_device(af, xs, cfg, 4)
    assert np.array_equal(T, T2)
    for i, t in enumerate(T):
        n = int(t) * M
        assert np.array_equal(vec[i, :n], direct[i, :n]), f"stream {i}: vector and scalar log-mel stores differ"
        assert not (vec[i, :n] == SENTINEL).any(), f"stream {i}: a log-mel value was not written"
        assert (vec[i, n:] == SENTINEL).all(), f"stream {i}: written past T x n_mels (vector stores)"
        assert (direct[i, n:] == SENTINEL).all(), f"stream {i}: written past T x n_mels (scalar stores)"
    return vec, T


# last steps with 1, 22, 31 and 32 valid frames, streams shorter than one tile (128 frames) and one without frames
FRAMES = [321, 22, 159, 384, 100, 1, 0, 2 * 128 + 31]


def _streams(seed):
    from audioflow import synth
    return [synth.stream(seed + i, _n_in_for_frames(T, extra=11 * i) / 48000.0, 48000, 1) for i, T in enumerate(FRAMES)]


@pytest.mark.parametrize("n_mels", [40, 64, 80, 81, 128])
def test_vector_and_scalar_stores_agree(af, n_mels):
    xs = _streams(1000 + n_mels)
    _, T = _check_pair(af, xs, af.pipeline_config(n_mels=n_mels, vad_enable=False))
    assert sorted(set(int(t) for t in T)) == sorted(set(FRAMES))


@pytest.mark.parametrize("log10,floor", [(True, 1e-10), (False, 1e-10), (False, 1e-6), (True, 3e-4)])
def test_vector_and_scalar_stores_agree_log_and_floor(af, log10, floor):
    xs = _streams(2000)
    _check_pair(af, xs, af.pipeline_config(n_mels=80, vad_enable=True, log10=log10, log_floor=floor))


def test_host_batch_of_several_sub_batches_matches_direct(af):
    """About 50 MB of input: a host batch of two sub-batches, each launched over its own step-balanced tile order."""
    from audioflow import synth
    rng = np.random.default_rng(7)
    secs = [float(s) for s in rng.uniform(20.0, 40.0, 10)] + [0.01, 2.7]
    xs = [synth.stream(3000 + i, s, 48000, 1) for i, s in enumerate(secs)]
    assert sum(len(x) for x in xs) * 4 > 40 << 20
    cfg = af.pipeline_config(n_mels=80)
    host = af.Pipeline(cfg).run_host([(x, 48000, 1) for x in xs])
    direct, T = _run_device(af, xs, cfg, 4)
    for i, (g, t) in enumerate(zip(host, T)):
        assert g["logmel"].shape == (int(t), 80)
        assert np.array_equal(g["logmel"].reshape(-1).view(np.uint32), direct[i, :int(t) * 80]), f"stream {i}"
