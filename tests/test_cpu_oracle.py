"""CPU tests (no GPU): the oracle restatement against the golden fixtures generated from the
UNMODIFIED reference (oracle/make_golden*.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

from beat_this_b200 import synthetic
from oracle import beat_this_oracle as O


def test_logmel_golden():
    g = np.load(os.path.join(GOLDEN, "logmel.npz"))
    assert int(g["fb_nnz"]) == int((O.mel_filterbank() != 0).sum()) == 1004
    for idx in (0, 1):
        x = synthetic.synth_clip(idx, float(g[f"clip{idx}_secs"]))
        m = O.logmel(torch.tensor(x, dtype=torch.float32)).numpy()
        assert m.shape == g[f"clip{idx}_mel"].shape
        assert np.abs(m - g[f"clip{idx}_mel"]).max() < 1e-4
        m64 = O.logmel(torch.tensor(x, dtype=torch.float32), torch.float64).numpy()
        assert np.abs(m64 - g[f"clip{idx}_mel"]).max() < 1e-3  # fp32 FFT noise under log1p(1000 x)


def test_chunking_golden():
    g = np.load(os.path.join(GOLDEN, "chunking.npz"))
    for T in g["Ts"]:
        T = int(T)
        assert np.array_equal(O.split_starts(T), g[f"starts_{T}"])
        chunks, starts = O.split_piece(torch.zeros(T, 2))
        assert [len(c) for c in chunks] == list(g[f"lens_{T}"])


def test_postp_minimal_golden():
    g = np.load(os.path.join(GOLDEN, "postp_minimal.npz"))
    for i in range(int(g["n"])):
        bt, dt = O.postp_minimal(torch.tensor(g[f"beat_{i}"]), torch.tensor(g[f"down_{i}"]))
        assert np.array_equal(bt, g[f"beat_times_{i}"]), i
        assert np.array_equal(dt, g[f"down_times_{i}"]), i


def test_dedup_known_answers():
    # SURVEY.md A.5: the merge compares against the running mean
    assert np.array_equal(O.deduplicate_peaks([10, 11, 12]), [10.5, 12])
    assert np.array_equal(O.deduplicate_peaks([]), [])
    assert np.array_equal(O.deduplicate_peaks([3, 4, 9, 10, 20]), [3.5, 9.5, 20])


def test_model_golden_small0(small0_ckpt):
    """BASELINE config 1 (Spect2Frames small0, one random 1500-frame spectrogram, CPU)."""
    g = np.load(os.path.join(GOLDEN, "model.npz"))
    sd = O.strip_prefix(torch.load(small0_ckpt, weights_only=True)["state_dict"])
    assert abs(synthetic.tensor_checksum(sd) - float(g["small0_ckpt_sum"])) < 1e-6 * abs(float(g["small0_ckpt_sum"]))
    torch.manual_seed(0)
    spect = torch.rand(1500, 128) * 7
    b, d = O.spect2frames(sd, spect)
    assert b.shape == (1500,) and b.dtype == torch.float32
    assert np.abs(b.numpy() - g["small0_spect1500_beat"]).max() < 2e-4
    assert np.abs(d.numpy() - g["small0_spect1500_down"]).max() < 2e-4


@pytest.mark.parametrize("variant", ["small0-nosum", "small0-nopartial"])
def test_model_golden_ablation_families(variant):
    """sum_head=False (Head, beat_tracker.py:333-346) and partial_transformers=False (nn.Identity,
    beat_tracker.py:151-152): fixtures written by the reference's own Spect2Frames (oracle/make_golden.py)."""
    from conftest import ckpt_path

    g = np.load(os.path.join(GOLDEN, "model.npz"))
    key = variant.replace("-", "_")
    ck = torch.load(ckpt_path(variant), weights_only=True)
    sd = O.strip_prefix(ck["state_dict"])
    assert abs(synthetic.tensor_checksum(sd) - float(g[f"{key}_ckpt_sum"])) < 1e-6 * abs(float(g[f"{key}_ckpt_sum"]))
    torch.manual_seed(5)
    spect = torch.rand(1700, 128) * 7
    b, d = O.spect2frames(sd, spect, sum_head=ck["hyper_parameters"]["sum_head"])
    assert np.abs(b.numpy() - g[f"{key}_spect1700_beat"]).max() < 2e-4
    assert np.abs(d.numpy() - g[f"{key}_spect1700_down"]).max() < 2e-4


def test_model_golden_final0_short_clip(final0_ckpt):
    g = np.load(os.path.join(GOLDEN, "model.npz"))
    sd = O.strip_prefix(torch.load(final0_ckpt, weights_only=True)["state_dict"])
    assert abs(synthetic.tensor_checksum(sd) - float(g["final0_ckpt_sum"])) < 1e-6 * abs(float(g["final0_ckpt_sum"]))
    x = synthetic.synth_clip(1, float(g["final0_clip1_secs"]))
    b, d = O.spect2frames(sd, O.signal2spect(x, 22050))
    assert np.abs(b.numpy() - g["final0_clip1_beat"]).max() < 5e-4
    assert np.abs(d.numpy() - g["final0_clip1_down"]).max() < 5e-4
    bt, dt = O.postp_minimal(b, d)
    assert np.array_equal(bt, g["final0_clip1_beat_times"]) and np.array_equal(dt, g["final0_clip1_down_times"])


def test_oracle_against_live_reference(small0_ckpt):
    """The reference's BeatThis module and split_piece, as recorded by oracle/make_golden_forward.py."""
    from oracle.make_golden_forward import FORWARD_SEED, SPLIT_LENGTHS

    g = np.load(os.path.join(GOLDEN, "reference_forward.npz"))
    sd = O.strip_prefix(torch.load(small0_ckpt, weights_only=True)["state_dict"])
    assert abs(synthetic.tensor_checksum(sd) - float(g["small0_ckpt_sum"])) < 1e-6 * abs(float(g["small0_ckpt_sum"]))
    # the reference's load_model loads strictly: the synthetic .ckpt must have its layout, name for name
    assert {k: str(tuple(v.shape)) for k, v in sd.items()} == dict(zip(g["state_keys"].tolist(), g["state_shapes"].tolist()))
    torch.manual_seed(FORWARD_SEED)
    x = torch.rand(2, 100, 128) * 7
    with torch.inference_mode():
        b, d = O.forward(sd, x)
        eb, ed = O.forward(sd, x, explicit=True)
    assert np.abs(g["beat"] - b.numpy()).max() < 1e-4 and np.abs(g["downbeat"] - d.numpy()).max() < 1e-4
    assert (eb - b).abs().max() < 1e-4
    for T in SPLIT_LENGTHS:
        assert np.array_equal(g[f"starts_{T}"], O.split_starts(T))


# ------------------------------------------------------------------------------------ resampler
@pytest.mark.parametrize("sr", [44100, 48000, 16000, 8000, 96000, 11025, 32000])
def test_resample_bank_equals_direct_form(sr):
    """The polyphase bank the CUDA kernel consumes (preprocessing.resample_filter_bank) reproduces the float64
    direct-form definition (oracle.resample_direct) -- bank construction and tap indexing are independent code."""
    from beat_this_b200 import preprocessing as P

    rng = np.random.default_rng(sr)
    x = rng.standard_normal(2500)
    coef, L, M, K = P.resample_filter_bank(sr)
    assert coef.shape == (L, K) and K % 2 == 0 and abs(coef.astype(np.float64).sum(1).mean() - 1.0) < 1e-6
    n_out = P.resampled_length(len(x), L, M)
    n = np.arange(n_out)
    j = ((n * M) // L)[:, None] - K // 2 + 1 + np.arange(K)[None, :]
    xv = np.where((j >= 0) & (j < len(x)), x[np.clip(j, 0, len(x) - 1)], 0.0)
    y_bank = (xv * coef[(n * M) % L].astype(np.float64)).sum(1)
    y = O.resample_direct(x, sr)
    assert y.shape == y_bank.shape and np.abs(y - y_bank).max() < 1e-6


def test_resample_filter_meets_its_design_targets():
    """Design targets stated in preprocessing.py (soxr-HQ-like): a 1 kHz and a 10 kHz tone pass 44.1 -> 22.05 kHz
    unchanged, a 12 kHz tone (above the new Nyquist) is rejected by more than 120 dB."""
    sr = 44100
    t = np.arange(sr // 2) / sr
    t2 = np.arange(len(t) // 2) / 22050
    for f, tol in ((1000.0, 1e-7), (10000.0, 1e-5)):
        y = O.resample_direct(np.sin(2 * np.pi * f * t), sr)
        assert len(y) == len(t2) and np.abs(y[400:-400] - np.sin(2 * np.pi * f * t2)[400:-400]).max() < tol
    y = O.resample_direct(np.sin(2 * np.pi * 12000.0 * t), sr)
    assert 20 * np.log10(np.abs(y[400:-400]).max()) < -120.0
