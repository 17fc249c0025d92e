"""Seeded synthetic checkpoints and audio for tests and benchmarks.

There is no network in the build/bench environment, so the published checkpoints
("final0", "small0", reference beat_this/inference.py:13,38-48) cannot be fetched.
This module writes checkpoints in the *exact* ``.ckpt`` layout the reference loads
(reference inference.py:56-87, key list in SURVEY.md App. B): a ``torch.save``d dict
with ``state_dict`` (keys prefixed ``model.``) and ``hyper_parameters``.

Conv2d weights follow the reference initialiser (beat_tracker.py:170-186, kaiming-normal
fan_out); Linear weights are variance-preserving N(0, 1/fan_in) rather than N(0, .02) so that
every residual branch carries signal and the logits vary in time; BatchNorm statistics and
affines, RMSNorm gammas and biases are randomised so that folding mistakes cannot hide
behind identity values.
"""
from __future__ import annotations

import math
import os
import tempfile
from collections import OrderedDict

import numpy as np
import torch

SAMPLE_RATE = 22050


def model_hparams(name: str = "final0") -> dict:
    """BeatThis constructor arguments as stored in ``hyper_parameters`` (pl_module.py:22-44)."""
    # "<base>-nosum" / "<base>-nopartial": the ablation families of the reference README (sum_head=False ->
    # Head, beat_tracker.py:333-346; partial_transformers=False -> nn.Identity, beat_tracker.py:151-152)
    base, _, variant = name.partition("-")
    dim = {"final0": 512, "small0": 128}[base] if base in ("final0", "small0") else int(base)
    return dict(
        spect_dim=128,
        fps=50,
        transformer_dim=dim,
        ff_mult=4,
        n_layers=6,
        stem_dim=32,
        dropout={"frontend": 0.1, "transformer": 0.2},
        lr=0.0008,
        weight_decay=0.01,
        pos_weights={"beat": 1, "downbeat": 1},
        head_dim=32,
        loss_type="shift_tolerant_weighted_bce",
        warmup_steps=1000,
        max_epochs=100,
        use_dbn=False,
        eval_trim_beats=5,
        sum_head=variant != "nosum",
        partial_transformers=variant != "nopartial",
    )


def _bn(sd, prefix, n, g, mean_range=(-0.2, 0.2), var_range=(0.5, 1.5)):
    sd[prefix + ".weight"] = torch.empty(n).uniform_(0.6, 1.4, generator=g)
    sd[prefix + ".bias"] = torch.empty(n).normal_(0, 0.1, generator=g)
    sd[prefix + ".running_mean"] = torch.empty(n).uniform_(*mean_range, generator=g)
    sd[prefix + ".running_var"] = torch.empty(n).uniform_(*var_range, generator=g)
    sd[prefix + ".num_batches_tracked"] = torch.tensor(1000, dtype=torch.int64)


def _linear(sd, prefix, n_out, n_in, g, bias=True, std=None):
    if std is None:
        # variance-preserving instead of the reference's N(0,.02): with .02 every residual
        # branch is ~0 and the logits come out flat in time (useless for parity testing)
        std = 1.0 / math.sqrt(n_in)
    sd[prefix + ".weight"] = torch.empty(n_out, n_in).normal_(0, std, generator=g)
    if bias:
        sd[prefix + ".bias"] = torch.empty(n_out).normal_(0, 0.02, generator=g)


def _conv(sd, key, c_out, c_in, kh, kw, g):
    std = math.sqrt(2.0 / (c_out * kh * kw))  # kaiming_normal_, fan_out, relu gain
    sd[key] = torch.empty(c_out, c_in, kh, kw).normal_(0, std, generator=g)


def _attention(sd, prefix, dim, g, head_dim=32):
    heads = dim // head_dim
    sd[prefix + ".rotary_embed.freqs"] = 1.0 / (
        10000 ** (torch.arange(0, head_dim, 2).float() / head_dim)
    )
    sd[prefix + ".norm.gamma"] = torch.empty(dim).uniform_(0.7, 1.3, generator=g)
    # wider than N(0,.02): scores get std ~1.4 so softmax is far from uniform and RoPE matters
    _linear(sd, prefix + ".to_qkv", 3 * dim, dim, g, bias=False, std=1.2 / math.sqrt(dim))
    _linear(sd, prefix + ".to_gates", heads, dim, g, bias=True)
    _linear(sd, prefix + ".to_out.0", dim, dim, g, bias=False)


def _feedforward(sd, prefix, dim, mult, g):
    sd[prefix + ".net.0.gamma"] = torch.empty(dim).uniform_(0.7, 1.3, generator=g)
    _linear(sd, prefix + ".net.1", dim * mult, dim, g)
    _linear(sd, prefix + ".net.4", dim, dim * mult, g)


def make_state_dict(hp: dict, seed: int = 0) -> "OrderedDict[str, torch.Tensor]":
    """Seeded BeatThis state_dict (un-prefixed keys), key order as in the reference module."""
    g = torch.Generator().manual_seed(seed)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    D = hp["transformer_dim"]
    stem = hp["stem_dim"]
    _bn(sd, "frontend.stem.bn1d", hp["spect_dim"], g, mean_range=(2.0, 4.0), var_range=(0.5, 2.0))
    _conv(sd, "frontend.stem.conv2d.weight", stem, 1, 4, 3, g)
    _bn(sd, "frontend.stem.bn2d", stem, g)
    c = stem
    for i in range(3):
        p = f"frontend.blocks.{i}"
        if hp.get("partial_transformers", True):
            _attention(sd, p + ".partial.attnF", c, g)
            _feedforward(sd, p + ".partial.ffF", c, 4, g)
            _attention(sd, p + ".partial.attnT", c, g)
            _feedforward(sd, p + ".partial.ffT", c, 4, g)
        _conv(sd, p + ".conv2d.weight", 2 * c, c, 2, 3, g)
        _bn(sd, p + ".norm", 2 * c, g)
        c *= 2
    f_out = hp["spect_dim"] // 4 // 8
    _linear(sd, "frontend.linear", D, c * f_out, g)
    for l in range(hp["n_layers"]):
        _attention(sd, f"transformer_blocks.layers.{l}.0", D, g)
        _feedforward(sd, f"transformer_blocks.layers.{l}.1", D, hp["ff_mult"], g)
    sd["transformer_blocks.norm.gamma"] = torch.empty(D).uniform_(0.7, 1.3, generator=g)
    # a wider head than N(0,.02) so that logits are not all hugging the 0 threshold
    _linear(sd, "task_heads.beat_downbeat_lin", 2, D, g, std=0.4)
    # head bias calibrated by hand (per model size, for seed 0) so that both logit tracks
    # straddle the 0 threshold on the synthetic clips and peak picking has work to do
    bias = {512: [4.5, -1.2], 128: [2.4, -0.8]}.get(D, [0.0, 0.0])
    sd["task_heads.beat_downbeat_lin.bias"] = torch.tensor(bias)
    return sd


def make_checkpoint(name: str = "final0", seed: int = 0) -> dict:
    hp = model_hparams(name)
    sd = make_state_dict(hp, seed)
    return {
        "state_dict": OrderedDict(("model." + k, v) for k, v in sd.items()),
        "hyper_parameters": hp,
        "datamodule_hyper_parameters": {},
        "pytorch-lightning_version": "2.1.0",
    }


def cache_dir() -> str:
    """Where tests and benchmarks keep the checkpoints and audio they generate: $BT_TEST_CACHE, else a directory of
    the calling user's own under the system's temporary directory (another user's copy there is not writable)."""
    return os.environ.get("BT_TEST_CACHE") or os.path.join(tempfile.gettempdir(), f"beat_this_b200_cache_{os.getuid()}")


def write_checkpoint(path: str, name: str = "final0", seed: int = 0) -> str:
    """Write the synthetic checkpoint (idempotent); returns ``path``."""
    if not os.path.exists(path):
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        tmp = f"{path}.tmp{os.getpid()}"
        torch.save(make_checkpoint(name, seed), tmp)
        os.replace(tmp, path)
    return path


def synth_clip(index: int, seconds: float = 30.0, sr: int = SAMPLE_RATE) -> np.ndarray:
    """Seeded synthetic mono clip: low noise plus decaying click/sine bursts on a per-clip
    tempo grid (60-180 BPM) so that the activations are not degenerate (SURVEY.md 8d)."""
    rng = np.random.default_rng(1000 + index)
    n = int(round(seconds * sr))
    x = 0.004 * rng.standard_normal(n)
    bpm = rng.uniform(60.0, 180.0)
    period = 60.0 / bpm
    phase = rng.uniform(0.0, period)
    burst_len = int(0.25 * sr)
    tt = np.arange(burst_len) / sr
    k = 0
    while True:
        t0 = phase + k * period
        s0 = int(t0 * sr)
        if s0 >= n:
            break
        f = 220.0 * (2.0 if k % 4 == 0 else 1.0) * (1.0 + 0.02 * rng.standard_normal())
        amp = 0.8 if k % 4 == 0 else 0.5
        burst = amp * np.exp(-tt * 30.0) * np.sin(2 * np.pi * f * tt)
        burst[:32] += amp * 0.5 * rng.standard_normal(32)  # click
        e = min(n, s0 + burst_len)
        x[s0:e] += burst[: e - s0]
        k += 1
    return np.clip(x, -1.0, 1.0).astype(np.float64)


def tensor_checksum(sd: dict) -> float:
    """Order-independent float64 checksum of a state dict (pins fixture <-> checkpoint)."""
    tot = 0.0
    for k in sorted(sd):
        v = sd[k].double()
        tot += float(v.sum()) + 1e-3 * float((v * v).sum())
    return tot


# int16 WAV material of the CLI byte-parity fixture (tests/golden/cli_beats.npz, oracle/make_golden_cli.py):
# (file name, seed of synth_clip, seconds, channels)
CLI_CASES = [("one.wav", 301, 10.0, 1), ("sub/two.wav", 302, 31.5, 1), ("sub/stereo.wav", 303, 7.0, 2)]


def pcm16(seed: int, secs: float, channels: int) -> np.ndarray:
    """16-bit PCM of synth_clip(seed, secs); the second channel of a stereo file is the reversed clip at half level."""
    data = np.round(synth_clip(seed, secs) * 32767).astype(np.int16)
    return data if channels == 1 else np.stack([data, data[::-1] // 2], axis=1)
