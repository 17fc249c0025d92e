"""CPU tests (no GPU) of the host logic: packed-parameter folds, the native chunk planner,
the C-ABI surface, the API mirror, TSV writer, multi-process (gloo) sharding + broadcast."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT

from beat_this_b200 import synthetic, weights


def test_abi_exports_every_declared_symbol(lib_built):
    hdr = open(os.path.join(ROOT, "include", "beatthis.h")).read()
    declared = set(re.findall(r"\b(bt_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"bt_ctx", "bt_hparams"}
    from beat_this_b200 import _lib

    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    for name in declared:
        assert hasattr(lib_built, name), name
    assert lib_built.bt_version() >= 100


def test_native_chunk_planner_matches_reference_table(lib_built):
    g = np.load(os.path.join(GOLDEN, "chunking.npz"))
    from beat_this_b200.inference import split_piece

    st = (ctypes.c_int64 * 64)()
    ln = (ctypes.c_int64 * 64)()
    for T in list(g["Ts"]) + [2, 13, 1487, 2975, 2976, 100000]:
        T = int(T)
        n = lib_built.bt_plan_chunks(T, st, ln, 64)
        chunks, starts = split_piece(torch.zeros(T, 1), 1500, 6, True)  # host mirror of the reference function
        if n <= 64:
            assert list(st[:n]) == list(starts), T
            assert list(ln[:n]) == [len(c) for c in chunks], T
        assert n == len(starts)
        if f"starts_{T}" in g:
            assert list(st[:n]) == list(g[f"starts_{T}"])
    assert lib_built.bt_plan_chunks(0, None, None, 0) == 0
    assert lib_built.bt_num_frames(661500) == 1501 and lib_built.bt_num_frames(440) == 1


def test_no_gpu_fails_loudly(lib_built):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from beat_this_b200 import _lib
    from beat_this_b200.inference import Spect2Frames

    hp = _lib.bt_hparams(128, 128, 4, 6, 32, 32, 1, 1)
    ctx = ctypes.c_void_p()
    code = lib_built.bt_create(ctypes.byref(ctx), 0, ctypes.byref(hp), 0)
    assert code != 0 and b"no CPU fallback" in lib_built.bt_last_error(None)
    with pytest.raises(RuntimeError):
        Spect2Frames("whatever.ckpt", "cpu")


@pytest.mark.parametrize("name", ["small0", "small0-nosum", "small0-nopartial"])
def test_packed_parameters_reproduce_the_oracle(name):
    """Fold/layout logic of weights.py: the kernel schedule emulated in torch with the packed
    parameters (tests/packed_forward.py) must equal the oracle forward, stage by stage."""
    import packed_forward as PF
    from oracle import beat_this_oracle as O

    hp = synthetic.model_hparams(name)
    sd = synthetic.make_state_dict(hp, 0)
    packed = weights.pack_parameters(sd, hp)
    torch.manual_seed(1)
    x = torch.rand(2, 90, 128) * 7
    t1, t2 = {}, {}
    with torch.inference_mode():
        b, d = O.forward(sd, x, t1, sum_head=hp["sum_head"])
        b2, d2 = PF.forward(packed, weights.filter_hparams(hp), x, t2)
    for k in t1:
        assert (t1[k] - t2[k]).abs().max() < 1e-4, k
    assert (b - b2).abs().max() < 1e-4 and (d - d2).abs().max() < 1e-4
    blob, names, sizes = weights.blob_from_packed(packed)
    back = weights.packed_from_blob(blob, names, sizes)
    assert all(np.array_equal(back[k], packed[k]) for k in packed)


def test_checkpoint_layout_roundtrip(small0_ckpt, monkeypatch):
    from beat_this_b200.inference import CHECKPOINT_URL, load_checkpoint

    ck = load_checkpoint(small0_ckpt)
    assert set(ck) >= {"state_dict", "hyper_parameters"}
    assert all(k.startswith("model.") for k in ck["state_dict"])
    assert len(ck["state_dict"]) == 166
    assert sum(v.numel() for v in ck["state_dict"].values()) == 2101357  # SURVEY.md App. B (small0)
    # a path that is not a file falls through to the URL path; the download is stubbed to fail as it does offline
    urls = []

    def no_network(url, **kw):
        urls.append(url)
        raise OSError("no network")

    monkeypatch.setattr(torch.hub, "load_state_dict_from_url", no_network)
    with pytest.raises(ValueError):
        load_checkpoint("/nonexistent/dir/nothing-here")
    assert urls == [f"{CHECKPOINT_URL}//nonexistent/dir/nothing-here.ckpt"]


def test_api_surface_matches_reference_names():
    import beat_this_b200.inference as I

    for name in ["load_checkpoint", "load_model", "zeropad", "split_piece", "aggregate_prediction", "Spect2Frames",
                 "Audio2Frames", "Audio2Beats", "File2Beats", "File2File", "CHECKPOINT_URL"]:
        assert hasattr(I, name), name
    assert issubclass(I.File2File, I.File2Beats) and issubclass(I.File2Beats, I.Audio2Beats)
    assert issubclass(I.Audio2Beats, I.Audio2Frames) and issubclass(I.Audio2Frames, I.Spect2Frames)
    # aggregate_prediction mirror: keep_first
    chunks, starts = I.split_piece(torch.arange(3001.0)[:, None].repeat(1, 2), 1500, 6, True)
    preds = [{"beat": c[:, 0] + 10000 * i, "downbeat": c[:, 1]} for i, c in enumerate(chunks)]
    b, d = I.aggregate_prediction(preds, starts, 3001, 1500, 6, "keep_first", "cpu")
    assert torch.equal(d, torch.arange(3001.0))
    assert b[1487] == 1487 and b[1488] == 1488 + 10000 and b[2976] == 2976 + 20000 and b[2975] == 2975 + 10000


def test_save_beat_tsv_and_beat_numbers(tmp_path):
    from beat_this_b200.utils import infer_beat_numbers, save_beat_tsv

    beats = np.array([0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 3.5])
    downs = np.array([1.0, 3.0])
    assert list(infer_beat_numbers(beats, downs)) == [4, 1, 2, 3, 4, 1, 2]
    with pytest.raises(ValueError):
        infer_beat_numbers(beats, np.array([0.75]))
    out = tmp_path / "sub" / "x.beats"
    save_beat_tsv(beats, downs, str(out))
    assert out.read_text().splitlines()[:2] == ["0.5\t4", "1.0\t1"]


def test_load_audio_wav(tmp_path):
    from scipy.io import wavfile

    from beat_this_b200.preprocessing import load_audio

    x = (np.sin(np.arange(2000) / 10) * 20000).astype(np.int16)
    wavfile.write(tmp_path / "a.wav", 22050, np.stack([x, x // 2], 1))
    wav, sr = load_audio(tmp_path / "a.wav")
    assert sr == 22050 and wav.shape == (2000, 2) and wav.dtype == np.float64
    assert np.allclose(wav[:, 0], x / 32768.0)
    with pytest.raises(RuntimeError):
        load_audio(tmp_path / "missing.wav")


def test_mel_constants_match_oracle_filterbank():
    from beat_this_b200.preprocessing import mel_constants, mel_filterbank
    from oracle import beat_this_oracle as O

    assert torch.equal(mel_filterbank(), O.mel_filterbank())
    c = mel_constants()
    ptr = c["mel.fb_ptr"].astype(int)
    assert ptr[-1] == 1004 and len(c["mel.fb_w"]) == 1004
    fb = O.mel_filterbank().numpy()
    for m in (0, 5, 64, 127):
        s = int(c["mel.fb_start"][m])
        w = c["mel.fb_w"][ptr[m]:ptr[m + 1]]
        assert np.array_equal(fb[s:s + len(w), m], w) and fb[:, m].sum() == pytest.approx(w.sum())


GLOO_WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from beat_this_b200 import synthetic, weights
from beat_this_b200.distributed import init_from_env, broadcast_packed, shard_indices, shard_by_cost, gather_results
rank, world, local = init_from_env("gloo")
packed = hp = None
if rank == 0:
    hp = weights.filter_hparams(synthetic.model_hparams("small0"))
    packed = weights.pack_parameters(synthetic.make_state_dict(synthetic.model_hparams("small0"), 0), hp)
packed, hp = broadcast_packed(packed, hp, "cpu")
chk = float(sum(float(np.abs(v).sum()) for v in packed.values()))
mine = shard_indices(10, rank, world)
res = gather_results({i: (i * i, rank) for i in mine}, world)
assert sorted(res) == list(range(10)) and all(res[i][0] == i * i for i in res)
parts = shard_by_cost([11, 1, 1, 1, 5, 5, 2], world)
assert sorted(sum(parts, [])) == list(range(7))
t = torch.tensor([chk], dtype=torch.float64)
lst = [torch.zeros_like(t) for _ in range(world)]
dist.all_gather(lst, t)
assert all(abs(float(x) - chk) < 1e-9 for x in lst), "ranks hold different weights"
if rank == 0:
    print("GLOO_OK", hp["transformer_dim"], len(packed))
dist.destroy_process_group()
"""


def test_world_size_2_gloo_broadcast_and_sharding(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="2")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", str(script), ROOT]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    assert "GLOO_OK 128" in res.stdout


def test_cli_output_naming_and_task_collection(tmp_path):
    """Output naming of the command line tool (reference cli.py:94-112,150-168): suffix replace / append, output
    directory keeps the path relative to the directory named on the command line, existing outputs and files that
    already carry the suffix are skipped."""
    from pathlib import Path

    from beat_this_b200 import cli

    f = Path("/music/a/song.wav")
    assert cli.output_path_for(f, ".beats", False) == Path("/music/a/song.beats")
    assert cli.output_path_for(f, ".beats", True) == Path("/music/a/song.wav.beats")
    assert cli.output_path_for(f, ".beats", False, Path("/out")) == Path("/out/song.beats")
    assert cli.output_path_for(f, ".beats", False, Path("/out"), root=Path("/music")) == Path("/out/a/song.beats")
    assert cli.output_path_for(f, ".txt", True, Path("/out"), root=Path("/music")) == Path("/out/a/song.wav.txt")

    (tmp_path / "in" / "sub").mkdir(parents=True)
    for name in ("x.wav", "sub/y.wav", "sub/y.beats", "z.flac"):
        (tmp_path / "in" / name).write_bytes(b"")
    tasks, single = cli.collect_tasks([str(tmp_path / "in")], str(tmp_path / "out"), ".beats", False, False)
    assert not single
    assert sorted(str(d.relative_to(tmp_path / "out")) for _, d in tasks) == ["sub/y.beats", "x.beats", "z.beats"]
    (tmp_path / "out").mkdir()
    (tmp_path / "out" / "x.beats").write_text("")
    tasks, _ = cli.collect_tasks([str(tmp_path / "in")], str(tmp_path / "out"), ".beats", False, True)
    assert sorted(s.name for s, _ in tasks) == ["y.wav", "z.flac"]
    tasks, single = cli.collect_tasks([str(tmp_path / "in" / "x.wav")], None, ".beats", False, False)
    assert single and tasks == [(tmp_path / "in" / "x.wav", tmp_path / "in" / "x.beats")]
    tasks, single = cli.collect_tasks([str(tmp_path / "in" / "x.wav")], str(tmp_path / "named.tsv"), ".beats", False, False)
    assert single and tasks[0][1] == tmp_path / "named.tsv"
    args = cli.build_parser().parse_args(["a.wav", "--float16", "--no-dbn", "-o", "o", "--touch-first"])
    assert args.float16 and not args.dbn and args.output == "o" and args.touch_first and args.suffix == ".beats"
    assert cli._claim(tmp_path / "lock" / "t.beats", True, True) and not cli._claim(tmp_path / "lock" / "t.beats", True, True)


def test_native_dbn_viterbi_equals_dense_bruteforce(lib_built):
    """The vectorised Viterbi of beat_this_b200/dbn.py (position shift + a small tempo matrix at beat boundaries)
    against a textbook dense O(T S^2) decoder built independently from the model's published definition."""
    from beat_this_b200.dbn import _BarModel

    rng = np.random.default_rng(0)
    for beats in (3, 4):
        m = _BarModel(beats, 60.0 * 10 / 215.0, 60.0 * 10 / 55.0, None, 100, 16)  # fps 10: 63 states per beat
        S = m.num_states
        per_beat = S // beats
        # dense log transition matrix A[prev, next]
        A = np.full((S, S), -np.inf)
        first = set(int(v) for v in m.first_states.ravel())
        for s_ in range(S):
            if s_ not in first:
                A[s_ - 1, s_] = 0.0
        starts = np.cumsum(np.r_[0, m.intervals[:-1]])
        for b in range(beats):
            for k_to, i_to in enumerate(m.intervals):
                for k_from, i_from in enumerate(m.intervals):
                    p = np.exp(-100 * abs(i_to / i_from - 1.0))
                    row = np.exp(-100 * np.abs(m.intervals / i_from - 1.0))
                    row[row <= np.spacing(1.0)] = 0.0
                    if p > np.spacing(1.0):
                        prev = ((b - 1) % beats) * per_beat + starts[k_from] + i_from - 1
                        A[prev, b * per_beat + starts[k_to]] = np.log(p / row.sum())
        act = rng.uniform(0.01, 0.3, (40, 2))  # rows sum to < 1 like (beat - downbeat, downbeat) probabilities
        act[::7] = (0.7, 0.05)
        act[::21] = (0.05, 0.8)
        dens = m.log_densities(act)[:, m.pointers]
        v = np.full(S, -np.log(S))
        bp = np.zeros((len(act), S), dtype=int)
        for t in range(len(act)):
            cand = v[:, None] + A
            bp[t] = cand.argmax(0)
            v = cand.max(0) + dens[t]
        st = int(v.argmax())
        ref_logp, ref_path = float(v[st]), []
        for t in range(len(act) - 1, -1, -1):
            ref_path.append(st)
            st = bp[t, st]
        for decode in (m.viterbi_numpy, m.viterbi):  # numpy form and the C++ decoder of the shared library
            path, logp = decode(act)
            assert abs(logp - ref_logp) < 1e-9 and np.array_equal(path, ref_path[::-1])


def test_dbn_state_space_known_answers():
    """Known answers for the bar-pointer state space, transition and observation model.  madmom is not installable
    offline, so these are the small examples of madmom's own published documentation (madmom.features.beats_hmm:
    the docstring examples of BeatStateSpace(1, 4) and BarStateSpace(2, 1, 4), exponential_transition and
    RNNDownBeatTrackingObservationModel) plus the sizes that follow from the reference's configuration
    (postprocessor.py:29-37: fps 50, 55..215 BPM -> beat intervals 14..55 frames)."""
    from beat_this_b200.dbn import DBNDownBeatTracker, _BarModel

    m = _BarModel(1, 1, 4, None, 100, 16)  # BeatStateSpace(1, 4)
    assert m.num_states == 10 and m.intervals.tolist() == [1, 2, 3, 4]
    assert m.first_states.tolist() == [[0, 1, 3, 6]] and m.last_states.tolist() == [[0, 2, 5, 9]]
    assert np.allclose(m.positions, [0, 0, 0.5, 0, 1 / 3, 2 / 3, 0, 0.25, 0.5, 0.75])
    m = _BarModel(2, 1, 4, None, 100, 16)  # BarStateSpace(2, 1, 4)
    assert m.num_states == 20
    assert m.first_states.tolist() == [[0, 1, 3, 6], [10, 11, 13, 16]]
    assert m.last_states.tolist() == [[0, 2, 5, 9], [10, 12, 15, 19]]
    assert np.allclose(m.positions[10:], np.asarray([0, 0, 0.5, 0, 1 / 3, 2 / 3, 0, 0.25, 0.5, 0.75]) + 1)
    # exponential_transition: exp(-lambda |to / from - 1|), values <= eps dropped, rows normalised
    m = _BarModel(1, 2, 4, None, 2.0, 16)
    raw = np.exp(-2.0 * np.abs(np.asarray([2, 3, 4])[None, :] / np.asarray([2, 3, 4])[:, None] - 1.0))
    assert np.allclose(np.exp(m.log_tempo), raw / raw.sum(1, keepdims=True))
    m = _BarModel(1, 14, 55, None, 100, 16)
    p = np.exp(m.log_tempo)
    assert np.allclose(p.sum(1), 1.0) and p[0, -1] == 0.0 and p[20, 20] == p[20].max()
    # observation pointers: the first 1/16 of every beat observes "beat", of the bar's first beat "downbeat"
    m = _BarModel(2, 16, 16, None, 100, 16)
    assert m.pointers.tolist() == [2] + [0] * 15 + [1] + [0] * 15
    # the reference's configuration
    trk = DBNDownBeatTracker()
    assert [mm.beats for mm in trk.models] == [3, 4]
    for mm in trk.models:
        assert mm.intervals.tolist() == list(range(14, 56)) and mm.num_states == mm.beats * 1449
    # num_tempi: log-spaced subset, as few intervals as requested
    assert len(_BarModel(4, 14, 55, 20, 100, 16).intervals) == 20


def test_native_dbn_tracks_synthetic_meters(lib_built):
    """4/4 at 120 BPM and 3/4 at 90 BPM impulse trains: beats on the impulses (after the `correct` step), bar
    positions counted 1..4 / 1..3, the right bar-length model wins, leading/trailing silence is trimmed, silence
    gives no beats; and Postprocessor(type='dbn') reaches it when madmom is not installed."""
    from beat_this_b200.dbn import DBNDownBeatTracker

    trk = DBNDownBeatTracker()
    assert [(m.beats, m.intervals[0], m.intervals[-1]) for m in trk.models] == [(3, 14, 55), (4, 14, 55)]
    T = 1000
    act = np.full((T, 2), 0.01)
    frames = list(range(110, 900, 25))
    for k, f in enumerate(frames):
        act[f, 1 if k % 4 == 0 else 0] = 0.9
    out = trk(act)
    assert np.array_equal(np.round(out[:, 0] * 50).astype(int), frames)
    assert np.array_equal(out[:, 1].astype(int), [k % 4 + 1 for k in range(len(frames))])
    act = np.full((T, 2), 0.01)
    frames = [int(round(7 + k * 100 / 3)) for k in range(29)]
    for k, f in enumerate(frames):
        act[f, 1 if k % 3 == 0 else 0] = 0.8
    out = trk(act)
    assert np.array_equal(np.round(out[:, 0] * 50).astype(int), frames)
    assert np.array_equal(out[:, 1].astype(int), [k % 3 + 1 for k in range(len(frames))])
    assert trk(np.full((200, 2), 0.001)).shape == (0, 2)


def test_native_dbn_cxx_tracker_equals_numpy_twin(lib_built):
    """bt_dbn_track (C++: model construction, Viterbi, peak correction, one thread per piece) against the numpy
    implementation of the same definition, on noisy pulse trains incl. silent / one-frame / frame-0-only pieces,
    and with log-spaced tempi (num_tempi smaller than the linear tempo grid)."""
    from beat_this_b200.dbn import DBNDownBeatTracker

    rng = np.random.default_rng(4)
    pieces = []
    for period, meter, T in ((23.7, 4, 900), (31.2, 3, 700), (17.0, 4, 400)):
        act = rng.uniform(0.001, 0.08, (T, 2))
        f, k = rng.uniform(0, period), 0
        while f < T:
            act[int(f)] = (0.05, 0.7) if k % meter == 0 else (0.75, 0.03)
            f += period * (1 + 0.02 * rng.standard_normal())
            k += 1
        pieces.append(act)
    only0 = np.full((50, 2), 0.001)
    only0[0, 0] = 0.9
    pieces += [np.full((120, 2), 0.001), np.full((1, 2), 0.4), only0]
    for kw in ({}, {"num_tempi": 20}, {"correct": False}):
        trk = DBNDownBeatTracker(**kw)
        got = trk.batch(pieces, n_threads=3)
        for act, g in zip(pieces, got):
            ref = trk.track_numpy(act)
            assert g.shape == ref.shape and np.array_equal(g, ref), kw
        assert np.array_equal(trk(pieces[0]), got[0])
    assert len(got[0]) > 20 and got[3].shape == (0, 2) and got[5].shape == (0, 2)
