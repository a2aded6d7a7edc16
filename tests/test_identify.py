"""`run.py identify` without a GPU: the track map, --window splitting, the command's help and its up-front limits."""
import os
import subprocess
import sys

import numpy as np
import pytest
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _wav(path, seconds, seed=0):
    from nafp_b200 import synth
    os.makedirs(os.path.dirname(path), exist_ok=True)
    synth.write_wav(path, synth.synth_track(seed, int(seconds * 8000)))


@pytest.fixture()
def corpus(tmp_path):
    """dummy: 2 files (12 s, 5 s); db: 3 files (10 s, 30 s, 3 s); a custom source of 2 files."""
    src = tmp_path / "music"
    for i, s in enumerate((12, 5)):
        _wav(str(src / f"test-dummy-db-100k-full/a/d{i:03d}.wav"), s, i)
    for i, s in enumerate((10, 30, 3)):
        _wav(str(src / f"test-query-db-500-30s/db/a/s{i:03d}.wav"), s, 10 + i)
        _wav(str(src / f"test-query-db-500-30s/query/a/s{i:03d}.wav"), s, 20 + i)
    for i, s in enumerate((7, 4)):
        _wav(str(tmp_path / f"custom/x{i}.wav"), s, 30 + i)
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "default.yaml")))
    cfg['DIR']['SOURCE_ROOT_DIR'] = str(src) + "/"
    cfg['DATA_SEL']['TEST_DUMMY_DB'] = '100k_full_icassp'
    return cfg, tmp_path


def _memmap_shapes(emb_dir, rows):
    os.makedirs(emb_dir, exist_ok=True)
    for key, n in rows.items():
        np.save(os.path.join(emb_dir, f"{key}_shape.npy"), np.array([n, 128]))


def test_track_map_dummy_then_db(corpus):
    from nafp_b200.eval.identify import track_map
    cfg, tmp = corpus
    emb = str(tmp / "emb") + "/"
    # segments: 12 s -> 23, 5 s -> 9; 10 s -> 19, 30 s -> 59, 3 s -> 5
    _memmap_shapes(emb, {"dummy_db": 32, "db": 83})
    tm = track_map(cfg, None, False, emb)
    assert tm.n_rows == 115
    assert tm.file_first.tolist() == [0, 23, 32, 51, 110, 115]
    key, path, off = tm.locate(0)
    assert key == "dummy_db" and path.endswith("d000.wav") and off == 0.0
    key, path, off = tm.locate(31)
    assert key == "dummy_db" and path.endswith("d001.wav") and off == 4.0
    key, path, off = tm.locate(32 + 19 + 40)          # row 40 of the 30 s db file
    assert key == "db" and path.endswith("s001.wav") and off == 20.0
    assert tm.locate(114)[1].endswith("s002.wav")
    with pytest.raises(IndexError):
        tm.locate(115)
    # --skip_dummy: the rows are db alone
    tm = track_map(cfg, None, True, emb)
    assert tm.n_rows == 83 and tm.locate(19)[1].endswith("s001.wav") and tm.locate(19)[2] == 0.0


def test_track_map_custom_source(corpus):
    from nafp_b200.eval.identify import track_map
    cfg, tmp = corpus
    emb = str(tmp / "emb_custom") + "/"
    _memmap_shapes(emb, {"custom_source": 13 + 7})     # 7 s -> 13, 4 s -> 7
    tm = track_map(cfg, str(tmp / "custom"), False, emb)
    assert tm.n_rows == 20
    key, path, off = tm.locate(15)
    assert key == "custom_source" and path.endswith("x1.wav") and off == 1.0


def test_track_map_refuses_a_row_count_mismatch(corpus):
    from nafp_b200.eval.identify import track_map
    cfg, tmp = corpus
    emb = str(tmp / "emb_bad") + "/"
    _memmap_shapes(emb, {"dummy_db": 32, "db": 84})
    with pytest.raises(ValueError, match="84 rows but its source files give 83 segments"):
        track_map(cfg, None, False, emb)


def test_window_splitting():
    from nafp_b200.eval.identify import split_clips, window_segments
    file_first = np.array([0, 59, 68, 168])            # files of 59, 9 and 100 segments
    off, fidx, first = split_clips(file_first)
    assert off.tolist() == [0, 59, 68, 168] and fidx.tolist() == [0, 1, 2] and first.tolist() == [0, 0, 0]
    w = window_segments(10.0, 0.5)
    assert w == 20
    off, fidx, first = split_clips(file_first, w)
    assert np.diff(off).tolist() == [20, 20, 19, 9, 20, 20, 20, 20, 20]
    assert fidx.tolist() == [0, 0, 0, 1, 2, 2, 2, 2, 2]
    assert first.tolist() == [0, 20, 40, 0, 0, 20, 40, 60, 80]
    assert off[-1] == 168
    assert window_segments(0.2, 0.5) == 1


def test_identify_help():
    r = subprocess.run([sys.executable, "-m", "nafp_b200.run", "identify", "--help"], cwd=ROOT, capture_output=True,
                       text=True, env=dict(os.environ, PYTHONPATH=ROOT))
    assert r.returncode == 0, r.stderr
    for opt in ("--query", "--emb_dir", "--source", "--skip_dummy", "--index_type", "--k_probe", "--top", "--window",
                "--output"):
        assert opt in r.stdout


@pytest.mark.parametrize("args, msg", [
    (["-k", "129"], "--k_probe 129"),
    (["-k", "0"], "--k_probe 0"),
    (["-i", "ivfpq", "-k", "103"], "nprobe x k_probe <= 4096"),
    (["--top", "101"], "--top 101"),
    (["--window", "2048.5"], "--window 2048.5"),
    (["-i", "ivfpq-rr", "-k", "33"], "ivfpq-rr"),
    (["-i", "hnsw"], "-i hnsw"),
])
def test_identify_limits_are_checked_up_front(args, msg, tmp_path):
    """The limits surface before any file is read: the query and the database here do not exist."""
    from click.testing import CliRunner
    from nafp_b200.run import cli
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "default.yaml")))
    cfg_path = str(tmp_path / "cfg.yaml")
    with open(cfg_path, "w") as f:
        yaml.safe_dump(cfg, f)
    r = CliRunner().invoke(cli, ["identify", "random-init:7", "-c", cfg_path, "--query", str(tmp_path / "missing.wav"),
                                 "--emb_dir", str(tmp_path / "missing")] + args)
    assert isinstance(r.exception, ValueError), r.output
    assert msg in str(r.exception)


def test_a_clip_longer_than_the_matcher_is_refused_before_loading(corpus):
    from nafp_b200.eval.identify import run_identify
    cfg, tmp = corpus
    long_wav = str(tmp / "long" / "rec.wav")
    os.makedirs(os.path.dirname(long_wav))
    from nafp_b200 import synth
    synth.write_wav(long_wav, np.zeros(2049 * 8000, np.int16))        # 4097 segments
    with pytest.raises(ValueError, match="4097 segments"):
        run_identify(cfg, "random-init:7", None, long_wav, emb_dir=str(tmp / "missing"))
