"""CPU: the resampling contract (oracle/resample.py against scipy.signal.resample_poly), and the segmenter's handling
of WAVs at any rate and channel count: segment counts from the resampled length, run windows, limits."""
import wave

import numpy as np
import pytest
import scipy.signal

from nafp_b200 import synth
from nafp_b200.model import dataset as D
from oracle import resample as R

RATES = [4000, 11025, 16000, 22050, 32000, 44100, 48000, 96000, 192000]


@pytest.mark.parametrize("fs_in", RATES)
def test_oracle_agrees_with_resample_poly(fs_in):
    up, down, hl = R.ratio(fs_in, 8000)
    np.testing.assert_allclose(R.filter_taps(fs_in, 8000),
                               scipy.signal.firwin(2 * hl + 1, 1.0 / max(up, down), window=('kaiser', 5.0)) * up,
                               rtol=0, atol=1e-15)
    rng = np.random.default_rng(fs_in)
    for n in (0, 1, 7, hl - 1, 100000):
        x = rng.integers(-32768, 32768, (n, 2)).astype(np.int16)
        y = R.resample_exact(x, fs_in, 8000)
        ref = scipy.signal.resample_poly(x.astype(np.float64).mean(axis=1), up, down)
        assert len(y) == len(ref) == R.out_length(n, fs_in, 8000) == D.resampled_length(n, fs_in, 8000)
        if n:
            assert np.abs(y - ref).max() <= 1e-9, (fs_in, n)
        # any output range is the matching slice of the whole track
        if n > 10:
            m0, k = len(y) // 3, len(y) // 3
            np.testing.assert_array_equal(R.resample_exact(x, fs_in, 8000, m0, k), y[m0:m0 + k])


def test_equal_rates_are_a_copy_or_a_rounded_mean():
    x = np.array([[1, 2], [3, 4], [-5, -6], [7, 8], [32767, 32767]], np.int16)
    np.testing.assert_array_equal(R.resample_pcm16(x[:, 0], 8000, 8000)[0], x[:, 0])
    np.testing.assert_array_equal(R.resample_pcm16(x, 8000, 8000)[0], [2, 4, -6, 8, 32767])   # half to even


def _wav(path, x, fs):
    synth.write_wav(str(path), x, fs)
    return str(path)


def _corpus(tmp_path):
    rng = np.random.default_rng(3)
    return [_wav(tmp_path / "a.wav", rng.integers(-9000, 9000, (441000, 2)).astype(np.int16), 44100),   # 10 s stereo
            _wav(tmp_path / "b.wav", rng.integers(-9000, 9000, 66150).astype(np.int16), 22050),         # 3 s mono
            _wav(tmp_path / "c.wav", synth.synth_track(4, 52000), 8000),                                 # 6.5 s
            _wav(tmp_path / "d.wav", rng.integers(-9000, 9000, (3000, 6)).astype(np.int16), 48000)]     # < 1 segment


def test_segment_counts_follow_the_resampled_length(tmp_path):
    files = _corpus(tmp_path)
    seq = D.SegmentSequence(files, bsz=7, resample=True)
    assert seq.file_len == [80000, 24000, 52000, 500]
    assert seq.file_nseg == [D.n_segments(n) for n in seq.file_len] == [19, 5, 12, 1]
    assert seq.n_samples == 37
    assert seq.native == [False, False, True, False]
    assert "44100 Hz 2 ch" in seq.conversions() and "22050 Hz mono" in seq.conversions()
    assert D.SegmentSequence(files[2:3], resample=True).conversions() is None


def _expected_window(m0, n_out, n, fs_in):
    up, down, hl = R.ratio(fs_in, 8000)
    lo = max(0, int(np.ceil((m0 * down - hl) / up)))
    hi = min(n - 1, int(np.floor(((m0 + n_out - 1) * down + hl) / up)))
    return lo, hi - lo + 1


@pytest.mark.parametrize("bsz,bpc", [(7, 1), (7, 3), (25, 2), (200, 1)])
def test_run_windows_cover_exactly_what_the_formula_needs(tmp_path, bsz, bpc):
    files = _corpus(tmp_path)
    seq = D.SegmentSequence(files, bsz=bsz, resample=True)
    raw = [seq._file_pcm(fi).copy() for fi in range(len(files))]
    seen = [[] for _ in files]
    for b in range(0, len(seq), bpc):
        pcm, off, valid, runs = seq.get_source_block(b, min(b + bpc, len(seq)))
        if runs is None:                  # a block of c.wav alone: the 8 kHz mono path
            assert {fi for fi, _, _ in seq._block_files(b, min(b + bpc, len(seq)))} == {2}
            runs = np.array([[0, 0, len(pcm), 1, 8000, -1, len(pcm)]], np.int64)
            m0 = int(np.floor(seq._block_files(b, min(b + bpc, len(seq)))[0][1] * 0.5 * 8000))
            runs[0, 1] = runs[0, 5] = m0
        assert runs.shape[1] == 7 and runs.dtype == np.int64
        assert len(off) == len(valid) == min((b + bpc) * bsz, seq.n_samples) - b * bsz
        base = 0
        for pos, f0, cnt, ch, rate, m0, n_out in runs:
            fi = [i for i in range(len(files)) if seq.file_info[i][0] == rate and seq.file_info[i][1] == ch][0]
            n = seq.file_info[fi][2]
            want = _expected_window(m0, n_out, n, rate) if rate != 8000 else (m0, n_out)
            assert (f0, cnt) == want, (fi, m0, n_out)
            np.testing.assert_array_equal(pcm[pos:pos + cnt * ch], raw[fi][f0 * ch:(f0 + cnt) * ch])
            seen[fi].append((m0, n_out, base))
            base += n_out
        assert int(runs[:, 6].sum()) == base
        assert (off >= 0).all() and (off + valid <= base).all()
    # every segment of every file lies inside the runs of its blocks
    for fi, runs_fi in enumerate(seen):
        m_lo = min(m0 for m0, _, _ in runs_fi)
        m_hi = max(m0 + n for m0, n, _ in runs_fi)
        assert m_lo == 0 and m_hi == seq.file_len[fi]


def test_native_block_is_the_track_block(tmp_path):
    files = [_wav(tmp_path / f"n{i}.wav", synth.synth_track(i, 30000 + 7000 * i), 8000) for i in range(3)]
    seq = D.SegmentSequence(files, bsz=5, resample=True)
    assert seq.conversions() is None and seq.file_len == [30000, 37000, 44000]
    for b in range(0, len(seq), 2):
        pcm, off, valid, runs = seq.get_source_block(b, min(b + 2, len(seq)))
        ref = seq.get_track_block(b, min(b + 2, len(seq)))
        assert runs is None
        for got, want in zip((pcm, off, valid), ref):
            assert got.dtype == want.dtype and np.array_equal(got, want)


def test_resampled_files_refuse_the_host_segment_paths(tmp_path):
    seq = D.SegmentSequence(_corpus(tmp_path)[:1], bsz=4, resample=True)
    with pytest.raises(NotImplementedError, match="resampled on the GPU"):
        seq.get_track_block(0, 1)
    with pytest.raises(NotImplementedError, match="resampled on the GPU"):
        seq.get_pcm(0)


def _raw_wav(path, rate, channels, width, n=100):
    with wave.open(str(path), "w") as w:
        w.setnchannels(channels)
        w.setsampwidth(width)
        w.setframerate(rate)
        w.writeframes(b"\0" * (n * channels * width))
    return str(path)


def test_limits_raise_with_their_messages(tmp_path):
    with pytest.raises(ValueError, match=r"44056 Hz -> 8000 Hz needs up 1000 / down 5507"):
        D.SegmentSequence([_raw_wav(tmp_path / "r.wav", 44056, 1, 2)], resample=True)
    with pytest.raises(ValueError, match="9 channels; 1..8 are supported"):
        D.SegmentSequence([_raw_wav(tmp_path / "c.wav", 8000, 9, 2)], resample=True)
    with pytest.raises(NotImplementedError, match="24-bit samples; only 16-bit PCM"):
        D.SegmentSequence([_raw_wav(tmp_path / "w.wav", 44100, 2, 3)], resample=True)
    assert D._wav_info(_raw_wav(tmp_path / "ok.wav", 192000, 8, 2), 8000, resample=True) == (192000, 8, 100)
    assert D.resample_ratio(44100, 8000) == (80, 441, 4410)
    assert D.resample_ratio(8000, 8000) == (1, 1, 0)


def test_without_resample_only_the_reference_format_is_read(tmp_path):
    """The default keeps the reference reader's contract; Dataset (generate / identify) reads with resample=True."""
    files = _corpus(tmp_path)
    with pytest.raises(ValueError, match="Sample rate should be 8000 but got 44100"):
        D.SegmentSequence(files[:1])
    with pytest.raises(NotImplementedError, match="only 16-bit mono PCM"):
        D.SegmentSequence([_wav(tmp_path / "st.wav", np.zeros((100, 2), np.int16), 8000)])
    assert D.SegmentSequence(files[2:3]).file_len == [52000]
    cfg = {'DIR': {'SOURCE_ROOT_DIR': str(tmp_path)}, 'DATA_SEL': {'TEST_DUMMY_DB': '10k_full', 'TEST_QUERY_DB': 'unseen_icassp'},
           'BSZ': {'TS_BATCH_SZ': 7}, 'MODEL': {'DUR': 1.0, 'HOP': 0.5, 'FS': 8000}}
    seq = D.Dataset(cfg).get_custom_db_ds(str(tmp_path))
    assert [p.rsplit('/', 1)[1] for p in seq.filenames] == ["a.wav", "b.wav", "c.wav", "d.wav", "st.wav"]
    assert seq.file_len == [80000, 24000, 52000, 500, 100]
