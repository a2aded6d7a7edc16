"""Host-side segmenter for fingerprint generation (SURVEY §8 a0).

Mirrors the no-augmentation data path of the reference: ``Dataset.get_test_dummy_db_ds`` /
``get_test_query_db_ds`` / ``get_custom_db_ds`` (``model/dataset.py:182-323``) build a
``genUnbalSequence(bsz == n_anchor == TS_BATCH_SZ, shuffle=False, drop_the_last_non_full_batch=False)``
whose batches are consecutive runs of TS_BATCH_SZ one-second segments (0.5 s hop) across file
boundaries (``model/utils/dataloader_keras.py:132-141,186-193,223-228``); segment enumeration and
loading follow ``model/utils/audio_utils.py:140-264``.

Differences by design (results identical): every WAV file is read ONCE (the reference re-opens the
file for each segment), the segments of a file are cut with one strided copy (``get_pcm_range``: the
per-segment Python loop was 4x slower than the GPU that consumes its output), and batches can be handed
over as int16 PCM so that the ``/ 2**15`` scaling (``audio_utils.py:243-244``) happens on the GPU.

Beyond the reference (which refuses them, ``audio_utils.py:176-181``): 16-bit WAVs at any rate with 1..8 channels.
Segment counts and offsets are those of the file resampled to ``fs`` (``resampled_length``), so they follow from the
header alone; the samples are downmixed and resampled on the GPU (``nafp_fingerprint_pcm16_sources_host``).
"""
from __future__ import annotations

import glob
import math
import wave

import numpy as np


def n_segments(n_frames, fs=8000, duration=1.0, hop=0.5):
    """``audio_utils.py:173-177``."""
    seg, hp = fs * duration, fs * hop
    if n_frames > seg:
        return int((n_frames - seg + hp) // hp)
    return 1


MAX_RATIO = 1024           # NAFP_RESAMPLE_MAX_RATIO: max(up, down) of a supported rate pair
MAX_CHANNELS = 8           # NAFP_RESAMPLE_MAX_CHANNELS


def resample_ratio(fs_in, fs_out):
    """(up, down, hl) of the polyphase resampler from ``fs_in`` to ``fs_out``: up / down in lowest terms and the
    half length of its filter (0 for equal rates, a copy).  Raises ValueError beyond max(up, down) = MAX_RATIO."""
    fs_in, fs_out = int(fs_in), int(fs_out)
    if fs_in <= 0 or fs_out <= 0:
        raise ValueError(f'sample rate {fs_in} Hz: must be positive')
    g = math.gcd(fs_in, fs_out)
    up, down = fs_out // g, fs_in // g
    if max(up, down) > MAX_RATIO:
        raise ValueError(f'{fs_in} Hz -> {fs_out} Hz needs up {up} / down {down}; rates with max(up, down) <= '
                         f'{MAX_RATIO} are supported (every common rate is)')
    return up, down, (0 if up == down else 10 * max(up, down))


def resampled_length(n_frames, fs_in, fs_out):
    """ceil(n_frames * up / down): the length ``scipy.signal.resample_poly`` gives."""
    up, down, _ = resample_ratio(fs_in, fs_out)
    return -(-int(n_frames) * up // down)


def source_window(m0, n_out, n_frames, fs_in, fs_out):
    """(frame0, count): the source frames that outputs m0 .. m0 + n_out - 1 read,
    ceil((m0 down - hl) / up) .. floor(((m0 + n_out - 1) down + hl) / up), clamped to [0, n_frames)."""
    up, down, hl = resample_ratio(fs_in, fs_out)
    lo = max(0, -(-(m0 * down - hl) // up))
    hi = min(int(n_frames) - 1, ((m0 + n_out - 1) * down + hl) // up)
    return (lo, hi - lo + 1) if n_out > 0 and hi >= lo else (0, 0)


def _wav_info(path, fs, resample=False):
    """(rate, channels, frames) of a WAV.  Without ``resample`` only what the reference's reader takes: ``fs`` 16-bit
    mono.  With it, 16-bit PCM with 1..MAX_CHANNELS channels at a rate that resamples to ``fs`` (``resample_ratio``)."""
    with wave.open(path, 'r') as w:
        rate, ch, width, n = w.getframerate(), w.getnchannels(), w.getsampwidth(), w.getnframes()
    if not resample:
        if rate != fs:
            raise ValueError('Sample rate should be {} but got {}'.format(str(fs), str(rate)))
        if width != 2 or ch != 1:
            raise NotImplementedError(f'{path}: only 16-bit mono PCM is supported (like the reference reader)')
        return rate, ch, n
    if width != 2:
        raise NotImplementedError(f'{path}: {8 * width}-bit samples; only 16-bit PCM is supported')
    if not 1 <= ch <= MAX_CHANNELS:
        raise ValueError(f'{path}: {ch} channels; 1..{MAX_CHANNELS} are supported')
    try:
        resample_ratio(rate, fs)
    except ValueError as e:
        raise ValueError(f'{path}: {e}') from None
    return rate, ch, n


class SegmentSequence:
    """Indexable sequence of batches, the role ``genUnbalSequence`` plays in ``generate.py:170-181``.

    By default the files must be what the reference's reader accepts (``fs`` 16-bit mono; anything else raises as
    ``audio_utils.py:176-181`` does).  ``resample=True`` accepts any rate and 1..MAX_CHANNELS channels, which the GPU
    resamples to ``fs`` mono (``get_source_block``); ``Dataset``, and so ``generate`` and ``identify``, read that way."""

    def __init__(self, filenames, bsz=125, duration=1.0, hop=0.5, fs=8000, resample=False):
        self.filenames = list(filenames)
        self.bsz = int(bsz)
        self.fs, self.duration, self.hop = int(fs), float(duration), float(hop)
        self.seg_len = int(self.duration * self.fs)
        # (file index, seg_idx) for every segment, in file order -- fns_event_seg_list
        self.file_info = [_wav_info(fn, self.fs, resample) for fn in self.filenames]  # (rate, channels, frames)
        self.native = [rate == self.fs and ch == 1 for rate, ch, _ in self.file_info]
        self.file_len = [resampled_length(n, rate, self.fs) for rate, _, n in self.file_info]   # samples at fs
        self.file_nseg = [n_segments(n, self.fs, self.duration, self.hop) for n in self.file_len]
        self.file_first = np.concatenate([[0], np.cumsum(self.file_nseg)]).astype(np.int64)
        self.n_samples = int(self.file_first[-1])
        self._cache_idx = -1
        self._cache_pcm = None

    def __len__(self):
        return int(np.ceil(self.n_samples / float(self.bsz)))

    def conversions(self):
        """One line naming the source formats that are resampled on the GPU, or None when every file is at fs mono."""
        counts = {}
        for (rate, ch, _), nat in zip(self.file_info, self.native):
            if not nat:
                counts[(rate, ch)] = counts.get((rate, ch), 0) + 1
        if not counts:
            return None
        parts = [f'{n} at {rate} Hz {"mono" if ch == 1 else f"{ch} ch"}' for (rate, ch), n in sorted(counts.items())]
        return f'Resampling to {self.fs} Hz mono on the GPU: ' + ', '.join(parts) + ' file(s)'

    def _file_pcm(self, fi):
        """The file's samples, interleaved int16 (frames x channels)."""
        if fi != self._cache_idx:
            with wave.open(self.filenames[fi], 'r') as w:
                raw = w.readframes(w.getnframes())
            self._cache_pcm = np.frombuffer(raw, dtype=np.int16)
            self._cache_idx = fi
        return self._cache_pcm

    def _native_pcm(self, fi):
        if not self.native[fi]:
            raise NotImplementedError(f'{self.filenames[fi]} is resampled on the GPU: fingerprint it through '
                                      f'get_source_block')
        return self._file_pcm(fi)

    def _segment_pcm(self, fi, seg_idx, out):
        pcm = self._native_pcm(fi)
        start = int(np.floor(seg_idx * self.hop * self.fs))
        x = pcm[start:start + self.seg_len]
        out[:len(x)] = x
        out[len(x):] = 0

    def get_pcm(self, idx):
        """Batch ``idx`` as int16 (n, seg_len); n == bsz except for the last batch."""
        lo, hi = idx * self.bsz, min((idx + 1) * self.bsz, self.n_samples)
        if lo >= hi:
            raise IndexError(idx)
        out = np.empty((hi - lo, self.seg_len), dtype=np.int16)
        fi = int(np.searchsorted(self.file_first, lo, side='right') - 1)
        for r, g in enumerate(range(lo, hi)):
            while g >= self.file_first[fi + 1]:
                fi += 1
            self._segment_pcm(fi, g - int(self.file_first[fi]), out[r])
        return out

    def get_pcm_range(self, b_lo, b_hi):
        """Batches ``b_lo .. b_hi-1`` as one int16 array (n, seg_len) -- the same rows as the concatenation of
        ``get_pcm(b)``, cut file by file: the segments s0..s1 of a file are rows of a strided view of its samples
        (start = floor(s * hop * fs), ``audio_utils.py:246-247``), copied in one assignment."""
        lo, hi = b_lo * self.bsz, min(b_hi * self.bsz, self.n_samples)
        if lo >= hi:
            raise IndexError((b_lo, b_hi))
        out = np.empty((hi - lo, self.seg_len), dtype=np.int16)
        fi = int(np.searchsorted(self.file_first, lo, side='right') - 1)
        g = lo
        while g < hi:
            while g >= self.file_first[fi + 1]:
                fi += 1
            s0 = g - int(self.file_first[fi])
            s1 = min(int(self.file_nseg[fi]), s0 + (hi - g))
            pcm = self._native_pcm(fi)
            starts = np.floor(np.arange(s0, s1) * self.hop * self.fs).astype(np.int64)
            need = int(starts[-1]) + self.seg_len
            if len(pcm) < need:                       # a file shorter than one segment: zero padded (audio_utils.py:249-252)
                pcm = np.concatenate([pcm, np.zeros(need - len(pcm), np.int16)])
            win = np.lib.stride_tricks.sliding_window_view(pcm, self.seg_len)
            out[g - lo:g - lo + (s1 - s0)] = win[starts]
            g += s1 - s0
        return out

    def _block_files(self, b_lo, b_hi):
        """(file index, first segment, end segment) of every file that batches ``b_lo .. b_hi-1`` touch, in order."""
        lo, hi = b_lo * self.bsz, min(b_hi * self.bsz, self.n_samples)
        if lo >= hi:
            raise IndexError((b_lo, b_hi))
        out = []
        fi = int(np.searchsorted(self.file_first, lo, side='right') - 1)
        g = lo
        while g < hi:
            while g >= self.file_first[fi + 1]:
                fi += 1
            s0 = g - int(self.file_first[fi])
            s1 = min(int(self.file_nseg[fi]), s0 + (hi - g))
            out.append((fi, s0, s1))
            g += s1 - s0
        return out

    def _windows(self, fi, s0, s1, base):
        """Segments s0 .. s1-1 of file fi as windows of its run of fs samples: (first, last) of the run, the
        segments' offsets (run placed at ``base``) and valid lengths."""
        n = self.file_len[fi]
        starts = np.floor(np.arange(s0, s1) * self.hop * self.fs).astype(np.int64)
        first, last = int(starts[0]), min(int(starts[-1]) + self.seg_len, n)
        return first, last, starts - first + base, np.minimum(self.seg_len, n - starts).astype(np.int32)

    def get_track_block(self, b_lo, b_hi):
        """Batches ``b_lo .. b_hi-1`` WITHOUT cutting the segments: (pcm, seg_off, seg_valid) -- the sample runs of
        the files the batches touch, back to back (int16), and for every segment its start offset in ``pcm`` (int64)
        and its number of real samples (int32, < seg_len only for a file shorter than one segment).  The GPU cuts
        the overlapping windows (``nafp_fingerprint_pcm16_tracks_host``): every sample is uploaded once.  Every file
        must be at fs mono (``get_source_block`` takes any)."""
        runs, offs, valid = [], [], []
        base = 0
        for fi, s0, s1 in self._block_files(b_lo, b_hi):
            pcm = self._native_pcm(fi)
            first, last, off, val = self._windows(fi, s0, s1, base)
            runs.append(pcm[first:last])
            offs.append(off)
            valid.append(val)
            base += last - first
        return np.concatenate(runs), np.concatenate(offs), np.concatenate(valid)

    def get_source_block(self, b_lo, b_hi):
        """Batches ``b_lo .. b_hi-1`` for any source format: (pcm, seg_off, seg_valid, runs).  When every file the
        batches touch is at fs mono, the first three are ``get_track_block``'s and runs is None.  Otherwise pcm holds,
        back to back, the interleaved source frames each file's run of fs samples reads (``source_window``), runs is
        (n_runs, 7) int64 (offset in pcm, frame0, n_frames, channels, rate, m0, n_out) -- the run is outputs
        m0 .. m0+n_out-1 of the resampled file -- and seg_off / seg_valid index the runs' outputs placed back to back
        (``nafp_fingerprint_pcm16_sources_host``)."""
        files = self._block_files(b_lo, b_hi)
        if all(self.native[fi] for fi, _, _ in files):
            return (*self.get_track_block(b_lo, b_hi), None)
        src, runs, offs, valid = [], [], [], []
        base = pos = 0
        for fi, s0, s1 in files:
            rate, ch, n_frames = self.file_info[fi]
            first, last, off, val = self._windows(fi, s0, s1, base)
            f0, cnt = source_window(first, last - first, n_frames, rate, self.fs)
            src.append(self._file_pcm(fi)[f0 * ch:(f0 + cnt) * ch])
            runs.append((pos, f0, cnt, ch, rate, first, last - first))
            offs.append(off)
            valid.append(val)
            pos += cnt * ch
            base += last - first
        return np.concatenate(src), np.concatenate(offs), np.concatenate(valid), np.asarray(runs, np.int64)

    def __getitem__(self, idx):
        """(Xa, Xp) like the reference generator: Xa float32 (n, 1, T), Xp empty."""
        xa = (self.get_pcm(idx) / 2 ** 15).astype(np.float32)[:, None, :]
        return xa, np.zeros((0, 1, self.seg_len), dtype=np.float32)


class Dataset:
    """File selection of ``model/dataset.py:35-323`` for the generation splits."""

    def __init__(self, cfg):
        self.source_root_dir = cfg['DIR']['SOURCE_ROOT_DIR']
        self.datasel_test_dummy_db = cfg['DATA_SEL']['TEST_DUMMY_DB']
        self.datasel_test_query_db = cfg['DATA_SEL']['TEST_QUERY_DB']
        self.ts_batch_sz = cfg['BSZ']['TS_BATCH_SZ']
        self.dur = cfg['MODEL']['DUR']
        self.hop = cfg['MODEL']['HOP']
        self.fs = cfg['MODEL']['FS']

    def _seq(self, fps):
        return SegmentSequence(fps, self.ts_batch_sz, self.dur, self.hop, self.fs, resample=True)

    def get_test_dummy_db_ds(self):
        fps = sorted(glob.glob(self.source_root_dir + 'test-dummy-db-100k-full/' + '**/*.wav', recursive=True))
        sel = str(self.datasel_test_dummy_db)
        if sel in ['10k_full', '10k_30s']:
            fps = fps[:10000]
        elif sel == '100k_full_icassp':
            pass
        elif sel.isnumeric():
            fps = fps[:int(sel)]
        else:
            raise NotImplementedError(sel)
        return self._seq(fps)

    def get_test_query_db_ds(self):
        if self.datasel_test_query_db == 'unseen_icassp':
            q = sorted(glob.glob(self.source_root_dir + 'test-query-db-500-30s/' + 'query/**/*.wav', recursive=True))
            d = sorted(glob.glob(self.source_root_dir + 'test-query-db-500-30s/' + 'db/**/*.wav', recursive=True))
            return self._seq(q), self._seq(d)
        if self.datasel_test_query_db == 'unseen_syn':
            raise NotImplementedError("'unseen_syn' synthesises queries with the training-time augmentation "
                                      "chain, which is outside the inference hot path")
        raise NotImplementedError(self.datasel_test_query_db)

    def get_custom_db_ds(self, source_root_dir):
        fps = sorted(glob.glob(source_root_dir + '/**/*.wav', recursive=True))
        return self._seq(fps)
