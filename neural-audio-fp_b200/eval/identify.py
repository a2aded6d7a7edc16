"""``run.py identify``: which database track does a recording come from, and where in that track.

The recording (one WAV or a directory of them) is fingerprinted exactly as ``generate --source`` fingerprints those
files, each file (or each ``--window`` of it) is one clip, and the clip matcher (``nafp_clip_match``) scores every
offset-compensated candidate sequence of the database built from the memmaps ``generate`` wrote.  A match is a
global row of that database; the track map turns it into (key, WAV path, offset in seconds) through the file lists
``generate`` used, rebuilt from the WAV headers alone.
"""
from __future__ import annotations

import json
import os

import numpy as np

CLIP_MAXL = 4096          # segments per clip (nafp_clip_match)
MAX_TOP = 100


def check_limits(k_probe, top, window=None, hop=0.5, index_type='l2'):
    """The matcher's and the search's limits, checked before any data is loaded.  The search's own rules (k_probe
    per index type) are ``eval_search``'s, applied to a clip as to one sequence length."""
    from .eval_search import _check_limits
    if index_type.lower() not in ('l2', 'ivfpq', 'ivf', 'ivfpq-rr'):
        raise ValueError(f"-i {index_type}: identify searches an 'l2', 'ivfpq', 'ivf' or 'ivfpq-rr' index")
    _check_limits(index_type, [1], int(k_probe))
    if not 1 <= int(top) <= MAX_TOP:
        raise ValueError(f"--top {top}: the clip matcher keeps 1..{MAX_TOP} matches per clip")
    if window is not None:
        if window <= 0:
            raise ValueError(f"--window {window}: must be positive")
        if window_segments(window, hop) > CLIP_MAXL:
            raise ValueError(f"--window {window}: a clip holds at most {CLIP_MAXL} segments "
                             f"({CLIP_MAXL * hop:.0f} s at the {hop} s hop)")


def window_segments(window, hop):
    """Segments per ``--window`` of ``window`` seconds: one segment starts every ``hop`` seconds."""
    return max(1, int(round(float(window) / float(hop))))


def split_clips(file_first, window_seg=None):
    """Clips over the query rows: one per file, or consecutive non-overlapping runs of ``window_seg`` segments of
    every file (the last run of a file may be shorter).  Returns (clip_off (n_clips+1,) int64, file index per clip,
    first segment of every clip within its file)."""
    off, fidx, first = [0], [], []
    for fi in range(len(file_first) - 1):
        n = int(file_first[fi + 1] - file_first[fi])
        step = n if window_seg is None else int(window_seg)
        for s in range(0, n, step):
            e = min(n, s + step)
            off.append(off[-1] + e - s)
            fidx.append(fi)
            first.append(s)
    return np.asarray(off, np.int64), np.asarray(fidx, np.int64), np.asarray(first, np.int64)


class TrackMap:
    """Global database row -> (key, WAV path, offset in seconds).  ``parts`` are (key, SegmentSequence) in row order."""

    def __init__(self, parts, hop):
        self.hop = float(hop)
        self.keys, self.paths, firsts = [], [], []
        base = 0
        for key, seq in parts:
            self.keys += [key] * len(seq.filenames)
            self.paths += list(seq.filenames)
            firsts.append(seq.file_first[:-1] + base)
            base += int(seq.n_samples)
        self.file_first = np.concatenate(firsts + [[base]]).astype(np.int64)
        self.n_rows = base

    def locate(self, row):
        """(key, path, offset_s) of the file that holds ``row`` (the first row of a match)."""
        row = int(row)
        if not 0 <= row < self.n_rows:
            raise IndexError(f"row {row} outside the {self.n_rows}-row database")
        fi = int(np.searchsorted(self.file_first, row, side='right') - 1)
        return self.keys[fi], self.paths[fi], (row - int(self.file_first[fi])) * self.hop


def db_keys(source, skip_dummy):
    """Memmap keys in the row order of the database: [dummy_db; db] (``evaluate``), or custom_source."""
    if source:
        return ['custom_source']
    return ['db'] if skip_dummy else ['dummy_db', 'db']


def track_map(cfg, source, skip_dummy, emb_dir):
    """The track map of the database in ``emb_dir``, from the file lists ``generate`` used (WAV headers only).
    Refuses a list whose segment count is not the memmap's row count."""
    from ..model.generate import get_data_source
    from .eval_search import load_memmap_data
    ds = get_data_source(cfg, source, skip_dummy)
    parts = []
    for key in db_keys(source, skip_dummy):
        n_mm = int(load_memmap_data(emb_dir, key, shape_only=True)[0])
        if ds[key].n_samples != n_mm:
            raise ValueError(f"{emb_dir}{key}.mm holds {n_mm} rows but its source files give {ds[key].n_samples} "
                             f"segments: the database was generated from other files "
                             f"(check --source / --skip_dummy / the config)")
        parts.append((key, ds[key]))
    return TrackMap(parts, cfg['MODEL']['HOP'])


def query_sequence(cfg, query):
    """SegmentSequence of the query WAV(s): the files, in the order, that ``generate --source`` would read."""
    from ..model.dataset import Dataset
    dataset = Dataset(cfg)
    if os.path.isdir(query):
        seq = dataset.get_custom_db_ds(query)
    elif os.path.isfile(query):
        seq = dataset._seq([query])
    else:
        raise FileNotFoundError(query)
    if not seq.filenames:
        raise FileNotFoundError(f"no .wav file under {query}")
    return seq


def fingerprint_sequence(m_fp, seq, batches_per_call=64):
    """Fingerprints of every segment of ``seq``, by the calls ``generate`` makes (whole TS_BATCH_SZ groups)."""
    out = np.empty((seq.n_samples, 128), np.float32)
    for i in range(0, len(seq), batches_per_call):
        j = min(i + batches_per_call, len(seq))
        emb = m_fp.fingerprint_block(seq.get_source_block(i, j), group_size=seq.bsz)
        out[i * seq.bsz:i * seq.bsz + len(emb)] = emb
    return out


def build_index(emb_dir, keys, index_type, max_train=1e7, device=0):
    """``get_index`` over the memmaps, trained on the first part as ``eval_search`` trains it on dummy_db."""
    from .eval_search import load_memmap_data
    from .utils.get_index import get_index
    parts = [load_memmap_data(emb_dir, key)[0] for key in keys]
    index = get_index(index_type, parts[0], parts[0].shape, True, max_train, device=device)
    for key, part in zip(keys, parts):
        index.add(part)
        print(f'{len(part)} items from {key}')
    return index


def run_identify(cfg, checkpoint_name, checkpoint_index, query, emb_dir=None, source=None, skip_dummy=False,
                 index_type='l2', k_probe=20, top=10, window=None, output=None, device=0):
    """Returns one dict per clip: query path, start within it (s), number of segments and its top matches."""
    hop = float(cfg['MODEL']['HOP'])
    check_limits(k_probe, top, window, hop, index_type)
    seq = query_sequence(cfg, query)               # WAV headers only
    if seq.conversions():
        print(seq.conversions())
    window_seg = None if window is None else window_segments(window, hop)
    clip_off, clip_file, clip_first = split_clips(seq.file_first, window_seg)
    longest = int(np.diff(clip_off).max())
    if longest > CLIP_MAXL:
        raise ValueError(f"a query clip of {longest} segments is longer than {CLIP_MAXL} "
                         f"({CLIP_MAXL * hop:.0f} s): split it with --window")

    from ..model.fp import build_fp
    from ..model.generate import load_checkpoint
    _, m_fp = build_fp(cfg, device=device)
    checkpoint_index = load_checkpoint(cfg['DIR']['LOG_ROOT_DIR'] + 'checkpoint/', checkpoint_name, checkpoint_index,
                                       m_fp)
    if emb_dir is None:          # where generate wrote the database (the directory evaluate reads)
        emb_dir = cfg['DIR']['OUTPUT_ROOT_DIR'] + f'/{checkpoint_name}/{checkpoint_index}/'
    emb_dir = emb_dir if emb_dir.endswith('/') else emb_dir + '/'
    tmap = track_map(cfg, source, skip_dummy, emb_dir)
    rows = fingerprint_sequence(m_fp, seq)
    print(f'{len(seq.filenames)} query file(s), {len(rows)} segments, {len(clip_off) - 1} clip(s)')

    index = build_index(emb_dir, db_keys(source, skip_dummy), index_type, device=device)
    pred, scores = index.clip_match(rows, clip_off, k_probe=k_probe, n_top=top)

    results = []
    for ci in range(len(clip_off) - 1):
        matches = []
        for r in range(top):
            if pred[ci, r] < 0:
                break
            key, path, offset_s = tmap.locate(pred[ci, r])
            matches.append(dict(rank=r + 1, key=key, file=path, offset_s=offset_s, score=float(scores[ci, r]),
                                row=int(pred[ci, r])))
        clip = dict(query=seq.filenames[clip_file[ci]], start_s=float(clip_first[ci] * hop),
                    segments=int(clip_off[ci + 1] - clip_off[ci]), matches=matches)
        results.append(clip)
        print(f"{clip['query']} @ {clip['start_s']:.1f} s ({clip['segments']} segments)")
        for m in matches:
            print(f"  {m['rank']:>3}  {m['file']}  {m['offset_s']:.1f} s  {m['score']:.4f}")
    if output:
        with open(output, 'w') as f:
            json.dump(results, f, indent=1)
        print(f'Wrote {output}')
    return results
