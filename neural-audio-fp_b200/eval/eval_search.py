"""Search + evaluation CLI: the reference's ``eval/eval_faiss.py`` over libnafp.

Same arguments and options (``eval_faiss.py:65-92``), same outputs (``raw_score.npy``,
``test_ids.npy``, the final hit-rate table).  What changes is how the hot loop (``:204-243``) runs:
the per-(test id, length) Python loop around ``index.search`` + numpy re-scoring becomes one
batched call per ``display_interval`` block of test ids (segment search for the longest length
serves every shorter one; offset compensation, unique candidates, sequence scores and top-10 are
CUDA kernels).  Deliberate deviations, both listed in DESIGN.md: ``dummy_db.mm`` is NOT extended on
disk (the reference's ``fake_recon_index``, ``:167-171``; the device index already holds [dummy; db]),
and ``--nogpu`` is refused (there is no CPU search path).

Multi-GPU: started under ``torchrun`` (WORLD_SIZE > 1) the database is row-sharded over the ranks
(``nafp_b200.dist.ShardedFlatIndex``: every rank reads only its block of the memmaps; per-rank top-k merged by an
NCCL all-gather, candidate scores by a max all-reduce; 'ivfpq-rr' merges its first level and its re-ranked top-k in
two such exchanges); rank 0 prints the table and writes the outputs.
"""
from __future__ import annotations

import glob
import os
import time

import click
import numpy as np

from .utils.get_index import get_index
from .utils.print_table import PrintTable


def load_memmap_data(source_dir, fname, append_extra_length=None, shape_only=False, display=True):
    """``eval_faiss.py:18-62``.  ``append_extra_length`` is accepted for signature parity but files
    are never opened for writing here."""
    path_shape = source_dir + fname + '_shape.npy'
    path_data = source_dir + fname + '.mm'
    data_shape = np.load(path_shape)
    if shape_only:
        return data_shape
    data = np.memmap(path_data, dtype='float32', mode='r', shape=(data_shape[0], data_shape[1]))
    if display:
        print(f'Load {data_shape[0]:,} items from \033[32m{path_data}\033[0m.')
    return data, data_shape


def hit_flags(pred_ids, gt_id):
    """``eval_faiss.py:236-243`` for one (test id, length); pred_ids is -1 padded."""
    p = pred_ids[pred_ids >= 0]
    if len(p) == 0:
        return 0, 0, 0, 0
    return (int(gt_id == p[0]), int(p[0] in [gt_id - 1, gt_id, gt_id + 1]),
            int(gt_id in p[:3]), int(gt_id in p[:10]))


def select_test_ids(test_ids, n_query, test_seq_len, rng=None):
    """``eval_faiss.py:178-186``."""
    if test_ids.lower() == 'all':
        return np.arange(0, n_query - max(test_seq_len), 1)
    if test_ids.lower() == 'icassp':
        found = glob.glob('./**/test_ids_icassp2021.npy', recursive=True)
        path = found[0] if found else os.path.join(os.path.dirname(os.path.abspath(__file__)), 'test_ids_icassp2021.npy')
        return np.load(path)
    if test_ids.isnumeric():
        rng = rng or np.random
        return rng.permutation(n_query - max(test_seq_len))[:int(test_ids)]
    return np.load(test_ids)


def _sharded_index(index_type, dummy_db, db, max_len, max_train, rank, world, device):
    """Row-sharded stand-in for ``get_index`` + the two ``index.add`` calls (``eval_faiss.py:141-151``)."""
    from ..dist import ShardedFlatIndex, TorchComm
    from .utils.get_index import FLAT_L2, IVF_FLAT, IVFPQ, IVFPQR
    kinds = {'l2': FLAT_L2, 'ivfpq': IVFPQ, 'ivf': IVF_FLAT, 'ivfpq-rr': IVFPQR}
    mode = index_type.lower()
    if mode not in kinds:
        raise NotImplementedError(f"index_type '{mode}' is not available row-sharded (l2, ivfpq, ivf, ivfpq-rr are)")
    comm = None
    if world > 1:
        import torch
        import torch.distributed as dist
        if not dist.is_initialized():
            torch.cuda.set_device(device)
            dist.init_process_group('nccl')
        comm = TorchComm()
    print(f'Creating index: \033[93m{mode}\033[0m (rank {rank} of {world}, rows sharded)')
    index = ShardedFlatIndex(len(dummy_db) + len(db), rank, world, max_len=max_len, device=device, comm=comm,
                             index_type=kinds[mode])
    if mode != 'l2':
        start_time = time.time()
        max_train = int(max_train)
        train = dummy_db
        if rank == 0 and len(dummy_db) > max_train:     # eval_faiss.py:107-113 (only rank 0 trains)
            sel = np.sort(np.random.default_rng(None).permutation(len(dummy_db))[:max_train])
            train = dummy_db[sel, :]
        index.train(train if rank == 0 else None)
        print('Elapsed time: {:.2f} seconds.'.format(time.time() - start_time))
    index.add_from([dummy_db, db])
    return index


def _check_limits(index_type, test_seq_len, k_probe, nprobe=40):
    """The kernels' table sizes, checked before any data is loaded (the reference has no such limits; all of its
    defaults -- lengths <= 19, k_probe 20, nprobe 40 -- are inside them; DESIGN.md section 1)."""
    if len(test_seq_len) == 0 or min(test_seq_len) < 1 or max(test_seq_len) > 32:
        raise ValueError(f"--test_seq_len {list(test_seq_len)}: sequence lengths must be in 1..32 (matcher kernels)")
    if k_probe < 1 or k_probe > 128 or k_probe * int(max(test_seq_len)) > 1024:
        raise ValueError(f"--k_probe {k_probe}: need 1 <= k_probe <= 128 and k_probe x max(test_seq_len) <= 1024 "
                         f"(candidate table of the matcher), got {k_probe * int(max(test_seq_len))}")
    mode = index_type.lower()
    if mode in ('ivfpq', 'ivf') and nprobe * k_probe > 4096:
        raise ValueError(f"--k_probe {k_probe}: index_type {mode} needs nprobe x k_probe <= 4096 (nprobe {nprobe})")
    if mode == 'ivfpq-rr' and 4 * k_probe > 128:
        raise ValueError(f"--k_probe {k_probe}: index_type ivfpq-rr re-ranks 4 x k_probe candidates, at most 128")


def run_eval(emb_dir, emb_dummy_dir=None, index_type='ivfpq', nogpu=False, max_train=1e7, test_ids='icassp',
             test_seq_len='1 3 5 9 11 19', k_probe=20, display_interval=5, device=0, live=None, sharded=None):
    test_seq_len = np.asarray(list(map(int, test_seq_len.split())))
    _check_limits(index_type, test_seq_len, int(k_probe))
    world, rank = int(os.environ.get('WORLD_SIZE', '1')), int(os.environ.get('RANK', '0'))
    if sharded is None:
        sharded = world > 1
    if not sharded:
        world, rank = 1, 0
    elif world > 1:
        device = int(os.environ.get('LOCAL_RANK', str(rank)))

    query, query_shape = load_memmap_data(emb_dir, 'query')
    db, db_shape = load_memmap_data(emb_dir, 'db')
    if emb_dummy_dir is None:
        emb_dummy_dir = emb_dir
    dummy_db, dummy_db_shape = load_memmap_data(emb_dummy_dir, 'dummy_db')

    if sharded:
        if nogpu:
            from .._lib import NafpError
            raise NafpError("--nogpu: nafp-b200 has no CPU search path (no fallback by design)")
        start_time = time.time()
        index = _sharded_index(index_type, dummy_db, db, int(max(test_seq_len)), max_train, rank, world, device)
    else:
        index = get_index(index_type, dummy_db, dummy_db.shape, (not nogpu), max_train, device=device)
        start_time = time.time()
        index.add(dummy_db); print(f'{len(dummy_db)} items from dummy DB')
        index.add(db); print(f'{len(db)} items from reference DB')
    t = time.time() - start_time
    print(f'Added total {index.ntotal} items to DB. {t:>4.2f} sec.')

    print(f'test_id: \033[93m{test_ids}\033[0m,  ', end='')
    test_ids = np.asarray(select_test_ids(test_ids, len(query), test_seq_len), dtype=np.int64)
    if sharded and world > 1:          # a random selection ('N' test ids) must be the same on every rank
        import torch
        t_ids = torch.from_numpy(test_ids).to(torch.device('cuda', device))
        index.comm.broadcast(t_ids, 0)
        test_ids = t_ids.cpu().numpy()
    n_test = len(test_ids)
    gt_ids = test_ids + dummy_db_shape[0]
    print(f'n_test: \033[93m{n_test:n}\033[0m')

    n_len = len(test_seq_len)
    top1_exact = np.zeros((n_test, n_len)).astype(int)
    top1_near = np.zeros((n_test, n_len)).astype(int)
    top3_exact = np.zeros((n_test, n_len)).astype(int)
    top10_exact = np.zeros((n_test, n_len)).astype(int)

    pt = PrintTable(test_seq_len=test_seq_len,
                    row_names=['Top1 exact', 'Top1 near', 'Top3 exact', 'Top10 exact'], live=live if rank == 0 else False)
    query_np = np.ascontiguousarray(query)
    # ids are processed in blocks; a block is one batched GPU call (the reference refreshes its table
    # every display_interval ids -- blocks are a multiple of that so the refresh points coincide)
    block = max(int(display_interval), 1) * max(1, 256 // max(int(display_interval), 1))
    avg_search_time = float('nan')
    for b0 in range(0, n_test, block):
        start_time = time.time()
        ids = test_ids[b0:b0 + block]
        assert (ids <= len(query)).all()
        # only the query rows this block can touch cross PCIe (ids of a block are close together for sorted id
        # lists such as the ICASSP one: ~1/8 of the query set per block instead of all of it every time)
        q_lo = int(ids.min())
        q_hi = min(int(ids.max()) + int(max(test_seq_len)), len(query_np))
        pred, _ = index.seq_match(query_np[q_lo:q_hi], ids - q_lo, test_seq_len, k_probe)
        for j in range(len(ids)):
            ti = b0 + j
            for si in range(n_len):
                f = hit_flags(pred[j, si], gt_ids[ti])
                top1_exact[ti, si], top1_near[ti, si], top3_exact[ti, si], top10_exact[ti, si] = f
        done = b0 + len(ids)
        avg_search_time = (time.time() - start_time) / len(ids) / n_len
        rates = tuple(100. * np.mean(a[:done, :], axis=0) for a in (top1_exact, top1_near, top3_exact, top10_exact))
        if rank == 0:
            pt.update_counter(done - 1, n_test, avg_search_time * 1000.)
            pt.update_table(rates)

    rates = tuple(100. * np.mean(a, axis=0) for a in (top1_exact, top1_near, top3_exact, top10_exact))
    if rank == 0:
        pt.update_counter(n_test - 1, n_test, avg_search_time * 1000.)
        pt.update_table(rates)
        pt.close_table()
        np.save(f'{emb_dir}/raw_score.npy', np.concatenate((top1_exact, top1_near, top3_exact, top10_exact), axis=1))
        np.save(f'{emb_dir}/test_ids.npy', test_ids)
        print(f'Saved test_ids and raw score to {emb_dir}.')
    return rates


@click.command()
@click.argument('emb_dir', required=True, type=click.STRING)
@click.option('--emb_dummy_dir', default=None, type=click.STRING,
              help="Specify a directory containing 'dummy_db.mm' and 'dummy_db_shape.npy' to use. Default is EMB_DIR.")
@click.option('--index_type', '-i', default='ivfpq', type=click.STRING,
              help="Index type must be one of {'L2', 'IVF', 'IVFPQ', 'IVFPQ-RR'}; all four row-shard under torchrun "
                   "('IVFPQ-ONDISK' and 'HNSW' are CPU-only in the reference).")
@click.option('--nogpu', default=False, is_flag=True, help='Refused: this build has no CPU search path.')
@click.option('--max_train', default=1e7, type=click.INT, help='Max number of items for index training. Default is 1e7.')
@click.option('--test_seq_len', default='1 3 5 9 11 19', type=click.STRING,
              help="A set of different number of segments to test. Numbers are separated by spaces. "
                   "Default is '1 3 5 9 11 19', which corresponds to '1s, 2s, 3s, 5s, 6s, 10s'.")
@click.option('--test_ids', '-t', default='icassp', type=click.STRING,
              help="One of {'all', 'icassp', 'path/file.npy', (int)}.")
@click.option('--k_probe', '-k', default=20, type=click.INT, help="Top k search for each segment. Default is 20")
@click.option('--display_interval', '-dp', default=10, type=click.INT, help="Display interval. Default is 10.")
def eval_faiss(emb_dir, emb_dummy_dir=None, index_type='ivfpq', nogpu=False, max_train=1e7, test_ids='icassp',
               test_seq_len='1 3 5 9 11 19', k_probe=20, display_interval=5):
    """Segment/sequence-wise audio search experiment and evaluation (B200).

    ex) python -m nafp_b200.eval.eval_search EMB_DIR --index_type l2

    EMB_DIR: Directory where {query, db, dummy_db}.mm files are located. The 'raw_score.npy' and
    'test_ids.npy' will be also created in the same directory.
    """
    run_eval(emb_dir, emb_dummy_dir, index_type, nogpu, max_train, test_ids, test_seq_len, k_probe, display_interval)


if __name__ == "__main__":
    eval_faiss()
