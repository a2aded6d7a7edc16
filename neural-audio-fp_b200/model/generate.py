"""Fingerprint extraction driver: the reference's ``model/generate.py`` over libnafp.

Same call surface (``generate_fingerprint(cfg, checkpoint_name, checkpoint_index, source_root_dir,
output_root_dir, skip_dummy)``), same outputs (``{key}.mm`` raw float32 C-order memmaps plus
``{key}_shape.npy`` for key in dummy_db / query / db or custom_source, ``generate.py:122-161``), same
batch grouping (consecutive ``BSZ.TS_BATCH_SZ`` segments share the log-mel max, ``:176-181``).

Checkpoints: ``{LOG_ROOT_DIR}checkpoint/{checkpoint_name}/ckpt-{index}`` is either the ``.npz`` exchange format
of ``model/weights.py`` or the reference's own TensorFlow checkpoint (``.index`` + ``.data-*``), which
``model/tf_checkpoint.py`` reads without TensorFlow.  The name ``random-init[:SEED]`` selects seeded Keras-default
initialisation (what the reference would hold before training).

Multi-GPU (SURVEY §8 e, "split by segment batch with no collective"): started once per GPU -- ``torchrun`` or any
launcher that sets RANK / WORLD_SIZE / LOCAL_RANK -- every rank fingerprints a contiguous range of whole
TS_BATCH_SZ batches and writes its own rows of the shared memmap.  The only synchronisation is a barrier around the
creation of each output file; it runs over a CPU (gloo) process group because no tensor ever crosses ranks.
"""
from __future__ import annotations

import glob
import os
import re
import sys

import numpy as np

from .dataset import Dataset
from .fp import build_fp, test_step  # noqa: F401  (test_step re-exported: reference name)
from .weights import init_weights, load_weights


def load_checkpoint(checkpoint_root_dir, checkpoint_name, checkpoint_index, m_fp):
    """Mirror of ``generate.py:26-52``: restore the latest or the given checkpoint into m_fp."""
    if checkpoint_name.startswith('random-init'):
        seed = int(checkpoint_name.split(':')[1]) if ':' in checkpoint_name else 7
        m_fp.load(init_weights(seed, norm=m_fp.norm))
        print(f'---Initialised random weights (seed {seed})---')
        return 0 if checkpoint_index is None else checkpoint_index
    checkpoint_dir = checkpoint_root_dir + f'/{checkpoint_name}/'
    # two on-disk forms: the .npz exchange file (model/weights.py) and the reference's own TensorFlow checkpoint
    # (ckpt-N.index + ckpt-N.data-*), which model/tf_checkpoint.py reads without TensorFlow
    from .tf_checkpoint import latest_checkpoint, load_tf_checkpoint
    if checkpoint_index is None:
        print("\x1b[1;32mArgument 'checkpoint_index' was not specified.\x1b[0m")
        print('\x1b[1;32mSearching for the latest checkpoint...\x1b[0m')
        found = []
        for p in glob.glob(checkpoint_dir + 'ckpt-*.npz'):
            m = re.search(r'ckpt-(\d+)\.npz$', p)
            if m:
                found.append(int(m.group(1)))
        tf_index, _ = latest_checkpoint(checkpoint_dir)
        if tf_index is not None:
            found.append(tf_index)
        if not found:
            raise FileNotFoundError(f'Cannot find checkpoint in {checkpoint_dir}')
        checkpoint_index = max(found)
    prefix = checkpoint_dir + 'ckpt-' + str(checkpoint_index)
    if os.path.exists(prefix + '.npz'):
        m_fp.load(load_weights(prefix + '.npz'))
        print(f'---Restored from {prefix}.npz---')
    elif os.path.exists(prefix + '.index'):
        m_fp.load(load_tf_checkpoint(prefix, norm=m_fp.norm))
        print(f'---Restored from {prefix} (TensorFlow checkpoint)---')
    else:
        raise FileNotFoundError(prefix + '.npz / .index')
    return checkpoint_index


def prevent_overwrite(key, target_path):
    if (key == 'dummy_db') & os.path.exists(target_path):
        answer = input(f'{target_path} exists. Will you overwrite (y/N)?')
        if answer.lower() not in ['y', 'yes']:
            sys.exit()


def get_data_source(cfg, source_root_dir, skip_dummy):
    dataset = Dataset(cfg)
    ds = dict()
    if source_root_dir:
        ds['custom_source'] = dataset.get_custom_db_ds(source_root_dir)
    else:
        if skip_dummy:
            print("Excluding \033[33m'dummy_db'\033[0m from source.")
        else:
            ds['dummy_db'] = dataset.get_test_dummy_db_ds()
        if dataset.datasel_test_query_db in ['unseen_icassp', 'unseen_syn']:
            ds['query'], ds['db'] = dataset.get_test_query_db_ds()
        else:
            raise ValueError(dataset.datasel_test_query_db)
    print(f'\x1b[1;32mData source: {ds.keys()}\x1b[0m', f'{dataset.datasel_test_query_db}')
    return ds


def _shard(n_batches, rank, world):
    """Contiguous range of whole batches for this rank (SURVEY §8 e: no collective)."""
    per, rem = divmod(n_batches, world)
    lo = rank * per + min(rank, rem)
    return lo, lo + per + (1 if rank < rem else 0)


def distributed_env():
    """(rank, world_size, device) of this process from the launcher's environment.  NAFP_DEVICE overrides the GPU
    (default LOCAL_RANK): several ranks may share one GPU, e.g. in the 2-rank test on a single-GPU box."""
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    device = int(os.environ.get('NAFP_DEVICE', os.environ.get('LOCAL_RANK', '0')))
    return rank, world, device


def _barrier_fn(world_size):
    """Barrier over the ranks of a generation job: a gloo (CPU) group -- the data path has no collective."""
    if world_size <= 1:
        return lambda: None
    import torch.distributed as dist
    if not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('gloo')
    group = dist.new_group(backend='gloo') if dist.get_backend() != 'gloo' else None
    return lambda: dist.barrier(group=group)


def generate_fingerprint(cfg, checkpoint_name, checkpoint_index, source_root_dir, output_root_dir, skip_dummy,
                         rank=None, world_size=None, device=None, batches_per_call=64):
    """See the module docstring.  ``rank`` / ``world_size`` / ``device`` default to the launcher's environment
    (RANK, WORLD_SIZE, LOCAL_RANK): every rank fingerprints a contiguous range of whole TS_BATCH_SZ batches on its
    own GPU and writes its rows of the shared memmap."""
    env_rank, env_world, env_device = distributed_env()
    rank = env_rank if rank is None else int(rank)
    world_size = env_world if world_size is None else int(world_size)
    if device is None:
        device = env_device if world_size > 1 else 0
    if not 0 <= rank < world_size:
        raise ValueError(f'rank {rank} outside world_size {world_size}')
    barrier = _barrier_fn(world_size)
    m_pre, m_fp = build_fp(cfg, device=device)
    checkpoint_root_dir = cfg['DIR']['LOG_ROOT_DIR'] + 'checkpoint/'
    checkpoint_index = load_checkpoint(checkpoint_root_dir, checkpoint_name, checkpoint_index, m_fp)

    ds = get_data_source(cfg, source_root_dir, skip_dummy)

    if output_root_dir:
        output_root_dir = output_root_dir + f'/{checkpoint_name}/{checkpoint_index}/'
    else:
        output_root_dir = cfg['DIR']['OUTPUT_ROOT_DIR'] + f'/{checkpoint_name}/{checkpoint_index}/'
    os.makedirs(output_root_dir, exist_ok=True)
    if not skip_dummy and rank == 0:
        prevent_overwrite('dummy_db', f'{output_root_dir}/dummy_db.mm')

    sz_check = dict()
    for key in ds.keys():
        bsz = int(cfg['BSZ']['TS_BATCH_SZ'])
        n_items = ds[key].n_samples
        dim = cfg['MODEL']['EMB_SZ']
        assert n_items > 0
        arr_shape = (n_items, dim)
        path = f'{output_root_dir}/{key}.mm'
        if rank == 0:
            arr = np.memmap(path, dtype='float32', mode='w+', shape=arr_shape)
            np.save(f'{output_root_dir}/{key}_shape.npy', arr_shape)
        barrier()                      # the file exists at its full size before any other rank maps it
        if rank != 0:
            arr = np.memmap(path, dtype='float32', mode='r+', shape=arr_shape)

        print(f"=== Generating fingerprint from \x1b[1;32m'{key}'\x1b[0m bsz={bsz}, {n_items} items, d={dim} ===")
        if rank == 0 and ds[key].conversions():
            print(ds[key].conversions())
        b_lo, b_hi = _shard(len(ds[key]), rank, world_size)
        # several whole batches per call (the library keeps TS_BATCH_SZ groups separate); the next block is cut
        # from the WAV files by a worker thread while the GPU works on this one (ctypes releases the GIL)
        from concurrent.futures import ThreadPoolExecutor
        blocks = [(i, min(i + batches_per_call, b_hi)) for i in range(b_lo, b_hi, batches_per_call)]
        with ThreadPoolExecutor(max_workers=1) as pool:
            nxt = pool.submit(ds[key].get_source_block, *blocks[0]) if blocks else None
            for n_blk, (i, j) in enumerate(blocks):
                block = nxt.result()
                nxt = pool.submit(ds[key].get_source_block, *blocks[n_blk + 1]) if n_blk + 1 < len(blocks) else None
                # whole-track sample runs + one window per segment: the GPU resamples the runs that are not 8 kHz mono
                # and cuts the overlapping segments
                emb = m_fp.fingerprint_block(block, group_size=bsz)
                arr[i * bsz:i * bsz + len(emb), :] = emb
                if rank == 0:
                    print(f'\r{j - b_lo}/{b_hi - b_lo}', end='', flush=True)
        if rank == 0:
            print()
        print(f'=== Succesfully stored {arr_shape[0]} fingerprint to {output_root_dir} ===')
        sz_check[key] = len(arr)
        arr.flush()
        del arr
        barrier()                      # every rank's rows are on disk before anyone moves on / returns

    if 'custom_source' in ds.keys():
        pass
    elif sz_check['db'] != sz_check['query']:
        print("\033[93mWarning: 'db' and 'qeury' size does not match. This can cause a problem in evaluataion stage.\033[0m")
    return
