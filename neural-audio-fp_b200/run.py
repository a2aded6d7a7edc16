"""Command line: ``generate`` and ``evaluate`` of the reference's ``run.py`` (``run.py:77-162``), and ``identify``
(recordings against the database ``generate`` wrote).  ``train`` is outside the inference hot path and is not
provided."""
from __future__ import annotations

import os
import sys

import click
import yaml


def load_config(config_fname):
    """``run.py:13-22``: YAML from ./config/NAME.yaml (or a direct path)."""
    config_filepath = config_fname if os.path.exists(config_fname) else './config/' + config_fname + '.yaml'
    if os.path.exists(config_filepath):
        print(f'cli: Configuration from {config_filepath}')
    else:
        sys.exit(f'cli: ERROR! Configuration file {config_filepath} is missing!!')
    with open(config_filepath, 'r') as f:
        return yaml.safe_load(f)


def update_config(cfg, key1: str, key2: str, val):
    cfg[key1][key2] = val
    return cfg


@click.group()
def cli():
    """nafp-b200: B200-native fingerprint generation and search of neural-audio-fp."""


@cli.command()
@click.argument('checkpoint_name', required=True)
@click.argument('checkpoint_index', required=False)
@click.option('--config', '-c', default='default', required=False, type=click.STRING,
              help="Name of the model configuration file located in 'config/'. Default is 'default'")
@click.option('--source', '-s', default=None, type=click.STRING, required=False,
              help="Custom source root directory. The source must be 16-bit 8 Khz mono WAV.")
@click.option('--output', '-o', default=None, type=click.STRING, required=False,
              help="Root directory where the generated embeddings (uncompressed) will be stored.")
@click.option('--skip_dummy', default=False, is_flag=True, help='Exclude dummy-DB from the default source.')
def generate(checkpoint_name, checkpoint_index, config, source, output, skip_dummy):
    """Generate fingerprints from a saved checkpoint ('random-init[:SEED]' for seeded random weights).

    Under torchrun (one process per GPU: RANK / WORLD_SIZE / LOCAL_RANK) the batches are split over the ranks."""
    from .model.generate import distributed_env, generate_fingerprint
    cfg = load_config(config)
    rank, world, device = distributed_env()
    if world > 1:
        print(f'cli: rank {rank} of {world} on GPU {device}')
    generate_fingerprint(cfg, checkpoint_name, checkpoint_index, source, output, skip_dummy,
                         rank=rank, world_size=world, device=device)


@cli.command()
@click.argument('checkpoint_name', required=True)
@click.argument('checkpoint_index', required=True)
@click.option('--config', '-c', default='default', required=False, type=click.STRING)
@click.option('--index_type', '-i', default='IVFPQ', type=click.STRING)
@click.option('--test_seq_len', default='1 3 5 9 11 19', type=click.STRING)
@click.option('--test_ids', '-t', default='icassp', type=click.STRING)
@click.option('--nogpu', default=False, is_flag=True)
def evaluate(checkpoint_name, checkpoint_index, config, index_type, test_seq_len, test_ids, nogpu):
    """Search and evaluation (``run.py:138-162``)."""
    from .eval.eval_search import eval_faiss
    cfg = load_config(config)
    emb_dir = cfg['DIR']['OUTPUT_ROOT_DIR'] + checkpoint_name + '/' + str(checkpoint_index) + '/'
    argv = [emb_dir, '--index_type', index_type, '--test_seq_len', test_seq_len, '--test_ids', test_ids]
    if nogpu:
        argv.append('--nogpu')
    eval_faiss(argv)


@cli.command()
@click.argument('checkpoint_name', required=True)
@click.argument('checkpoint_index', required=False)
@click.option('--config', '-c', default='default', required=False, type=click.STRING)
@click.option('--query', '-q', required=True, type=click.STRING,
              help="A 16-bit 8 kHz mono WAV, or a directory of them, to identify.")
@click.option('--emb_dir', default=None, type=click.STRING,
              help="Directory of the database memmaps. Default is OUTPUT_ROOT_DIR/CHECKPOINT_NAME/CHECKPOINT_INDEX/.")
@click.option('--source', '-s', default=None, type=click.STRING,
              help="The --source the database was generated from (its rows are then custom_source).")
@click.option('--skip_dummy', default=False, is_flag=True, help="The database was generated with --skip_dummy.")
@click.option('--index_type', '-i', default='l2', type=click.STRING, help="One of {'l2', 'ivfpq', 'ivf', 'ivfpq-rr'}.")
@click.option('--k_probe', '-k', default=20, type=click.INT, help="Top k search for each segment (<= 128). Default is 20.")
@click.option('--top', default=10, type=click.INT, help="Matches reported per clip (<= 100). Default is 10.")
@click.option('--window', default=None, type=click.FLOAT,
              help="Identify consecutive windows of this many seconds separately (recordings of several tracks).")
@click.option('--output', '-o', default=None, type=click.STRING, help="Write the matches to this JSON file.")
def identify(checkpoint_name, checkpoint_index, config, query, emb_dir, source, skip_dummy, index_type, k_probe, top,
             window, output):
    """Identify recordings: for each query file (or --window of it), the database tracks and offsets it matches.

    ex) python -m nafp_b200.run identify CKPT 100 -c default --query rec.wav -i l2"""
    from .eval.identify import run_identify
    cfg = load_config(config)
    run_identify(cfg, checkpoint_name, checkpoint_index, query, emb_dir=emb_dir, source=source, skip_dummy=skip_dummy,
                 index_type=index_type, k_probe=k_probe, top=top, window=window, output=output)


if __name__ == '__main__':
    cli()
