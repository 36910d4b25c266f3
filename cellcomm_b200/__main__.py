"""Entry point: `python3 src` / `python3 -m cellcomm_b200`.

Behaviour of the reference's src/__main__.py:30-99: with no argument train
`ContinuousCellBiGan` (Z = 3, batch 128, one iteration) on the second GSE122930 source with
the stdout / CSV / MongoDB interceptors; `convert <matrix.mtx> <cells.csv>` writes the dense
cell file `load_cells` reads.  The run's log directory `logs/<MM-DD-HHMM>_<RUN_ID>_e<Z>` must
not exist yet; Ctrl-C ends the process with exit status 0.

The module-level names other code may import are kept (`SOURCE_IDS`, `SOURCES`, `RUN_ID`,
`DATA_SOURCES`, `run_training`, `create_interceptors`, `check_log_dir`,
`store_converted_cell_file`).  `generate <checkpoint.npz> <source-matrix-file> <n-cells>
<target-matrix-file>` (not in the reference) writes n generated cells of a trained checkpoint
as a 10x .mtx with the source matrix's gene ids.  `score <checkpoint.npz> <source-matrix-file>
<matrix-file> <scores.csv>` (not in the reference) scores every cell of a matrix with a trained
checkpoint: one CSV row `barcode,mse,d-real,z0,...` per cell (reconstruction error,
discriminator probability, encoding; `BasicBiGan.score_cells`).  Environment knobs the
reference does not have: CELLCOMM_DATA_DIR (directory of the `<source>_matrix.mtx /
_barcodes.tsv / _genes.tsv` files, default `<repo>/data`), CELLCOMM_ITERATIONS,
CELLCOMM_BATCH_SIZE, CELLCOMM_SEED, and CELLCOMM_VALIDATION_MATRIX=<file.mtx>: held-out cells
(read against the same genes.tsv) scored after every iteration into `validation.csv`.

Reproducible runs: CELLCOMM_SEED=<int> seeds numpy's global state (the batch sampler) and the
network (weights, device RNG key, host priors).  With CELLCOMM_B200_DETERMINISTIC=1 as well,
two runs on the same data, GPU count and build write identical losses (DESIGN.md section 2).

Data parallel: `torchrun --nproc-per-node N -m cellcomm_b200` (or `... src`) runs one process
per GPU.  Every rank loads the matrix and trains on its contiguous share of each global
batch of `batch_size` cells; rank 0 alone creates the log directory and the interceptors
(stdout, CSV, MongoDB) and the encode-all-cells pass they trigger is sharded by rows over
all ranks (`CellTraining.run`).
"""
import os
import signal
import sys
import time

import numpy as np

from . import intercepts
from .cell_type_training import CellTraining, load_matrix

ENCODING_SIZE = 3
DATA_DIR = os.environ.get('CELLCOMM_DATA_DIR') or os.path.normpath(
    os.path.join(os.path.dirname(os.path.abspath(__file__)), os.pardir, 'data'))
SOURCE_FILES = {'matrix': 'mtx', 'barcodes': 'tsv', 'genes': 'tsv'}

SOURCE_IDS = [f'GSE122930_{name}' for name in
              ('TAC_1_week_repA+B', 'TAC_4_weeks_repA+B', 'Sham_1_week', 'Sham_4_weeks_repA+B')]
SOURCES = [{kind: os.path.join(DATA_DIR, f'{sid}_{kind}.{ext}') for kind, ext in SOURCE_FILES.items()}
           for sid in SOURCE_IDS]
RUN_ID = 'test'
DATA_SOURCES = SOURCES[1]


def _env_int(name, default):
    return int(os.environ.get(name, default))


def check_log_dir(log_dir):
    """Create the run's log directory; an existing one means the run id was used before."""
    if os.path.exists(log_dir):
        raise AssertionError(f'duplicate run-id, log-dir: {log_dir}')
    os.makedirs(log_dir)


def create_interceptors(encoding_size, trainer, sources):
    """stdout losses + losses.csv + the MongoDB recorder (every iteration from the first), and
    with CELLCOMM_VALIDATION_MATRIX set, validation.csv: that matrix, aligned to the training
    matrix's gene ids, scored after every iteration."""
    validation_file = os.environ.get('CELLCOMM_VALIDATION_MATRIX', '').strip()
    held_out = None
    if validation_file:
        held_out = load_matrix(validation_file).reindex_columns(trainer.data.columns)
    full_run_id = f"{time.strftime('%m-%d-%H%M')}_{RUN_ID}_e{encoding_size}"
    log_dir = os.path.join('logs', full_run_id)
    check_log_dir(log_dir)
    recorder = intercepts.DbRecorder(RUN_ID, sources)
    recorder.setup()
    record = intercepts.skip_iterations(1, recorder.create_interceptor(trainer))
    sink = intercepts.SinkIntercepts(log_dir)
    chain = [intercepts.print_losses(full_run_id), sink.save_losses(),
             intercepts.offset_iterations(0, record)]
    if held_out is not None:
        chain.append(sink.save_validation(trainer, held_out))
    return intercepts.combined_interceptors(chain)


def init_data_parallel():
    """Under torchrun (WORLD_SIZE > 1): bind this process to its GPU and join the NCCL group.
    -> (rank, world_size)."""
    world = _env_int('WORLD_SIZE', 1)
    if world <= 1:
        return 0, 1
    import torch
    import torch.distributed as dist
    if not dist.is_initialized():
        if torch.cuda.is_available() and os.environ.get('CELLCOMM_B200_DEVICE', 'cuda') != 'cpu':
            local = _env_int('LOCAL_RANK', 0)
            torch.cuda.set_device(local)
            dist.init_process_group('nccl', device_id=torch.device('cuda', local))
        else:
            dist.init_process_group('gloo')
    return dist.get_rank(), dist.get_world_size()


def env_seed():
    """CELLCOMM_SEED as an int, or None when unset or empty."""
    v = os.environ.get('CELLCOMM_SEED', '').strip()
    return int(v) if v else None


def run_training(batch_size=128):
    rank, world = init_data_parallel()
    cells = load_matrix(DATA_SOURCES['matrix'], verbose=rank == 0)
    seed = env_seed()
    if seed is not None:
        np.random.seed(seed)      # the batch sampler draws from numpy's global state
    trainer = CellTraining(cells, batch_size=batch_size, encoding_size=ENCODING_SIZE, seed=seed)
    # side effects (log directory, Mongo documents, stdout) belong to rank 0 alone
    interceptors = create_interceptors(ENCODING_SIZE, trainer, DATA_SOURCES) if rank == 0 else None
    trainer.run(_env_int('CELLCOMM_ITERATIONS', 1), interceptors)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def store_converted_cell_file(matrix_file, cell_file):
    print('converting matrix file:')
    cells = load_matrix(matrix_file, verbose=True)
    print('storing cell file:', cell_file, '... ', end='', flush=True)
    cells.to_csv(cell_file)
    print('done')


def _restore_network(checkpoint_file, matrix_file, verb):
    """-> (the network of a checkpoint written by save_checkpoint, the source matrix).  The
    variant and sizes come from the checkpoint; the source's gene count is checked before a
    network is built.  One process (no data-parallel group); the checkpoint's host RNG states
    are restored with the weights, so what follows draws the same numbers every time."""
    with np.load(checkpoint_file, allow_pickle=False) as f:
        variant = str(f['meta/variant'])
        encoding_size = int(f['meta/encoding_size'])
        gene_size = int(f['meta/gene_size'])
    source = load_matrix(matrix_file)
    if source.shape[1] != gene_size:
        raise ValueError(f'{checkpoint_file} {verb} {gene_size} genes, but {matrix_file} '
                         f'has {source.shape[1]}')
    if variant == 'cont':
        from .bigan_cont import ContinuousCellBiGan as Network
    elif variant == 'classify':
        from .bigan_classify import ClassifyCellBiGan as Network
    else:
        raise ValueError(f'{checkpoint_file}: unknown network variant {variant!r}')
    network = Network(encoding_size, gene_size)
    network.load_checkpoint(checkpoint_file)
    return network, source


def generate_matrix_file(checkpoint_file, matrix_file, n_cells, target_file):
    """n generated cells from a checkpoint written by save_checkpoint, as a 10x .mtx file whose
    gene ids are the source matrix's.  The same checkpoint and n always write the same file."""
    n = int(n_cells)
    if n < 1:
        raise ValueError(f'n-cells must be at least 1, got {n}')
    network, source = _restore_network(checkpoint_file, matrix_file, 'generates')
    encodings = network.random_encoding_vector(n)
    cells = network.generate_cell_matrix(encodings, columns=source.columns)
    print('storing generated cells:', target_file, '... ', end='', flush=True)
    cells.to_mtx(target_file)
    print('done')


def write_score_file(path, barcodes, scores):
    """`barcode,mse,d-real,z0,...,z{Z-1}`, one row per cell; floats as %.9g (round-trips
    float32).  The file appears atomically: written under a temporary name in the same
    directory and renamed into place, so a failed write leaves no partial file at `path`."""
    Z = scores.encodings.shape[1]
    tmp = f'{path}.{os.getpid()}.tmp'
    try:
        with open(tmp, 'w') as f:
            f.write(','.join(['barcode', 'mse', 'd-real'] + [f'z{k}' for k in range(Z)]) + '\n')
            for b, m, d, z in zip(barcodes, scores.mse, scores.d_real, scores.encodings):
                f.write(f'{int(b)},' + ','.join('%.9g' % float(v) for v in (m, d, *z)) + '\n')
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise
    return path


def score_matrix_file(checkpoint_file, matrix_file, cells_file, scores_file):
    """Score every cell of `cells_file` with a checkpoint written by save_checkpoint and write
    the CSV of write_score_file.  The cells are aligned to the source matrix's gene ids first
    (CellMatrix.reindex_columns: genes the source lacks are dropped, missing ones are zero).
    The same checkpoint and cells always write the same file."""
    network, source = _restore_network(checkpoint_file, matrix_file, 'scores')
    cells = load_matrix(cells_file).reindex_columns(source.columns)
    scores = network.score_cells(cells)
    print('storing cell scores:', scores_file, '... ', end='', flush=True)
    write_score_file(scores_file, cells.index, scores)
    print('done')


def _stop(_signum, _frame):
    print('\tstopped')
    sys.exit(0)


def main(argv):
    signal.signal(signal.SIGINT, _stop)
    commands = {'convert': (2, store_converted_cell_file,
                            'convert <source-matrix-file> <convert-target-file>'),
                'generate': (4, generate_matrix_file,
                             'generate <checkpoint.npz> <source-matrix-file> <n-cells> '
                             '<target-matrix-file>'),
                'score': (4, score_matrix_file,
                          'score <checkpoint.npz> <source-matrix-file> <matrix-file> '
                          '<scores.csv>')}
    if len(argv) < 2:
        run_training(_env_int('CELLCOMM_BATCH_SIZE', 128))
        return
    name, params = argv[1], argv[2:]
    if name not in commands:
        print('unrecognised command:', name)
        return
    n_params, handler, usage = commands[name]
    assert len(params) == n_params, f'required parameters missing: {usage}'
    handler(*params)


if __name__ == '__main__':
    main(sys.argv)
