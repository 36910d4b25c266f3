"""`losses.csv` / `accuracy.csv` interceptors (API of the reference's
src/intercepts/sink_intercepts.py:6-31), and `validation.csv` (not in the reference): each
appends one row per iteration through a `DataSink` that is drained at interpreter exit.

    losses.csv      iteration,total-loss,g-loss,e-loss,d-loss
    accuracy.csv    iteration,pos-pct,neg-pct   (fractions of a freshly sampled batch that
                                                 the discriminator classifies correctly)
    validation.csv  iteration,mse,d-real,real-pct   (score_cells over fixed held-out cells:
                                                 mean reconstruction error, mean discriminator
                                                 probability, fraction with round(d) == 1)
"""
import atexit

import numpy as np

from .data_sink import DataSink

LOSS_COLUMNS = ('iteration', 'total-loss', 'g-loss', 'e-loss', 'd-loss')
ACCURACY_COLUMNS = ('iteration', 'pos-pct', 'neg-pct')
VALIDATION_COLUMNS = ('iteration', 'mse', 'd-real', 'real-pct')


class SinkIntercepts:
    def __init__(self, log_dir):
        self.sink = DataSink(log_dir=log_dir)
        atexit.register(self.sink.drain_data)

    def _open(self, graph_id, columns):
        self.sink.add_graph_header(graph_id, list(columns))
        return lambda row: self.sink.add_data(graph_id, row)

    def save_losses(self):
        write = self._open('losses', LOSS_COLUMNS)

        def store_record(it, all_losses):
            # device-resident LossScalars become host floats here (one read per iteration)
            g, e, d = map(float, all_losses)
            write([it, g + e + d, g, e, d])

        return store_record

    def save_accuracy(self, trainer):
        write = self._open('accuracy', ACCURACY_COLUMNS)

        def intercept(it, _losses):
            batch = trainer.sample_cell_data()
            true_pos, true_neg = trainer.network.evaluate_discriminator_accuracy(batch)
            write([it, true_pos / len(batch), true_neg / len(batch)])

        return intercept

    def save_validation(self, trainer, cells, noise_seed=0):
        """Score the held-out `cells` (same gene ids as trainer.data, e.g. a matrix aligned with
        CellMatrix.reindex_columns) with the network being trained, once per iteration.  The
        generator noise is drawn once, here, from np.random.default_rng(noise_seed): every
        iteration scores the same cells with the same noise, and the run's own RNG streams
        (numpy's global state, the prior generator, the device counter) are never touched."""
        if not np.array_equal(np.asarray(cells.columns), np.asarray(trainer.data.columns)):
            raise ValueError('validation cells must have the gene ids of the training matrix '
                             '(align them with CellMatrix.reindex_columns)')
        if len(cells) == 0:
            raise ValueError('validation needs at least one cell')
        network = trainer.network
        noise = np.random.default_rng(noise_seed).random((len(cells), network.encoding_size),
                                                          dtype=np.float32)
        write = self._open('validation', VALIDATION_COLUMNS)

        def intercept(it, _losses):
            scores = network.score_cells(cells, noise)
            d_real = scores.d_real.astype(np.float64)
            write([it, float(np.mean(scores.mse, dtype=np.float64)), float(np.mean(d_real)),
                   float(np.mean(np.round(d_real) == 1))])

        return intercept
