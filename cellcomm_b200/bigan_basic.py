"""Drop-in for the reference's `src/bigan_basic.py` (BasicBiGan :10-81, components_changed
:84-89): same constructor, attributes and method names.  The three components are whatever the
injected factories return (the reference's tests inject MagicMocks, test/bigans_basic_test.py:
12-18), so this base class only relies on `.predict`, `.summary` and `.layers`.
"""
from abc import abstractmethod
from collections import namedtuple
from typing import Callable

import numpy as np

try:
    from typing import final
except ImportError:  # pragma: no cover
    def final(f):
        return f

# per-cell scores of score_cells: encodings [n, Z], mse [n], d_real [n], all float32
CellScores = namedtuple("CellScores", ["encodings", "mse", "d_real"])


class BasicBiGan:
    def __init__(self, encoding_size, gene_size,
                 generator_factory: Callable[[int, int], object],
                 encoder_factory: Callable[[int, int], object],
                 discriminator_factory: Callable[[int, int], object]
                 ):
        self.encoding_size = encoding_size
        self._generator = generator_factory(encoding_size, gene_size)
        self._encoder = encoder_factory(encoding_size, gene_size)
        self._discriminator = discriminator_factory(encoding_size, gene_size)
        self.all_components = self._generator, self._encoder, self._discriminator
        # the reference snapshots the weights here (src/bigan_basic.py:21-22); engine-backed
        # components have no weights until the subclass binds them, which then calls
        # _snapshot_params() itself
        self.__prev_params = None
        if not any(callable(getattr(c, 'weight_fingerprint', None)) and not _is_mock(c)
                   for c in self.all_components):
            self._snapshot_params()
        # private host RNG for the uniform priors: tf.random.uniform in the reference draws
        # from TensorFlow's generator, never from numpy's global state (which the batch sampler
        # and the classify prior use), so the numpy stream stays reference-identical.
        self._prior_rng = np.random.default_rng()

    @final
    def summary(self):
        for component in self.all_components:
            component.summary()

    @final
    def encoding_prediction(self, cell_data):
        return self._encoder.predict(cell_data)

    @abstractmethod
    def random_encoding_vector(self, batch_size):
        pass

    def random_uniform_vector(self, batch_size):
        """tf.random.uniform(shape=(batch_size, encoding_size), 0, 1): float32 in [0, 1)."""
        return self._prior_rng.random((batch_size, self.encoding_size), dtype=np.float32)

    @final
    def generate_cells(self, encoding_in, random_in=None):
        if random_in is None:
            random_in = self.random_uniform_vector(len(encoding_in))
        prediction = self._generator.predict((encoding_in, random_in))
        return np.round(prediction)          # round half to even, like tf.math.round

    def generate_cell_matrix(self, encoding_in, random_in=None, columns=None):
        """generate_cells(encoding_in, random_in) as a sparse CellMatrix: cells are rows with
        barcode ids 1..n, genes are columns with ids `columns` (default 1..gene_size).  This is
        the definition; engine-backed subclasses stream the same numbers without a dense
        (n, genes) intermediate."""
        try:
            from .cell_type_training import CellMatrix
        except ImportError:  # imported as a top-level module (PYTHONPATH=src style)
            from cellcomm_b200.cell_type_training import CellMatrix
        return CellMatrix.from_dense(self.generate_cells(encoding_in, random_in), columns=columns)

    def score_cells(self, cell_data, random_in=None):
        """Per-cell scores of a trained network on cells it may never have seen -> CellScores:
            encodings = encoding_prediction(cell_data)                        (z)
            mse       = mean over genes of (G.predict((z, random_in)) - x)^2  (the cycle loss of
                        the generator-with-encoder sub-step, per cell, before rounding)
            d_real    = D.predict((z, cell_data))                   (the real pair's probability)
        random_in=None draws the generator noise with random_uniform_vector, as generate_cells
        does.  This is the definition; engine-backed subclasses stream the same numbers without
        a dense (n, genes) intermediate."""
        encodings = self.encoding_prediction(cell_data)
        if random_in is None:
            random_in = self.random_uniform_vector(len(encodings))
        prediction = self._generator.predict((encodings, random_in))
        diff = np.asarray(prediction, dtype=np.float64) - np.asarray(cell_data, dtype=np.float64)
        mse = np.mean(np.square(diff, out=diff), axis=-1)
        d_real = self._discriminator.predict((encodings, cell_data))
        return CellScores(np.asarray(encodings, dtype=np.float32), mse.astype(np.float32),
                          np.asarray(d_real, dtype=np.float32).reshape(-1))

    @abstractmethod
    def trainings_step(self, sampled_batch):
        pass

    def evaluate_discriminator_accuracy(self, sampled_batch):
        """
            return format: ( true-positives, true-negatives )
        """
        batch_size = len(sampled_batch)
        random_encodings = self.random_encoding_vector(batch_size)
        generated_cells = self.generate_cells(random_encodings)
        result = self._discriminator.predict((random_encodings, generated_cells), use_multiprocessing=True)
        false_negatives = np.count_nonzero(np.round(result))

        encodings = self.encoding_prediction(sampled_batch)
        result = self._discriminator.predict((encodings, sampled_batch), use_multiprocessing=True)
        true_positives = np.count_nonzero(np.round(result))

        return true_positives, batch_size - false_negatives

    def _snapshot_params(self):
        self.__prev_params = self.__last_layer_params()

    def print_params_changes(self, msg):
        curr_params = self.__last_layer_params()
        if self.__prev_params is None:
            self.__prev_params = curr_params
        changed = [components_changed(p_now, p_orig) for p_now, p_orig in zip(curr_params, self.__prev_params)]
        print(msg, 'G|E|D changed:', f'{changed[0]:1} | {changed[1]:1} | {changed[2]:1},')
        self.__prev_params = curr_params

    def __last_layer_params(self):
        def collect_weights(component):
            fingerprint = getattr(component, 'weight_fingerprint', None)
            if callable(fingerprint) and not _is_mock(component):
                return [fingerprint()]       # device-side digest instead of a 3.4 GiB host copy
            collected_weights = []
            for lay in component.layers:
                weights = lay.get_weights()
                if len(weights) == 2:
                    collected_weights.extend(np.array(w, copy=True) for w in weights)
            return collected_weights

        return list(map(collect_weights, self.all_components))


def _is_mock(obj):
    return type(obj).__module__.startswith('unittest.mock')


def components_changed(p_now, p_orig):
    for n, o in zip(p_now, p_orig):
        if not np.all(np.equal(n, o)):
            return True
    return False
