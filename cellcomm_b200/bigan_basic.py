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

# per-group, per-gene statistics of gene_statistics: cells int64 [K]; mean, var (unbiased) and
# detected (fraction of the group's cells where the gene is non-zero) float64 [K, genes]
GeneStatistics = namedtuple("GeneStatistics", ["cells", "mean", "var", "detected"])

# compare_cells: the real cells' and the generated cells' GeneStatistics, same groups
CellComparison = namedtuple("CellComparison", ["real", "generated"])

# one row of comparison_summary per group
GroupSummary = namedtuple("GroupSummary", [
    "group", "real_cells", "generated_cells", "real_library_size", "generated_library_size",
    "real_genes_detected", "generated_genes_detected", "log1p_mean_r", "detected_r"])


def statistics_from_sums(cells, s1, s2, nonzero):
    """GeneStatistics of K groups from their cell counts n [K] and per-gene sums S1 = sum v,
    S2 = sum v^2 and nonzero counts [K, genes]:
        mean = S1 / n,  var = max(S2 - S1 * S1 / n, 0) / (n - 1),  detected = nonzero / n
    var is NaN for n <= 1, every value NaN for an empty group.  Every path (the dense
    definitions and the streamed device passes) ends here, so they agree bit for bit whenever
    their sums do."""
    n = np.array(cells, dtype=np.int64).reshape(-1)
    s1 = np.asarray(s1, dtype=np.float64)
    s2 = np.asarray(s2, dtype=np.float64)
    nz = np.asarray(nonzero, dtype=np.int64)
    if s1.ndim != 2 or s1.shape[0] != len(n) or s2.shape != s1.shape or nz.shape != s1.shape:
        raise ValueError("statistics_from_sums: cells is [K] and the sums are [K, genes]")
    nn = n.astype(np.float64)[:, None]
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = s1 / nn
        var = np.maximum(s2 - s1 * s1 / nn, 0.0) / (nn - 1)
        detected = nz / nn
    var[n <= 1] = np.nan
    mean[n == 0] = np.nan
    detected[n == 0] = np.nan
    return GeneStatistics(n, mean, var, detected)


def group_labels(groups, n_groups, n):
    """(int64 labels [n], K) of gene_statistics' grouping: groups=None puts every cell in group
    0 (K = n_groups or 1); otherwise one integer label in [0, K) per cell, K = n_groups or
    max(label) + 1."""
    if groups is None:
        labels = np.zeros(n, dtype=np.int64)
        K = 1 if n_groups is None else int(n_groups)
    else:
        labels = np.asarray(groups)
        if labels.ndim != 1 or len(labels) != n:
            raise ValueError(f"groups must hold one label per cell ({n}), got shape "
                             f"{labels.shape}")
        if len(labels) and not np.issubdtype(labels.dtype, np.integer):
            raise ValueError(f"groups must be integer labels, got {labels.dtype}")
        labels = labels.astype(np.int64)
        K = int(n_groups) if n_groups is not None else (int(labels.max()) + 1 if n else 1)
        if n and (labels.min() < 0 or labels.max() >= K):
            raise ValueError(f"group labels must lie in [0, {K})")
    if K < 1:
        raise ValueError(f"n_groups must be at least 1, got {K}")
    return labels, K


def require_sorted(labels):
    """generated_gene_statistics streams its rows in order: each group must be one run."""
    if np.any(np.diff(labels) < 0):
        raise ValueError("generated_gene_statistics: rows must be sorted by group")


def _pearson(a, b):
    """Pearson r of two vectors in fp64; NaN when either holds a NaN or is constant."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if len(a) < 2 or np.isnan(a).any() or np.isnan(b).any():
        return float("nan")
    da, db = a - a.mean(), b - b.mean()
    den = np.sqrt(np.dot(da, da) * np.dot(db, db))
    return float(np.dot(da, db) / den) if den > 0 else float("nan")


def comparison_summary(comparison):
    """One GroupSummary per group of a CellComparison: the real and generated cell counts, the
    mean library size (sum over genes of the mean count), the mean number of genes detected
    per cell (sum over genes of the detection rate), and the Pearson r over genes, real vs
    generated, of log1p(mean) and of the detection rate.  NaN where a group is empty or a
    vector is constant."""
    real, gen = comparison
    rows = []
    with np.errstate(invalid="ignore"):
        for k in range(len(real.cells)):
            rows.append(GroupSummary(
                k, int(real.cells[k]), int(gen.cells[k]),
                float(np.sum(real.mean[k])), float(np.sum(gen.mean[k])),
                float(np.sum(real.detected[k])), float(np.sum(gen.detected[k])),
                _pearson(np.log1p(real.mean[k]), np.log1p(gen.mean[k])),
                _pearson(real.detected[k], gen.detected[k])))
    return rows


# two_sample_test, per group k: the cells tested on each side (int64 [K]), the lower median of
# the pooled squared distances (float64 [K]), MMD^2 and its permutation p-value per bandwidth
# scale of MMD_SCALES (float64 [K, 3]), and the Kolmogorov-Smirnov D of the per-cell library
# size and genes detected, real against generated (float64 [K])
TwoSampleTest = namedtuple("TwoSampleTest", [
    "real_cells", "generated_cells", "sqdist_median", "mmd2", "p_value", "library_size_ks",
    "genes_detected_ks"])

MMD_SCALES = (0.5, 1.0, 2.0)      # kernel bandwidths s * median
MAX_TEST_CELLS = 16384            # per group and side: bounds the [2n, 2n] Gram matrix


def mmd_from_sums(n, xx, yy, xy):
    """Unbiased MMD^2 of two samples of n cells each from their kernel sums over ordered pairs
    i != j: XX (both in X), YY (both in Y), XY (i in X, j in Y):
        XX / (n (n - 1)) + YY / (n (n - 1)) - 2 XY / n^2
    Every path (the dense definition and the streamed device pass) ends here."""
    n = float(n)
    xx, yy, xy = (np.asarray(v, dtype=np.float64) for v in (xx, yy, xy))
    return xx / (n * (n - 1)) + yy / (n * (n - 1)) - 2.0 * xy / (n * n)


def permutation_p_value(mmd2):
    """p = (1 + #{p >= 1 : MMD^2_p >= MMD^2_0}) / L over the first axis of mmd2 ([L, ...]):
    labelling 0 is the observed one, 1..L-1 the permutations."""
    mmd2 = np.asarray(mmd2, dtype=np.float64)
    return (1.0 + np.sum(mmd2[1:] >= mmd2[0], axis=0)) / len(mmd2)


def ks_statistic(a, b):
    """Two-sample Kolmogorov-Smirnov statistic D = max |F_a - F_b| of the empirical CDFs."""
    a = np.sort(np.asarray(a, dtype=np.float64))
    b = np.sort(np.asarray(b, dtype=np.float64))
    if len(a) == 0 or len(b) == 0:
        return float("nan")
    v = np.concatenate([a, b])
    fa = np.searchsorted(a, v, side="right") / len(a)
    fb = np.searchsorted(b, v, side="right") / len(b)
    return float(np.max(np.abs(fa - fb)))


def bf16_round(x):
    """float32 -> the float32 value of its bf16 rounding, half to even; NaN stays NaN."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    r = ((u.astype(np.uint64) + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint32)
    r = np.where(nan, (u >> 16) | 0x40, r)
    return (r << 16).astype(np.uint32).view(np.float32)


def log1p_features(v):
    """The test's per-gene feature bf16(float32(log1p(float64(v))))."""
    return bf16_round(np.log1p(np.asarray(v, dtype=np.float64)).astype(np.float32))


def two_sample_args(max_cells, permutations, seed):
    """Checked (max_cells, permutations, seed) of two_sample_test."""
    max_cells, permutations, seed = int(max_cells), int(permutations), int(seed)
    if not 2 <= max_cells <= MAX_TEST_CELLS:
        raise ValueError(f"max_cells must lie in [2, {MAX_TEST_CELLS}], got {max_cells}")
    if permutations < 0:
        raise ValueError(f"permutations must be >= 0, got {permutations}")
    if seed < 0:
        raise ValueError(f"seed must be >= 0, got {seed}")
    return max_cells, permutations, seed


def two_sample_cells(labels, K, max_cells, seed):
    """Per group k, the real cells two_sample_test takes (row numbers, ascending): all of the
    group's cells, or max_cells of them drawn with default_rng([seed, 0, k]) and sorted."""
    picks = []
    for k in range(K):
        rows = np.flatnonzero(labels == k).astype(np.int64)
        if len(rows) > max_cells:
            rows = rows[np.sort(np.random.default_rng([seed, 0, k]).choice(
                len(rows), max_cells, replace=False))]
        picks.append(rows)
    return picks


def two_sample_labellings(n, permutations, seed, k):
    """bool [permutations + 1, 2n]: row 0 puts the first n pooled cells in X, row p >= 1 the
    cells rng.permutation(2n)[:n], drawn in order from rng = default_rng([seed, 1, k])."""
    N = 2 * n
    out = np.zeros((permutations + 1, N), dtype=bool)
    out[0, :n] = True
    rng = np.random.default_rng([seed, 1, k])
    for p in range(1, permutations + 1):
        out[p, rng.permutation(N)[:n]] = True
    return out


def pack_labellings(labellings):
    """bool [L, N] -> uint32 [L, ceil(N / 32)]: bit i % 32 of word i // 32 is cell i."""
    L, N = labellings.shape
    W = (N + 31) // 32
    padded = np.zeros((L, W * 32), dtype=bool)
    padded[:, :N] = labellings
    return np.packbits(padded, axis=1, bitorder="little").view("<u4").astype(np.uint32)


def kernel_sums(d2, masks, scale_bandwidths):
    """Definition of the kernel sums: fp64 [L, len(scale_bandwidths), 3] of XX, YY, XY per
    labelling (bool masks [L, N], True = X) with k = exp(-d2 / h) for every h, summed over
    ordered pairs i != j."""
    d2 = np.asarray(d2, dtype=np.float64)
    B = np.asarray(masks, dtype=np.float64)
    out = np.empty((len(B), len(scale_bandwidths), 3))
    for b, h in enumerate(scale_bandwidths):
        k = np.exp(-d2 / h)
        np.fill_diagonal(k, 0.0)
        r = k.sum(1)
        xx = np.einsum("pi,ip->p", B, k @ B.T)
        rb = B @ r
        out[:, b, 0] = xx
        out[:, b, 1] = r.sum() - 2.0 * rb + xx
        out[:, b, 2] = rb - xx
    return out


def lower_median(values):
    v = np.sort(np.asarray(values).reshape(-1))
    return float(v[(len(v) - 1) // 2]) if len(v) else float("nan")


def two_sample_result(counts, medians, sums, lib, det):
    """TwoSampleTest from per-group cell counts n_k, medians, kernel sums ([L, 3, 3] or None for
    a group without a test) and (real, generated) pairs of per-cell library sizes and genes
    detected.  Every path ends here."""
    K = len(counts)
    n = np.asarray(counts, dtype=np.int64)
    med = np.full(K, np.nan)
    mmd2 = np.full((K, len(MMD_SCALES)), np.nan)
    p = np.full((K, len(MMD_SCALES)), np.nan)
    lib_ks = np.full(K, np.nan)
    det_ks = np.full(K, np.nan)
    for k in range(K):
        if n[k] < 2:
            continue
        med[k] = medians[k]
        lib_ks[k] = ks_statistic(*lib[k])
        det_ks[k] = ks_statistic(*det[k])
        if sums[k] is not None and med[k] > 0:
            stats = mmd_from_sums(n[k], sums[k][..., 0], sums[k][..., 1], sums[k][..., 2])
            mmd2[k] = stats[0]
            p[k] = permutation_p_value(stats)
    return TwoSampleTest(n, n.copy(), med, mmd2, p, lib_ks, det_ks)


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

    def gene_statistics(self, cell_data, groups=None, n_groups=None):
        """Per-group, per-gene statistics of cells -> GeneStatistics (statistics_from_sums):
        groups holds one integer label in [0, K) per cell (K = n_groups or max + 1; None: one
        group).  This is the definition, fp64 numpy over the dense cells; engine-backed
        subclasses stream the same sums without a dense (n, genes) intermediate."""
        x = np.asarray(cell_data, dtype=np.float64)
        if x.ndim != 2:
            raise ValueError(f"expected cells of shape (n, genes), got {x.shape}")
        labels, K = group_labels(groups, n_groups, len(x))
        s1 = np.zeros((K, x.shape[1]))
        s2 = np.zeros((K, x.shape[1]))
        nz = np.zeros((K, x.shape[1]), dtype=np.int64)
        for k in range(K):
            rows = x[labels == k]
            s1[k] = rows.sum(0)
            s2[k] = (rows * rows).sum(0)
            nz[k] = np.count_nonzero(rows, axis=0)
        return statistics_from_sums(np.bincount(labels, minlength=K), s1, s2, nz)

    def generated_gene_statistics(self, encoding_in, random_in=None, groups=None,
                                  n_groups=None):
        """gene_statistics(generate_cells(encoding_in, random_in), groups, n_groups); the rows
        must already be sorted by group (ValueError otherwise, before anything is drawn).
        random_in=None draws the noise as generate_cells does.  This is the definition;
        engine-backed subclasses stream the generator instead."""
        labels, K = group_labels(groups, n_groups, len(encoding_in))
        require_sorted(labels)
        return self.gene_statistics(self.generate_cells(encoding_in, random_in), labels, K)

    def compare_cells(self, cell_data):
        """Real cells against as many generated ones, per group -> CellComparison.  The groups
        come from _comparison_groups (one group here and in the continuous variant; the
        classify variant groups by the encoder's class).  Group k generates as many cells as it
        has real ones, in group order, with the encodings of _comparison_encodings drawn first
        and then random_uniform_vector(total) for the noise, so a restored checkpoint always
        gives the same numbers."""
        labels, K = self._comparison_groups(cell_data)
        real = self.gene_statistics(cell_data, labels, K)
        encodings = self._comparison_encodings(real.cells)
        noise = self.random_uniform_vector(len(encodings))
        generated = self.generated_gene_statistics(
            encodings, noise, np.repeat(np.arange(K, dtype=np.int64), real.cells), K)
        return CellComparison(real, generated)

    def _comparison_groups(self, cell_data):
        """-> (int64 group label per cell, K) for compare_cells: every cell in one group."""
        return np.zeros(len(cell_data), dtype=np.int64), 1

    def _comparison_encodings(self, counts):
        """Generated-cell encodings for compare_cells, counts[k] of them for group k in group
        order: random_encoding_vector over all of them."""
        return self.random_encoding_vector(int(np.sum(counts)))

    def two_sample_test(self, cell_data, max_cells=4096, permutations=1000, seed=0):
        """Kernel two-sample test of real against generated cells, per group -> TwoSampleTest.
        Groups come from _comparison_groups.  Group k tests its real cells (max_cells of them,
        two_sample_cells, when it has more) against as many generated ones; the generated
        cells are drawn as compare_cells draws them (_comparison_encodings for every group,
        then random_uniform_vector(total), generate_cells).  Per cell, the features are
        log1p_features(v) over genes (v the count; the generator's rounded output), and the
        pooled Gram matrix G = F F^T (real cells first) gives d2_ij = max(G_ii + G_jj - 2 G_ij,
        0).  With m the lower median of d2 over i < j, MMD^2 (mmd_from_sums) is taken for
        k(i, j) = exp(-d2_ij / (s m)), s in MMD_SCALES, on the observed split and on
        `permutations` random ones (two_sample_labellings), giving permutation_p_value.  KS D
        of the library size and genes detected per cell closes the result.  Groups with fewer
        than 2 cells report their counts and NaN; a zero median gives NaN MMD^2 and p.  The
        subsample and labellings are seeded from `seed` alone.  This is the definition, dense
        fp64 numpy; engine-backed subclasses stream it on the device."""
        max_cells, permutations, seed = two_sample_args(max_cells, permutations, seed)
        x = np.asarray(cell_data, dtype=np.float64)
        if x.ndim != 2:
            raise ValueError(f"expected cells of shape (n, genes), got {x.shape}")
        if np.any(x < 0):
            raise ValueError("two_sample_test: the cells hold negative counts")
        labels, K = self._comparison_groups(cell_data)
        picks = two_sample_cells(labels, K, max_cells, seed)
        counts = [len(p) for p in picks]
        encodings = self._comparison_encodings(counts)
        noise = self.random_uniform_vector(len(encodings))
        generated = np.asarray(self.generate_cells(encodings, noise), dtype=np.float64)
        medians, sums, lib, det = [], [], [], []
        off = 0
        for k in range(K):
            n = counts[k]
            real, gen = x[picks[k]], generated[off:off + n]
            off += n
            lib.append((real.sum(1), gen.sum(1)))
            det.append((np.count_nonzero(real, axis=1), np.count_nonzero(gen, axis=1)))
            if n < 2:
                medians.append(np.nan)
                sums.append(None)
                continue
            F = np.concatenate([log1p_features(real), log1p_features(gen)]).astype(np.float64)
            G = F @ F.T
            g = np.diag(G)
            d2 = np.maximum(g[:, None] + g[None, :] - 2.0 * G, 0.0)
            m = lower_median(d2[np.triu_indices(2 * n, 1)])
            medians.append(m)
            sums.append(kernel_sums(d2, two_sample_labellings(n, permutations, seed, k),
                                    [s * m for s in MMD_SCALES]) if m > 0 else None)
        return two_sample_result(counts, medians, sums, lib, det)

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
