"""Comparing generated cells with real ones, without a GPU: statistics_from_sums, the
definitions of gene_statistics / generated_gene_statistics / compare_cells on mocked
components, the grouping and draw order of both variants, comparison_summary, the CSV writers
and the `compare` command's argument checks."""
import os
from unittest.mock import MagicMock

import numpy as np
import pytest

from cellcomm_b200.bigan_basic import (BasicBiGan, CellComparison, GeneStatistics,
                                       comparison_summary, statistics_from_sums)
from cellcomm_b200.cell_type_training import CellMatrix


def _same(a, b):
    """bit-identical GeneStatistics (NaN included)"""
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and x.shape == y.shape
        assert x.tobytes() == y.tobytes()


# ------------------------------------------------------------------ statistics_from_sums
def test_statistics_hand_case():
    # group 0: genes over cells [1, 2, 3] and [0, 0, 4]; group 1: one cell [5, 0]
    s = statistics_from_sums([3, 1], [[6.0, 4.0], [5.0, 0.0]], [[14.0, 16.0], [25.0, 0.0]],
                             [[3, 1], [1, 0]])
    assert isinstance(s, GeneStatistics)
    assert s.cells.dtype == np.int64 and s.mean.dtype == np.float64
    np.testing.assert_array_equal(s.cells, [3, 1])
    np.testing.assert_array_equal(s.mean[0], [2.0, 4.0 / 3])
    np.testing.assert_array_equal(s.var[0], [1.0, (16.0 - 16.0 / 3) / 2])
    np.testing.assert_array_equal(s.detected[0], [1.0, 1.0 / 3])
    np.testing.assert_array_equal(s.mean[1], [5.0, 0.0])
    np.testing.assert_array_equal(s.detected[1], [1.0, 0.0])
    assert np.isnan(s.var[1]).all()                         # n = 1: no unbiased variance


def test_statistics_empty_group_is_nan_and_variance_is_clamped():
    s1 = np.array([[0.0, 0.0], [0.3, 0.1 + 0.2]])
    s2 = np.array([[0.0, 0.0], [0.03 - 1e-18, 0.09 / 3 * 0.999]])   # S2 < S1^2 / n: clamp
    s = statistics_from_sums([0, 3], s1, s2, np.array([[0, 0], [3, 3]]))
    for a in (s.mean, s.var, s.detected):
        assert np.isnan(a[0]).all()
    assert np.all(s.var[1] == 0.0)
    with pytest.raises(ValueError, match=r"\[K, genes\]"):
        statistics_from_sums([1], [[1.0]], [[1.0, 2.0]], [[1]])


# ------------------------------------------------------------------ the definitions
class _Basic(BasicBiGan):
    def random_encoding_vector(self, n):
        return self._prior_rng.random((n, self.encoding_size), dtype=np.float32)

    def trainings_step(self, batch):
        pass


def _generate(inputs):
    """a generator whose output depends on both inputs, with halves, negatives and -0.4"""
    z, r = (np.asarray(a, dtype=np.float32) for a in inputs)
    base = np.array([0.5, 1.5, 2.5, -0.4, 3.0], np.float32)
    return (base[None, :] * (1 + 2 * z[:, :1]) + 4 * r[:, :1]).astype(np.float32)


def _mocked(encode=None, Z=2, G=5, cls=_Basic, **kw):
    comps = [MagicMock() for _ in range(3)]
    comps[0].predict = MagicMock(side_effect=_generate)
    comps[1].predict = MagicMock(side_effect=encode)
    net = cls(Z, G, *(MagicMock(return_value=c) for c in comps), **kw)
    net._prior_rng = np.random.default_rng(5)
    return net, comps


def _numpy_statistics(x, labels, K):
    out = []
    for k in range(K):
        rows = x[labels == k]
        n = len(rows)
        with np.errstate(divide="ignore", invalid="ignore"):
            mean = rows.sum(0) / n
            var = np.maximum((rows * rows).sum(0) - rows.sum(0) ** 2 / n, 0) / (n - 1)
            det = (rows != 0).sum(0) / n
        if n <= 1:
            var[:] = np.nan
        out.append((n, mean, var, det))
    return out


def test_gene_statistics_definition_groups_and_counts():
    net, _ = _mocked()
    rng = np.random.default_rng(0)
    x = rng.integers(0, 4, (20, 5)).astype(np.float64)
    labels = rng.integers(0, 3, 20)
    labels[labels == 1] = 0                                   # group 1 is empty
    labels[0] = 3                                             # group 3 has one cell
    s = net.gene_statistics(x, labels, 5)                     # group 4: empty, by n_groups
    assert s.mean.shape == (5, 5)
    for k, (n, mean, var, det) in enumerate(_numpy_statistics(x, labels, 5)):
        assert s.cells[k] == n
        np.testing.assert_array_equal(s.mean[k], mean)
        np.testing.assert_array_equal(s.var[k], var)
        np.testing.assert_array_equal(s.detected[k], det)
    assert np.isnan(s.mean[1]).all() and np.isnan(s.mean[4]).all() and np.isnan(s.var[3]).all()
    # None: one group; a CellMatrix is read as its dense cells
    _same(net.gene_statistics(x), net.gene_statistics(CellMatrix.from_dense(x), np.zeros(20, int)))
    with pytest.raises(ValueError, match="one label per cell"):
        net.gene_statistics(x, labels[:5])
    with pytest.raises(ValueError, match=r"\[0, 2\)"):
        net.gene_statistics(x, labels, 2)
    with pytest.raises(ValueError, match="integer"):
        net.gene_statistics(x, labels.astype(np.float64))


def test_minus_zero_is_not_detected():
    net, _ = _mocked()
    s = net.gene_statistics(np.array([[-0.0, 1.0], [0.0, -0.0]]))
    np.testing.assert_array_equal(s.detected[0], [0.0, 0.5])


def test_generated_gene_statistics_is_the_composed_definition():
    net, comps = _mocked()
    enc = np.random.default_rng(1).random((9, 2), dtype=np.float32)
    r = np.random.default_rng(2).random((9, 2), dtype=np.float32)
    groups = np.array([0, 0, 0, 2, 2, 2, 2, 2, 2])
    got = net.generated_gene_statistics(enc, r, groups, 3)
    _same(got, net.gene_statistics(net.generate_cells(enc, r), groups, 3))
    assert np.isnan(got.mean[1]).all()
    # the cells are rounded half to even: 0.5 -> 0, 2.5 -> 2, -0.4 -> -0.0 (not detected)
    zero = np.zeros((1, 2), np.float32)
    s = net.generated_gene_statistics(zero, zero)
    np.testing.assert_array_equal(s.mean[0], [0.0, 2.0, 2.0, 0.0, 3.0])
    np.testing.assert_array_equal(s.detected[0], [0.0, 1.0, 1.0, 0.0, 1.0])


def test_generated_gene_statistics_rejects_unsorted_rows_before_drawing():
    net, comps = _mocked()
    net.random_uniform_vector = MagicMock(side_effect=AssertionError("drew noise"))
    with pytest.raises(ValueError, match="sorted by group"):
        net.generated_gene_statistics(np.zeros((3, 2), np.float32), None, [0, 1, 0])
    assert not comps[0].predict.called


def test_generated_gene_statistics_draws_like_generate_cells():
    net, comps = _mocked()
    state = net._prior_rng.bit_generator.state
    net.generated_gene_statistics(np.zeros((4, 2), np.float32))
    g = np.random.default_rng()
    g.bit_generator.state = state
    np.testing.assert_array_equal(comps[0].predict.call_args[0][0][1],
                                  g.random((4, 2), dtype=np.float32))


# ------------------------------------------------------------------ compare_cells
def _draws(state, *shapes):
    g = np.random.default_rng()
    g.bit_generator.state = state
    return [g.random(s, dtype=np.float32) for s in shapes]


def test_basic_compare_cells_one_group_encodings_then_noise():
    net, comps = _mocked()
    x = np.random.default_rng(3).integers(0, 3, (6, 5)).astype(np.float64)
    state = net._prior_rng.bit_generator.state
    c = net.compare_cells(x)
    assert isinstance(c, CellComparison)
    enc, noise = _draws(state, (6, 2), (6, 2))
    z, r = comps[0].predict.call_args[0][0]
    np.testing.assert_array_equal(z, enc)
    np.testing.assert_array_equal(r, noise)
    _same(c.real, net.gene_statistics(x))
    _same(c.generated, net.gene_statistics(np.round(_generate((enc, noise)))))
    np.testing.assert_array_equal(c.real.cells, [6])
    np.testing.assert_array_equal(c.generated.cells, [6])


def _classify(encode, Z=3):
    from cellcomm_b200.bigan_classify import ClassifyCellBiGan
    return _mocked(encode, Z=Z, cls=ClassifyCellBiGan)


def test_classify_compare_cells_groups_by_argmax_and_generates_one_hot():
    pred = np.array([[0.1, 0.7, 0.2], [0.5, 0.5, 0.0], [0.2, 0.2, 0.6], [0.0, 0.9, 0.9],
                     [0.3, 0.3, 0.3], [0.1, 0.8, 0.1], [0.0, 1.0, 0.0]], np.float32)
    net, comps = _classify(lambda cells: pred)
    assert net._engine is None
    x = np.random.default_rng(4).integers(0, 5, (7, 5)).astype(np.float64)
    np_state = np.random.get_state()
    state = net._prior_rng.bit_generator.state
    c = net.compare_cells(x)
    groups = np.argmax(pred, -1)                              # ties: the first maximum
    np.testing.assert_array_equal(groups, [1, 0, 2, 1, 0, 1, 1])
    np.testing.assert_array_equal(c.real.cells, [2, 4, 1])
    np.testing.assert_array_equal(c.generated.cells, c.real.cells)
    _same(c.real, net.gene_statistics(x, groups, 3))
    z, r = comps[0].predict.call_args[0][0]
    np.testing.assert_array_equal(z, np.eye(3, dtype=np.float32)[[0, 0, 1, 1, 1, 1, 2]])
    (noise,) = _draws(state, (7, 3))                          # the encodings draw nothing
    np.testing.assert_array_equal(r, noise)
    assert np.random.get_state()[1].tobytes() == np_state[1].tobytes()
    _same(c.generated, net.gene_statistics(np.round(_generate((z, noise))),
                                           [0, 0, 1, 1, 1, 1, 2], 3))


def test_classify_compare_cells_keeps_empty_classes():
    net, comps = _classify(lambda cells: np.tile([[0.0, 0.0, 1.0]], (len(cells), 1)))
    c = net.compare_cells(np.ones((4, 5)))
    np.testing.assert_array_equal(c.real.cells, [0, 0, 4])
    np.testing.assert_array_equal(c.generated.cells, [0, 0, 4])
    assert np.isnan(c.generated.mean[:2]).all() and not np.isnan(c.generated.mean[2]).any()


def test_continuous_variant_compares_one_group_with_random_encodings():
    from cellcomm_b200.bigan_cont import ContinuousCellBiGan
    assert ContinuousCellBiGan._comparison_groups is BasicBiGan._comparison_groups
    assert ContinuousCellBiGan._comparison_encodings is BasicBiGan._comparison_encodings
    net = ContinuousCellBiGan.__new__(ContinuousCellBiGan)
    net.encoding_size = 2
    net._prior_rng = np.random.default_rng(8)
    state = net._prior_rng.bit_generator.state
    labels, K = net._comparison_groups(np.zeros((5, 4)))
    assert K == 1 and labels.tolist() == [0] * 5
    (enc,) = _draws(state, (5, 2))
    np.testing.assert_array_equal(net._comparison_encodings(np.array([5])), enc)


# ------------------------------------------------------------------ comparison_summary
def test_comparison_summary_rows():
    real = statistics_from_sums([4, 0, 2], [[4.0, 8.0, 0.0], [0, 0, 0], [2.0, 2.0, 2.0]],
                                [[4.0, 20.0, 0.0], [0, 0, 0], [2.0, 2.0, 2.0]],
                                [[4, 3, 0], [0, 0, 0], [2, 2, 2]])
    gen = statistics_from_sums([4, 0, 2], [[8.0, 4.0, 4.0], [0, 0, 0], [0.0, 2.0, 6.0]],
                               [[16.0, 8.0, 4.0], [0, 0, 0], [0.0, 2.0, 18.0]],
                               [[4, 2, 1], [0, 0, 0], [0, 2, 2]])
    rows = comparison_summary(CellComparison(real, gen))
    assert [r.group for r in rows] == [0, 1, 2]
    r0 = rows[0]
    assert (r0.real_cells, r0.generated_cells) == (4, 4)
    assert r0.real_library_size == 3.0 and r0.generated_library_size == 4.0
    assert r0.real_genes_detected == 1.75 and r0.generated_genes_detected == 1.75
    a, b = np.log1p([1.0, 2.0, 0.0]), np.log1p([2.0, 1.0, 1.0])
    assert r0.log1p_mean_r == pytest.approx(np.corrcoef(a, b)[0, 1], rel=1e-12)
    assert r0.detected_r == pytest.approx(np.corrcoef([1, 0.75, 0], [1, 0.5, 0.25])[0, 1],
                                          rel=1e-12)
    assert rows[1].real_cells == 0 and all(np.isnan(v) for v in rows[1][3:])
    assert np.isnan(rows[2].log1p_mean_r) and np.isnan(rows[2].detected_r)  # real is constant


# ------------------------------------------------------------------ the CSV writers
def _comparison(K=2, G=4, seed=0):
    rng = np.random.default_rng(seed)

    def stats():
        n = rng.integers(2, 9, K)
        return GeneStatistics(n, rng.random((K, G)) * 1e3, rng.random((K, G)) / 3, rng.random((K, G)))
    c = CellComparison(stats(), stats())
    c.real.var[0, 1] = np.nan
    c.generated.mean[1, 0] = 0.1 + 0.2
    return c


def test_gene_file_rows_round_trip_float64(tmp_path):
    from cellcomm_b200.__main__ import GENE_COLUMNS, write_gene_file
    c = _comparison()
    genes = np.array([3, 7, 11, 40])
    path = write_gene_file(str(tmp_path / "genes.csv"), genes, c)
    lines = open(path).read().splitlines()
    assert lines[0] == ",".join(GENE_COLUMNS) == ("group,gene,real-mean,real-var,real-detected,"
                                                   "generated-mean,generated-var,generated-detected")
    assert len(lines) == 1 + 2 * 4
    got = np.array([[float(v) for v in line.split(",")] for line in lines[1:]])
    np.testing.assert_array_equal(got[:, 0], [0] * 4 + [1] * 4)
    np.testing.assert_array_equal(got[:, 1], np.tile(genes, 2))
    assert lines[1].split(",")[:2] == ["0", "3"]
    for j, a in enumerate((c.real.mean, c.real.var, c.real.detected, c.generated.mean,
                           c.generated.var, c.generated.detected)):
        assert got[:, 2 + j].tobytes() == a.reshape(-1).tobytes()
    assert lines[2].split(",")[3] == "nan"
    assert lines[5].split(",")[5] == "%.17g" % (0.1 + 0.2)
    assert sorted(os.listdir(tmp_path)) == ["genes.csv"]


def test_group_file_rows(tmp_path):
    from cellcomm_b200.__main__ import GROUP_COLUMNS, write_group_file
    rows = comparison_summary(_comparison(K=3, seed=1))
    path = write_group_file(str(tmp_path / "groups.csv"), rows)
    lines = open(path).read().splitlines()
    assert lines[0] == ",".join(GROUP_COLUMNS)
    assert len(lines) == 4
    for line, row in zip(lines[1:], rows):
        f = line.split(",")
        assert f[:3] == [str(row.group), str(row.real_cells), str(row.generated_cells)]
        got = np.array([float(v) for v in f[3:]])
        assert got.tobytes() == np.array(row[3:], dtype=np.float64).tobytes()


def test_gene_file_write_is_atomic(tmp_path):
    from cellcomm_b200.__main__ import write_gene_file
    target = tmp_path / "genes.csv"
    target.write_text("old\n")

    class Boom(Exception):
        pass

    class Failing:
        def __iter__(self):
            yield 1
            raise Boom()

    with pytest.raises(Boom):
        write_gene_file(str(target), Failing(), _comparison())
    assert target.read_text() == "old\n"
    assert sorted(os.listdir(tmp_path)) == ["genes.csv"]


# ------------------------------------------------------------------ the compare command
def _main(*args):
    from cellcomm_b200.__main__ import main
    main(["", "compare", *args])


def _meta_checkpoint(path, gene_size, variant="cont"):
    np.savez(path, **{"meta/variant": variant, "meta/encoding_size": 3,
                      "meta/gene_size": gene_size})
    return str(path)


def _source(tmp_path, genes, name="source.mtx"):
    return CellMatrix.from_dense(np.ones((2, genes))).to_mtx(str(tmp_path / name))


@pytest.mark.parametrize("args", [(), ("a.npz", "b.mtx", "c.mtx"),
                                  ("a.npz", "b.mtx", "c.mtx", "out", "extra")])
def test_compare_command_wants_four_parameters(args):
    with pytest.raises(AssertionError, match="compare <checkpoint.npz> <source-matrix-file> "
                                             "<matrix-file> <output-dir>"):
        _main(*args)


def _no_network(monkeypatch):
    import cellcomm_b200.bigan_cont as cont
    built = MagicMock(side_effect=AssertionError("a network was built"))
    monkeypatch.setattr(cont, "ContinuousCellBiGan", built)
    return built


def test_compare_command_rejects_gene_count_mismatch(tmp_path, monkeypatch):
    built = _no_network(monkeypatch)
    ckpt = _meta_checkpoint(tmp_path / "c.npz", 5)
    cells = _source(tmp_path, 5, "cells.mtx")
    with pytest.raises(ValueError, match="compares 5 genes.*has 4"):
        _main(ckpt, _source(tmp_path, 4), cells, str(tmp_path / "out"))
    assert not built.called
    assert not os.path.exists(tmp_path / "out")


@pytest.mark.parametrize("missing", [0, 1, 2])
def test_compare_command_rejects_a_missing_file(tmp_path, monkeypatch, missing):
    built = _no_network(monkeypatch)
    args = [_meta_checkpoint(tmp_path / "c.npz", 4), _source(tmp_path, 4),
            _source(tmp_path, 4, "cells.mtx")]
    args[missing] = str(tmp_path / "nowhere")
    with pytest.raises(FileNotFoundError, match="nowhere"):
        _main(*args, str(tmp_path / "out"))
    assert not built.called
    assert not os.path.exists(tmp_path / "out")
