"""Cell scores without a GPU: CellMatrix.reindex_columns against dense numpy, the definition of
BasicBiGan.score_cells on mocked components, the `score` command's argument checks and CSV
writer, and the validation.csv interceptor."""
import os
from types import SimpleNamespace
from unittest.mock import MagicMock

import numpy as np
import pytest

from cellcomm_b200.bigan_basic import BasicBiGan, CellScores
from cellcomm_b200.cell_type_training import CellMatrix


def _assert_same(a, b):
    for name in ("rowptr", "colidx", "index", "columns"):
        np.testing.assert_array_equal(getattr(a, name), getattr(b, name), err_msg=name)
        assert getattr(a, name).dtype == getattr(b, name).dtype, name
    assert a.values64.tobytes() == b.values64.tobytes()      # bit-exact float64


def _reindexed_dense(dense, columns, new_columns):
    """DataFrame.reindex(columns=new_columns, fill_value=0) in numpy"""
    out = np.zeros((dense.shape[0], len(new_columns)), dtype=np.float64)
    where = {c: j for j, c in enumerate(columns)}
    for k, c in enumerate(new_columns):
        if c in where:
            out[:, k] = dense[:, where[c]]
    return out


# ------------------------------------------------------------------ reindex_columns
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_reindex_columns_matches_dense_reindex(seed):
    rng = np.random.default_rng(seed)
    rows, cols = 40, 60
    dense = np.where(rng.random((rows, cols)) < 0.3, rng.integers(1, 500, (rows, cols)), 0)
    dense = dense.astype(np.float64)
    dense[3] = 0.0                                   # an empty row
    dense[7, :5] = [0.1 + 0.2, 1e-300, 2.0 ** 40, 7.5, 3.0]   # awkward doubles
    columns = np.sort(rng.choice(np.arange(1, 200), cols, replace=False))
    m = CellMatrix.from_dense(dense, index=np.arange(rows) * 2 + 5, columns=columns)
    # keep some genes, drop others, add genes the matrix does not have (also past both ends)
    new = np.union1d(rng.choice(columns, cols // 2, replace=False),
                     np.concatenate([[0], rng.integers(1, 250, 20), [999]]))
    got = m.reindex_columns(new)
    want = CellMatrix.from_dense(_reindexed_dense(dense, columns, new), index=m.index,
                                 columns=new)
    _assert_same(got, want)
    assert got.values32.tobytes() == want.values32.tobytes()


def test_reindex_columns_keeps_explicit_zeros_and_trailing_empty_rows():
    # gene 5: explicit zero in row 0; the last two rows are empty
    m = CellMatrix.from_coo([5, 7, 9, 7], [1, 1, 2, 2], [0.0, 2.0, 3.0, 4.0])
    m = CellMatrix(np.concatenate([m.rowptr, [m.nnz, m.nnz]]), m.colidx, m.values64,
                   [1, 2, 3, 4], m.columns)
    got = m.reindex_columns([5, 6, 7])
    np.testing.assert_array_equal(got.rowptr, [0, 2, 3, 3, 3])
    np.testing.assert_array_equal(got.colidx, [0, 2, 2])
    np.testing.assert_array_equal(got.values64, [0.0, 2.0, 4.0])
    np.testing.assert_array_equal(got.to_numpy(), _reindexed_dense(m.to_numpy(), m.columns,
                                                                   [5, 6, 7]))
    same = m.reindex_columns(m.columns)
    _assert_same(same, m)
    empty = m.reindex_columns(np.zeros(0, np.int64))
    assert empty.shape == (4, 0) and empty.nnz == 0


@pytest.mark.parametrize("bad", [[3, 2, 5], [1, 1, 2], [[1, 2]]])
def test_reindex_columns_rejects_non_ascending_ids(bad):
    m = CellMatrix.from_dense(np.ones((2, 3)))
    with pytest.raises(ValueError, match="ascending"):
        m.reindex_columns(bad)


# ------------------------------------------------------------------ the definition
class _Basic(BasicBiGan):
    def random_encoding_vector(self, n):
        return np.zeros((n, 2), np.float32)

    def trainings_step(self, batch):
        pass


def _mocked(enc, pred, d):
    gen, encoder, disc = MagicMock(), MagicMock(), MagicMock()
    encoder.predict = MagicMock(return_value=enc)
    gen.predict = MagicMock(return_value=pred)
    disc.predict = MagicMock(return_value=d)
    b = _Basic(2, 3, MagicMock(return_value=gen), MagicMock(return_value=encoder),
               MagicMock(return_value=disc))
    return b, gen, encoder, disc


def test_basic_score_cells_is_the_composed_definition():
    cells = np.array([[0.0, 4000.0, 1.0], [2.0, 0.0, 0.0]])
    enc = np.array([[0.1, 0.9], [0.7, 0.3]], np.float32)
    pred = np.array([[0.5, 4000.25, 1.0], [2.0, -1.0, 3.0]], np.float32)
    d = np.array([[0.8], [0.3]], np.float32)
    b, gen, encoder, disc = _mocked(enc, pred, d)
    rnd = np.full((2, 2), 0.5, np.float32)
    s = b.score_cells(cells, rnd)
    assert isinstance(s, CellScores)
    assert all(a.dtype == np.float32 for a in s)
    np.testing.assert_array_equal(s.encodings, enc)
    np.testing.assert_array_equal(s.mse, np.array([(0.25 + 0.0625) / 3, 10.0 / 3], np.float32))
    np.testing.assert_array_equal(s.d_real, d.reshape(-1))
    assert encoder.predict.call_args[0][0] is cells
    g_in = gen.predict.call_args[0][0]
    assert g_in[0] is enc and g_in[1] is rnd
    d_in = disc.predict.call_args[0][0]
    assert d_in[0] is enc and d_in[1] is cells


def test_basic_score_cells_random_in_none_draws_through_random_uniform_vector():
    enc = np.zeros((2, 2), np.float32)
    b, gen, _, _ = _mocked(enc, np.zeros((2, 3), np.float32), np.zeros((2, 1), np.float32))
    drawn = np.full((2, 2), 0.25, np.float32)
    b.random_uniform_vector = MagicMock(return_value=drawn)
    b.score_cells(CellMatrix.from_dense(np.ones((2, 3))))
    b.random_uniform_vector.assert_called_once_with(2)
    assert gen.predict.call_args[0][0][1] is drawn


# ------------------------------------------------------------------ the score command
def _main(*args):
    from cellcomm_b200.__main__ import main
    main(["", "score", *args])


def _meta_checkpoint(path, gene_size, variant="cont"):
    np.savez(path, **{"meta/variant": variant, "meta/encoding_size": 3,
                      "meta/gene_size": gene_size})
    return str(path)


def _source(tmp_path, genes, name="source.mtx"):
    return CellMatrix.from_dense(np.ones((2, genes))).to_mtx(str(tmp_path / name))


@pytest.mark.parametrize("args", [(), ("a.npz",), ("a.npz", "b.mtx", "c.mtx"),
                                  ("a.npz", "b.mtx", "c.mtx", "d.csv", "extra")])
def test_score_command_wants_four_parameters(args):
    with pytest.raises(AssertionError, match="score <checkpoint.npz> <source-matrix-file> "
                                             "<matrix-file> <scores.csv>"):
        _main(*args)


def test_score_command_rejects_gene_count_mismatch(tmp_path, monkeypatch):
    import cellcomm_b200.bigan_cont as cont
    built = MagicMock(side_effect=AssertionError("a network was built"))
    monkeypatch.setattr(cont, "ContinuousCellBiGan", built)
    ckpt = _meta_checkpoint(tmp_path / "c.npz", 5)
    cells = _source(tmp_path, 5, "cells.mtx")
    with pytest.raises(ValueError, match="scores 5 genes.*has 4"):
        _main(ckpt, _source(tmp_path, 4), cells, str(tmp_path / "out.csv"))
    assert not built.called
    assert not os.path.exists(tmp_path / "out.csv")


def test_score_command_rejects_unknown_variant(tmp_path):
    ckpt = _meta_checkpoint(tmp_path / "c.npz", 4, variant="other")
    with pytest.raises(ValueError, match="unknown network variant"):
        _main(ckpt, _source(tmp_path, 4), _source(tmp_path, 4, "cells.mtx"),
              str(tmp_path / "out.csv"))


def _scores(n, Z, seed=0):
    rng = np.random.default_rng(seed)
    return CellScores(rng.normal(size=(n, Z)).astype(np.float32),
                      (rng.random(n) * 1e3).astype(np.float32),
                      rng.random(n).astype(np.float32))


def test_score_file_format_round_trips_float32(tmp_path):
    from cellcomm_b200.__main__ import write_score_file
    s = _scores(50, 3)
    s.mse[0], s.d_real[1], s.encodings[2, 0] = 1e-38, 0.1, np.float32(1 / 3)
    path = write_score_file(str(tmp_path / "s.csv"), np.arange(50) * 7 + 3, s)
    lines = open(path).read().splitlines()
    assert lines[0] == "barcode,mse,d-real,z0,z1,z2"
    assert len(lines) == 51
    got = np.array([[float(v) for v in line.split(",")] for line in lines[1:]])
    np.testing.assert_array_equal(got[:, 0], np.arange(50) * 7 + 3)
    assert lines[1].split(",")[0] == "3"
    assert got[:, 1].astype(np.float32).tobytes() == s.mse.tobytes()
    assert got[:, 2].astype(np.float32).tobytes() == s.d_real.tobytes()
    assert got[:, 3:].astype(np.float32).tobytes() == s.encodings.tobytes()
    assert lines[2].split(",")[2] == "%.9g" % float(np.float32(0.1))
    assert sorted(os.listdir(tmp_path)) == ["s.csv"]


def test_score_file_write_is_atomic(tmp_path):
    from cellcomm_b200.__main__ import write_score_file
    target = tmp_path / "s.csv"
    target.write_text("old\n")

    class Boom(Exception):
        pass

    class Failing:
        """barcodes that fail half way through the file"""
        def __iter__(self):
            yield 1
            raise Boom()

    with pytest.raises(Boom):
        write_score_file(str(target), Failing(), _scores(3, 2))
    assert target.read_text() == "old\n"
    assert sorted(os.listdir(tmp_path)) == ["s.csv"]


# ------------------------------------------------------------------ validation.csv
def _emulated_trainer(tmp_path, columns, seed=11):
    """a BasicBiGan over mocked components whose predictions are functions of their inputs,
    so score_cells runs its definition; trainer.data with the given gene ids"""
    G, Z = len(columns), 2

    def encode(cells):
        x = np.asarray(cells, dtype=np.float64)
        return np.stack([x.sum(1), x[:, 0]], 1).astype(np.float32) / 100

    def generate(inputs):
        z, r = inputs
        return (np.asarray(z).sum(1, keepdims=True) + np.asarray(r).sum(1, keepdims=True)
                + np.zeros((1, G), np.float32)).astype(np.float32)

    def discriminate(inputs):
        z, _ = inputs
        return (1 / (1 + np.exp(-np.asarray(z)[:, :1] + 0.05))).astype(np.float32)

    comps = [MagicMock() for _ in range(3)]
    comps[0].predict = MagicMock(side_effect=generate)
    comps[1].predict = MagicMock(side_effect=encode)
    comps[2].predict = MagicMock(side_effect=discriminate)
    net = _Basic(Z, G, *(MagicMock(return_value=c) for c in comps))
    net._prior_rng = np.random.default_rng(seed)
    data = CellMatrix.from_dense(np.ones((4, G)), columns=columns)
    return SimpleNamespace(data=data, network=net)


def test_save_validation_rows_and_untouched_rng(tmp_path):
    from cellcomm_b200.intercepts import SinkIntercepts
    cols = np.array([2, 5, 9, 11])
    trainer = _emulated_trainer(tmp_path, cols)
    rng = np.random.default_rng(1)
    held = CellMatrix.from_dense(rng.integers(0, 5, (30, 4)).astype(np.float64), columns=cols)
    sink = SinkIntercepts(str(tmp_path))
    np.random.seed(123)
    global_state = np.random.get_state()
    prior_state = trainer.network._prior_rng.bit_generator.state
    intercept = sink.save_validation(trainer, held, noise_seed=4)
    for it in (0, 1, 2):
        intercept(it, (1.0, 2.0, 3.0))
    sink.sink.drain_data()
    g2 = np.random.get_state()
    assert all(np.array_equal(a, b) for a, b in zip(global_state, g2))
    assert trainer.network._prior_rng.bit_generator.state == prior_state
    lines = open(tmp_path / "validation.csv").read().splitlines()
    assert lines[0] == "iteration,mse,d-real,real-pct"
    assert [line.split(",")[0] for line in lines[1:]] == ["0", "1", "2"]
    # every iteration: the same cells with the same noise (drawn once from default_rng(4))
    assert len(set(line.split(",", 1)[1] for line in lines[1:])) == 1
    noise = np.random.default_rng(4).random((30, 2), dtype=np.float32)
    s = trainer.network.score_cells(held, noise)
    want = [float(np.mean(s.mse, dtype=np.float64)), float(np.mean(s.d_real.astype(np.float64))),
            float(np.mean(np.round(s.d_real) == 1))]
    assert [float(v) for v in lines[1].split(",")[1:]] == want
    assert 0.0 < want[2] < 1.0


def test_save_validation_rejects_other_genes(tmp_path):
    from cellcomm_b200.intercepts import SinkIntercepts
    trainer = _emulated_trainer(tmp_path, np.array([2, 5, 9, 11]))
    held = CellMatrix.from_dense(np.ones((3, 4)), columns=np.array([2, 5, 9, 12]))
    sink = SinkIntercepts(str(tmp_path))
    with pytest.raises(ValueError, match="gene ids of the training matrix"):
        sink.save_validation(trainer, held)
    assert not os.path.exists(tmp_path / "validation.csv")
    # aligned with reindex_columns, the same cells are accepted
    sink.save_validation(trainer, held.reindex_columns(trainer.data.columns))
    assert os.path.exists(tmp_path / "validation.csv")
