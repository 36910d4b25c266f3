"""Generated cells without a GPU: the .mtx writer (cc_mtx_write -> cc_mtx_load_csr round trip,
header, atomic CellMatrix.to_mtx), the definition of BasicBiGan.generate_cell_matrix, and the
argument checks of `python -m cellcomm_b200 generate`."""
import ctypes
import os
from unittest.mock import MagicMock

import numpy as np
import pytest

from cellcomm_b200 import _lib
from cellcomm_b200.cell_type_training import CellMatrix, load_matrix


def _assert_same(a, b):
    for name in ("rowptr", "colidx", "index", "columns"):
        np.testing.assert_array_equal(getattr(a, name), getattr(b, name), err_msg=name)
    assert a.values64.tobytes() == b.values64.tobytes()      # bit-exact float64


def _roundtrip(m, tmp_path, name="m.mtx"):
    return load_matrix(m.to_mtx(str(tmp_path / name)))


def _header(path):
    with open(path) as f:
        return [f.readline() for _ in range(4)]


def test_integer_matrix_roundtrip_and_header(tmp_path):
    dense = np.array([[0, 2, 0, 7], [1, 0, 3, 0], [0, 0, 0, 120000]], dtype=np.float64)
    m = CellMatrix.from_dense(dense)
    p = m.to_mtx(str(tmp_path / "int.mtx"))
    lines = open(p).read().splitlines()
    assert lines[0] == "%%MatrixMarket matrix coordinate integer general"
    assert lines[1] == "%"
    assert lines[2] == "4 3 5"                     # genes barcodes nnz
    assert lines[3:] == ["2 1 2", "4 1 7", "1 2 1", "3 2 3", "4 3 120000"]   # barcode-major
    _assert_same(load_matrix(p), m)


def test_real_values_explicit_zeros_and_sparse_ids(tmp_path):
    # non-contiguous ids, an explicit zero (keeps its row and column alive), awkward doubles
    genes = [5, 7, 5, 900, 7, 12]
    barcodes = [10, 10, 12, 30, 30, 31]
    vals = [1.0, 2.5, 0.0, -3.0, 1e-300, 0.1 + 0.2]
    m = CellMatrix.from_coo(genes, barcodes, vals)
    p = m.to_mtx(str(tmp_path / "real.mtx"))
    assert _header(p)[0] == "%%MatrixMarket matrix coordinate real general\n"
    assert _header(p)[2] == "4 4 6\n"
    r = load_matrix(p)
    _assert_same(r, m)
    np.testing.assert_array_equal(r.index, [10, 12, 30, 31])
    np.testing.assert_array_equal(r.columns, [5, 7, 12, 900])


def test_one_by_one(tmp_path):
    m = CellMatrix.from_dense(np.array([[3.0]]), index=np.array([42]), columns=np.array([7]))
    p = m.to_mtx(str(tmp_path / "one.mtx"))
    assert open(p).read() == "%%MatrixMarket matrix coordinate integer general\n%\n1 1 1\n7 42 3\n"
    _assert_same(load_matrix(p), m)


def test_random_roundtrip_many_threads(tmp_path):
    """large enough that the writer formats on several threads and in several blocks"""
    rng = np.random.default_rng(3)
    rows, cols = 3000, 700
    dense = np.where(rng.random((rows, cols)) < 0.6, rng.integers(1, 50, (rows, cols)), 0)
    dense = dense.astype(np.float64)
    dense[0, :] = 1.0                    # every column holds an entry
    dense[:, 0] = 1.0                    # every row holds an entry
    dense[5, 3] = 2.0 / 3.0              # one real value switches the banner
    m = CellMatrix.from_dense(dense, index=np.arange(rows) * 3 + 1, columns=np.arange(cols) * 2 + 5)
    assert m.nnz > (1 << 20)
    p = m.to_mtx(str(tmp_path / "big.mtx"))
    assert _header(p)[0].split()[3] == "real"
    _assert_same(load_matrix(p), m)


def test_empty_rows_and_columns_vanish_on_reload(tmp_path):
    dense = np.array([[0, 0, 0], [0, 4, 0], [0, 0, 0]], dtype=np.float64)
    r = _roundtrip(CellMatrix.from_dense(dense), tmp_path)
    np.testing.assert_array_equal(r.index, [2])
    np.testing.assert_array_equal(r.columns, [2])
    assert r.values64.tolist() == [4.0]


def test_writer_rejects_inconsistent_csr(tmp_path):
    lib = _lib.load()
    rowptr = np.array([0, 2], dtype=np.int64)
    colidx = np.array([0, 5], dtype=np.int32)          # column 5 of 2
    vals = np.array([1.0, 2.0])
    ids = np.array([1, 2], dtype=np.int64)
    path = str(tmp_path / "bad.mtx").encode()
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    rc = lib.cc_mtx_write(path, 1, 2, 2, ptr(rowptr), ptr(colidx), ptr(vals), ptr(ids), ptr(ids))
    assert rc != 0 and b"column index" in lib.cc_last_error()
    rc = lib.cc_mtx_write(path, 1, 2, 3, ptr(rowptr), ptr(colidx), ptr(vals), ptr(ids), ptr(ids))
    assert rc != 0 and b"rowptr" in lib.cc_last_error()
    assert not os.path.exists(path)


def test_to_mtx_is_atomic(tmp_path, monkeypatch):
    """a write that fails half way leaves neither a partial target nor a temporary file, and an
    existing target keeps its old content"""
    target = tmp_path / "out.mtx"
    target.write_text("old\n")
    real = _lib.load()

    class Failing:
        def __getattr__(self, name):
            return getattr(real, name)

        @staticmethod
        def cc_mtx_write(path, *args):
            with open(path, "w") as f:
                f.write("%%MatrixMarket matrix coordinate integer general\n%\n1 1 1\n1 1")
            return -1

        @staticmethod
        def cc_last_error():
            return b"disk full"

    monkeypatch.setattr(_lib, "load", lambda: Failing())
    m = CellMatrix.from_dense(np.array([[1.0]]))
    with pytest.raises(_lib.CCError, match="disk full"):
        m.to_mtx(str(target))
    assert target.read_text() == "old\n"
    assert sorted(os.listdir(tmp_path)) == ["out.mtx"]
    with pytest.raises(_lib.CCError):
        m.to_mtx(str(tmp_path / "new.mtx"))
    assert sorted(os.listdir(tmp_path)) == ["out.mtx"]


def test_basic_generate_cell_matrix_is_from_dense_of_generate_cells():
    from cellcomm_b200.bigan_basic import BasicBiGan

    class B(BasicBiGan):
        def random_encoding_vector(self, n):
            return np.zeros((n, 2), np.float32)

        def trainings_step(self, batch):
            pass

    gen = MagicMock()
    dense = np.array([[0.4, 2.6, 0.0], [1.5, 0.0, 2.5]], dtype=np.float32)
    gen.predict = MagicMock(return_value=dense)
    b = B(2, 3, MagicMock(return_value=gen), MagicMock(), MagicMock())
    enc = np.ones((2, 2), np.float32)
    rnd = np.full((2, 2), 0.5, np.float32)
    m = b.generate_cell_matrix(enc, rnd, columns=np.array([4, 8, 9]))
    want = CellMatrix.from_dense(b.generate_cells(enc, rnd), columns=np.array([4, 8, 9]))
    _assert_same(m, want)
    np.testing.assert_array_equal(m.to_numpy(np.float32), [[0, 3, 0], [2, 0, 2]])
    np.testing.assert_array_equal(m.index, [1, 2])
    inputs = gen.predict.call_args[0][0]
    assert inputs[0] is enc and inputs[1] is rnd
    # random_in=None draws the noise like generate_cells does
    m2 = b.generate_cell_matrix(enc)
    assert gen.predict.call_args[0][0][1].shape == (2, 2)
    np.testing.assert_array_equal(m2.columns, [1, 2, 3])


# ------------------------------------------------------------------ the generate command
def _main(*args):
    from cellcomm_b200.__main__ import main
    main(["", "generate", *args])


def _meta_checkpoint(path, gene_size, variant="cont"):
    np.savez(path, **{"meta/variant": variant, "meta/encoding_size": 3,
                      "meta/gene_size": gene_size})
    return str(path)


def _source(tmp_path, genes):
    return CellMatrix.from_dense(np.ones((2, genes))).to_mtx(str(tmp_path / "source.mtx"))


@pytest.mark.parametrize("args", [(), ("a.npz",), ("a.npz", "b.mtx", "10"),
                                  ("a.npz", "b.mtx", "10", "c.mtx", "extra")])
def test_generate_command_wants_four_parameters(args):
    with pytest.raises(AssertionError, match="generate <checkpoint.npz> <source-matrix-file> "
                                             "<n-cells> <target-matrix-file>"):
        _main(*args)


@pytest.mark.parametrize("n", ["0", "-3"])
def test_generate_command_rejects_fewer_than_one_cell(tmp_path, n):
    ckpt = _meta_checkpoint(tmp_path / "c.npz", 4)
    with pytest.raises(ValueError, match="n-cells must be at least 1"):
        _main(ckpt, _source(tmp_path, 4), n, str(tmp_path / "out.mtx"))
    assert not os.path.exists(tmp_path / "out.mtx")


def test_generate_command_rejects_gene_count_mismatch(tmp_path):
    ckpt = _meta_checkpoint(tmp_path / "c.npz", 5)
    with pytest.raises(ValueError, match="generates 5 genes.*has 4"):
        _main(ckpt, _source(tmp_path, 4), "10", str(tmp_path / "out.mtx"))
    assert not os.path.exists(tmp_path / "out.mtx")
