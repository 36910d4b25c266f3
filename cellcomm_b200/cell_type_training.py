"""Drop-in for the reference's `src/cell_type_training.py` (same names, same call semantics):

    load_matrix(matrix_file, verbose=False)      reference :9-17
    load_cells(cells_file, verbose=False)        reference :20-26
    CellTraining(data, batch_size, encoding_size, batches_per_iteration=10)   :29-50

The reference returns a dense pandas DataFrame (30k x 33,694 float64 = 8.1 GB) and gathers
dense rows on the host.  Here `load_matrix` returns a `CellMatrix`: the same matrix as a
device-resident CSR (bit-exact with the pandas pivot, see tests/test_loader.py) that quacks
like the bits of DataFrame the callers use (`shape`, `len`, `sample`, `index`, `columns`,
`values`, `to_csv`).  `sample()` draws the same rows as `DataFrame.sample` (same numpy RNG
calls) and returns a `CellBatch` of row indices; the dense bf16 minibatch is produced on the
GPU by the gather kernel.
"""
from typing import Any, Callable

import numpy as np

from . import _lib


class CellBatch:
    """A sampled minibatch: row positions into a CellMatrix (dense rows are gathered on the
    device).  `len()`, `.shape`, `.values`/`to_numpy()` mirror the DataFrame the reference
    passes to `trainings_step`."""

    def __init__(self, matrix, positions):
        self.matrix = matrix
        self.positions = np.ascontiguousarray(positions, dtype=np.int64)

    def __len__(self):
        return len(self.positions)

    @property
    def shape(self):
        return (len(self.positions), self.matrix.shape[1])

    @property
    def index(self):
        return self.matrix.index[self.positions]

    @property
    def columns(self):
        return self.matrix.columns

    def to_numpy(self, dtype=np.float64):
        return self.matrix.dense_rows(self.positions, dtype)

    @property
    def values(self):
        return self.to_numpy()

    def __array__(self, dtype=None, copy=None):
        return self.to_numpy(dtype or np.float64)


class CellMatrix:
    """cells x genes count matrix: host CSR (exact float64 + float32 values) and, lazily, the
    device-resident CSR the gather kernel reads."""

    def __init__(self, rowptr, colidx, values64, row_ids, col_ids):
        self.rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
        self.colidx = np.ascontiguousarray(colidx, dtype=np.int32)
        self.values64 = np.ascontiguousarray(values64, dtype=np.float64)
        self.values32 = self.values64.astype(np.float32)
        self.index = np.ascontiguousarray(row_ids, dtype=np.int64)      # barcode ids (ascending)
        self.columns = np.ascontiguousarray(col_ids, dtype=np.int64)    # gene ids (ascending)
        self._dev = {}

    # ---------------------------------------------------------------- construction
    @classmethod
    def from_csr_handle(cls, lib, h):
        import ctypes as C
        rows, cols, nnz = lib.cc_csr_rows(h), lib.cc_csr_cols(h), lib.cc_csr_nnz(h)

        def arr(ptr, n, ctype, dtype):
            if n == 0:
                return np.zeros(0, dtype=dtype)
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(n,)).copy()

        m = cls(arr(lib.cc_csr_rowptr(h), rows + 1, C.c_int64, np.int64),
                arr(lib.cc_csr_colidx(h), nnz, C.c_int32, np.int32),
                arr(lib.cc_csr_values64(h), nnz, C.c_double, np.float64),
                arr(lib.cc_csr_row_ids(h), rows, C.c_int64, np.int64),
                arr(lib.cc_csr_col_ids(h), cols, C.c_int64, np.int64))
        return m

    @classmethod
    def from_mtx(cls, path):
        import ctypes as C
        lib = _lib.load()
        h = C.c_void_p()
        _lib.check(lib.cc_mtx_load_csr(str(path).encode(), C.byref(h)))
        try:
            return cls.from_csr_handle(lib, h)
        finally:
            lib.cc_csr_destroy(h)

    @classmethod
    def from_coo(cls, gene, barcode, val):
        import ctypes as C
        lib = _lib.load()
        g = np.ascontiguousarray(gene, dtype=np.int64)
        b = np.ascontiguousarray(barcode, dtype=np.int64)
        v = np.ascontiguousarray(val, dtype=np.float64)
        h = C.c_void_p()
        _lib.check(lib.cc_coo_to_csr(g.ctypes.data, b.ctypes.data, v.ctypes.data, len(v),
                                     C.byref(h)))
        try:
            return cls.from_csr_handle(lib, h)
        finally:
            lib.cc_csr_destroy(h)

    @classmethod
    def from_dense(cls, dense, index=None, columns=None):
        """Wrap a dense host matrix (e.g. what load_cells reads) as a CellMatrix."""
        dense = np.asarray(dense, dtype=np.float64)
        rows, cols = dense.shape
        nz = dense != 0
        rowptr = np.zeros(rows + 1, dtype=np.int64)
        np.cumsum(nz.sum(1), out=rowptr[1:])
        colidx = np.nonzero(nz)[1].astype(np.int32)
        return cls(rowptr, colidx, dense[nz],
                   np.arange(1, rows + 1) if index is None else index,
                   np.arange(1, cols + 1) if columns is None else columns)

    # ---------------------------------------------------------------- DataFrame-ish surface
    @property
    def shape(self):
        return (len(self.index), len(self.columns))

    def __len__(self):
        return len(self.index)

    @property
    def nnz(self):
        return len(self.colidx)

    def sample(self, n=None, random_state=None):
        """DataFrame.sample(n, random_state): without replacement; int seed -> RandomState(seed),
        None -> the GLOBAL numpy state; positions = rs.permutation(N)[:n] (SURVEY.md A.2;
        golden rows [2,0,1] for seed 0, test/cell_type_training_test.py:36-41)."""
        n = 1 if n is None else int(n)
        N = len(self)
        if n > N:
            raise ValueError("Cannot take a larger sample than population when 'replace=False'")
        if random_state is None:
            rs = np.random
        elif isinstance(random_state, np.random.RandomState):
            rs = random_state
        else:
            rs = np.random.RandomState(random_state)
        return CellBatch(self, rs.permutation(N)[:n])

    def dense_rows(self, positions, dtype=np.float64):
        positions = np.asarray(positions, dtype=np.int64)
        out = np.zeros((len(positions), self.shape[1]), dtype=dtype)
        for i, r in enumerate(positions):
            b, e = self.rowptr[r], self.rowptr[r + 1]
            out[i, self.colidx[b:e]] = self.values64[b:e]
        return out

    def to_numpy(self, dtype=np.float64):
        return self.dense_rows(np.arange(len(self)), dtype)

    @property
    def values(self):
        return self.to_numpy()

    def __array__(self, dtype=None, copy=None):
        return self.to_numpy(dtype or np.float64)

    def to_csv(self, path):
        """`python3 src convert` (src/__main__.py:76-81): dense CSV, first column = barcode id,
        header = gene ids (what DataFrame.to_csv writes for the pivoted frame)."""
        all_int = bool(np.all(self.values64 == np.round(self.values64)))
        with open(path, "w") as f:
            f.write("barcode," + ",".join(str(int(c)) for c in self.columns) + "\n")
            for i in range(len(self)):
                row = self.dense_rows([i])[0]
                cells = (f"{v:.1f}" for v in row) if all_int else (repr(float(v)) for v in row)
                f.write(str(int(self.index[i])) + "," + ",".join(cells) + "\n")

    # ---------------------------------------------------------------- device residency
    def device_csr(self, device="cuda"):
        """(rowptr int64, colidx int32, values float32) resident on `device` (uploaded once)."""
        import torch
        key = str(torch.device(device))
        d = self._dev.get(key)
        if d is None:
            d = (torch.from_numpy(self.rowptr).to(device), torch.from_numpy(self.colidx).to(device),
                 torch.from_numpy(self.values32).to(device))
            self._dev[key] = d
        return d


def load_matrix(matrix_file, verbose=False):
    if verbose:
        print(f'============ Loading {matrix_file}...')
    df = CellMatrix.from_mtx(matrix_file)
    if verbose:
        print(f'============ DONE! barcodes: {df.shape[0]}, genes: {df.shape[1]}')
    return df


def load_cells(cells_file, verbose=False):
    """pd.read_csv(cells_file, index_col=0): the dense CSV written by `python3 src convert`."""
    if verbose:
        print(f'============ Loading {cells_file}...')
    with open(cells_file) as f:
        header = f.readline().rstrip("\n").split(",")[1:]
        idx, rows = [], []
        for line in f:
            parts = line.rstrip("\n").split(",")
            if len(parts) < 2:
                continue
            idx.append(int(float(parts[0])))
            rows.append([float(p) for p in parts[1:]])
    df = CellMatrix.from_dense(np.array(rows, dtype=np.float64).reshape(len(rows), len(header)),
                               np.array(idx, dtype=np.int64),
                               np.array([int(float(c)) for c in header], dtype=np.int64))
    if verbose:
        print(f'============ DONE! barcodes: {df.shape[0]}, genes: {df.shape[1]}')
    return df


class CellTraining:
    def __init__(self, data, batch_size, encoding_size, batches_per_iteration=10, *, seed=None):
        """seed (not in the reference): seeds the network's weights, device RNG and priors."""
        try:
            from .bigan_cont import ContinuousCellBiGan
        except ImportError:  # imported as a top-level module (PYTHONPATH=src style)
            from bigan_cont import ContinuousCellBiGan
        self.batch_size = batch_size
        self.data = data
        self.batches_per_iteration = batches_per_iteration
        kwargs = {} if seed is None else {"seed": seed}
        self.network = ContinuousCellBiGan(encoding_size, gene_size=self.data.shape[1], **kwargs)

    def sample_cell_data(self, random_seed=None):
        return self.data.sample(self.batch_size, random_state=random_seed)

    def run(self, iterations, interceptor: Callable[[int, Any], None] = None, start_iteration=0):
        """The reference's loop (src/cell_type_training.py:40-50).  `start_iteration` (not in the
        reference) numbers the iterations of a resumed run.

        Data parallel (torchrun, one process per GPU): every rank runs this loop; each step is
        ONE global batch of `batch_size` cells split contiguously over the ranks.  The
        interceptor runs on rank 0 only, while the other ranks serve the collective parts of
        what it calls (the row-sharded encode-all-cells pass, checkpoint gathers)."""
        net = self.network
        world = net._world() if hasattr(net, "_world") and callable(getattr(net, "_world")) else 1
        if not isinstance(world, int):
            world = 1                       # mocked networks
        has_interceptor = interceptor is not None
        if world > 1:
            net.sync_host_rng()
            # rank 0 decides whether the workers have interceptor work to serve
            has_interceptor = net.broadcast_from_coordinator(has_interceptor)
        for it in range(start_iteration, start_iteration + iterations):
            g_losses = e_losses = d_losses = 0
            for batch_it in range(self.batches_per_iteration):
                batch = self.sample_cell_data()
                gl, el, dl = net.trainings_step(batch)
                g_losses += gl
                e_losses += el
                d_losses += dl
            if has_interceptor:
                if world == 1:
                    interceptor(it, (g_losses, e_losses, d_losses))
                elif net.is_coordinator():
                    net.begin_interceptors()
                    try:
                        interceptor(it, (g_losses, e_losses, d_losses))
                    except BaseException:
                        net.release_workers(failed=True)
                        raise
                    net.release_workers()
                else:
                    net.serve(self.data)
