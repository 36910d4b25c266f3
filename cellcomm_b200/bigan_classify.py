"""Drop-in for the reference's `src/bigan_classify.py`: the categorical-code BiGAN, the
network factories (`_build_generator/_build_encoder/_build_discriminator`, reference :10-75),
the five compiled training graphs with their freeze pattern (:83-115) and `trainings_step`
(:126-155).

The factories return `NetModel` handles over layer graphs (cellcomm_b200.engine); the
arithmetic of `train_on_batch` / `predict` runs in libcellcomm_b200.so through
`BiGanEngine` (tcgen05 GEMMs + tail kernels).  If a factory returns something else (the
reference's tests inject mocks), no engine is built and only the wiring is available.
"""
import json
import os
from typing import Callable

import numpy as np

try:
    from .bigan_basic import BasicBiGan
    from . import engine as _engine
    from .models import NetModel, RMSprop, losses, activations  # noqa: F401
    from .cell_type_training import CellBatch, CellMatrix
except ImportError:  # imported as top-level modules (PYTHONPATH=src style)
    from bigan_basic import BasicBiGan
    from cellcomm_b200 import engine as _engine
    from cellcomm_b200.models import NetModel, RMSprop, losses, activations  # noqa: F401
    from cellcomm_b200.cell_type_training import CellBatch, CellMatrix


def _build_generator(encoding_size, gene_size):
    return NetModel(_engine.classify_generator_graph(encoding_size, gene_size), "G",
                    [("gen_encoding_in", "z"), ("gen_random_in", "r")])


def _build_encoder(encoding_size, gene_size):
    return NetModel(_engine.classify_encoder_graph(encoding_size, gene_size), "E",
                    [("enc_cell_in", "cell")])


def _build_discriminator(encoding_size, gene_size):
    return NetModel(_engine.discriminator_graph(encoding_size, gene_size), "D",
                    [("encoding_input", "z"), ("cell_input", "cell")])


def print_dot():
    print('.', end='', flush=True)


class TrainGraph:
    """One of the reference's five compiled training models: which component it updates, which
    it runs frozen, its loss and the (shared) optimizer.  `train_on_batch` runs the matching
    sub-step of the engine."""

    def __init__(self, owner, name, substep, trained, layers, input_shape, loss, optimizer):
        self._owner, self.name, self._substep, self._trained = owner, name, substep, trained
        self.layers, self.input_shape, self.output_shape = layers, input_shape, layers[-1].output_shape
        self.loss, self.optimizer, self._is_compiled = loss, optimizer, True

    def train_on_batch(self, x, y=None):
        return self._owner._train_on_batch(self._substep, x, y)


class ClassifyCellBiGan(BasicBiGan):
    VARIANT = "classify"

    def __init__(self, encoding_size, gene_size,
                 generator_factory: Callable[[int, int], object] = _build_generator,
                 encoder_factory: Callable[[int, int], object] = _build_encoder,
                 discriminator_factory: Callable[[int, int], object] = _build_discriminator,
                 device=None, seed=None, dist=None, deterministic=None):
        """seed: the weights, the device RNG key and the host prior stream (None: random).
        deterministic: fixed-order reductions, so that the same seed and data give the same
        bits on every run (BiGanEngine); None reads CELLCOMM_B200_DETERMINISTIC (default 0)."""
        super().__init__(encoding_size, gene_size, generator_factory, encoder_factory, discriminator_factory)
        if seed is not None:
            self._prior_rng = np.random.default_rng([int(seed), 1])
        if deterministic is None:
            deterministic = os.environ.get("CELLCOMM_B200_DETERMINISTIC", "0") == "1"
        self.deterministic = bool(deterministic)
        self.gene_size = gene_size
        discr_optimizer = RMSprop(learning_rate=0.0075, rho=0.85, momentum=0.1)
        self._optimizer = discr_optimizer
        G, E, D = self._generator, self._encoder, self._discriminator
        self._engine = None
        self._staged = None
        if all(isinstance(m, NetModel) for m in (G, E, D)):
            if device is None:
                device = os.environ.get("CELLCOMM_B200_DEVICE", "cuda")
            if dist is None:
                dist = _engine.default_dist()
            self._engine = _engine.BiGanEngine(
                self.VARIANT, encoding_size, gene_size, max_batch=1, device=device, seed=seed,
                dist=dist, graphs={"G": G.graph, "E": E.graph, "D": D.graph},
                deterministic=self.deterministic)
            for m in (G, E, D):
                m._bind(self, self._engine)
            z = (None, encoding_size)
            bce, mse = losses.binary_crossentropy, losses.mse
            # freeze pattern of the five graphs, reference :90-115
            self._train_gen_w_discr = TrainGraph(self, 'train-generator-with-discriminator', 1, "G",
                                                 [G, D], [z, z], bce, discr_optimizer)
            self._train_gen_w_enc = TrainGraph(self, 'train-generator-with-encoder', 2, "G",
                                               [E, G], [(None, gene_size), z], mse, discr_optimizer)
            self._train_enc_w_discr = TrainGraph(self, 'train-encoder-with-discriminator', 3, "E",
                                                 [E, D], (None, gene_size), bce, discr_optimizer)
            self._train_enc_w_gen = TrainGraph(self, 'train-encoder-with-generator', 4, "E",
                                               [G, E], [z, z], mse, discr_optimizer)
            D.compile(optimizer=discr_optimizer, loss=bce)
            G.trainable, E.trainable, D.trainable = False, False, True
            self._snapshot_params()             # reference src/bigan_basic.py:21-22
        self._workers_serving = False

    # ------------------------------------------------------------------ priors
    def random_encoding_vector(self, batch_size):
        """to_categorical(np.random.randint(0, Z, B), Z) on numpy's GLOBAL state (reference
        :117-119; golden np.random.seed(21) -> [1,3,0,0,0], test/bigans_cc_test.py:57-63)."""
        rand_ixs = np.random.randint(0, self.encoding_size, batch_size)
        out = np.zeros((batch_size, self.encoding_size), dtype=np.float32)
        out[np.arange(batch_size), rand_ixs] = 1.0
        return out

    def trainings_encoding_prediction(self, cell_data):
        prediction = np.asarray(self.encoding_prediction(cell_data))
        argmax = np.argmax(prediction, -1)
        out = np.zeros((len(argmax), self.encoding_size), dtype=np.float32)
        out[np.arange(len(argmax)), argmax] = 1.0
        return out

    # ------------------------------------------------------------------ the step
    def trainings_step(self, batch):
        """Six updates + two predicts, reference :126-142, as one pass of BiGanEngine.train_step
        (the sub-step order, freeze pattern and loss bookkeeping live in engine.py).

        Data parallel (one process per GPU): every rank calls this with the SAME global batch
        (`CellTraining.sample_cell_data` draws one `permutation(N)[:B]` on every rank) and
        draws the same global priors; rank r then works on the contiguous rows
        [r*B/W, (r+1)*B/W).  BN statistics, gradients and losses are summed over ranks inside
        the engine, so the step is the reference's step on the global batch."""
        eng = self._require_engine()
        batch_size = len(batch)
        encodings = self.random_encoding_vector(batch_size)
        noise = self.random_uniform_vector(batch_size)
        lo, hi = self._local_rows(batch_size)
        if hi - lo != batch_size:
            encodings, noise = encodings[lo:hi], noise[lo:hi]
            batch = _rows(batch, lo, hi)
        n = hi - lo
        if (isinstance(batch, CellBatch) and eng.device.type == "cuda" and
                eng.peer_graphable() and os.environ.get("CELLCOMM_B200_GRAPH", "1") != "0"):
            # the whole step (gather + every kernel, in data-parallel runs also the gradient
            # exchange over peer memory) is one CUDA-graph launch
            gs = eng.capture_step(batch.matrix.device_csr(eng.device), batch.matrix.shape[1],
                                  n, latents="host")
            eng.z32[:n].copy_(_as_f32(encodings), non_blocking=True)
            eng.r32[:n].copy_(_as_f32(noise), non_blocking=True)
            return gs.replay(batch.positions)
        x16 = self._stage_cells(batch)
        eng.set_latents(encodings, noise, n)
        g_loss, e_loss, d_loss = eng.train_step(x16)
        return g_loss, e_loss, d_loss

    # ------------------------------------------------------------------ data parallel
    def _world(self):
        return self._engine.dist.world_size if self._engine is not None else 1

    def _rank(self):
        return self._engine.dist.rank if self._engine is not None else 0

    def _local_rows(self, n):
        """This rank's contiguous share [lo, hi) of n global rows."""
        W = self._world()
        if W == 1:
            return 0, n
        if n % W:
            raise ValueError(f"data parallel over {W} GPUs needs a batch divisible by {W}, got {n}")
        r = self._rank()
        return r * (n // W), (r + 1) * (n // W)

    def is_coordinator(self):
        """True on the process that runs the interceptors (rank 0; always when single-process)."""
        return self._rank() == 0

    def sync_host_rng(self):
        """Give every rank rank 0's host RNG states (numpy's global state, which the batch
        sampler and the classify prior draw from, and the private prior generator), so all
        ranks draw the same global batch and priors.  Collective; `CellTraining.run` calls it."""
        if self._world() == 1:
            return
        state = self._engine.dist.broadcast_object(
            (np.random.get_state(), self._prior_rng.bit_generator.state)
            if self.is_coordinator() else None)
        np.random.set_state(state[0])
        self._prior_rng.bit_generator.state = state[1]

    def broadcast_from_coordinator(self, obj):
        """rank 0's (picklable) value on every rank.  Collective."""
        return self._engine.dist.broadcast_object(obj if self.is_coordinator() else None)

    def begin_interceptors(self):
        """Rank 0, before it runs the interceptors of an iteration: from now on the other ranks
        sit in `serve()` and execute the collective parts of whatever rank 0 calls."""
        self._workers_serving = self._world() > 1

    def release_workers(self, failed=False):
        if getattr(self, "_workers_serving", False):
            self._workers_serving = False
            self._engine.dist.broadcast_object(("abort",) if failed else ("release",))

    def serve(self, data):
        """Ranks != 0 during the interceptors: run this rank's share of every collective
        operation rank 0 announces -- the row-sharded encode-all-cells pass over `data`
        (encode: no communication but the final gather of the (N_i, Z) pieces), and the
        gathers a checkpoint needs -- until rank 0 releases the workers."""
        dist = self._engine.dist
        while True:
            cmd = dist.broadcast_object(None)
            if cmd[0] == "release":
                return
            if cmd[0] == "abort":
                raise RuntimeError("rank 0 failed inside an interceptor")
            if cmd[0] == "encode_all":
                self._encode_all_sharded(data)
            elif cmd[0] == "state":
                self._engine.state_dict()
            else:
                raise RuntimeError(f"unknown data-parallel command {cmd!r}")

    def _announce(self, *cmd):
        if getattr(self, "_workers_serving", False):
            self._engine.dist.broadcast_object(cmd)

    def _encode_all_sharded(self, mat):
        """encoding_prediction over ALL cells of a CellMatrix with the rows sharded contiguously
        over the ranks (SURVEY.md 8e: no communication in the pass itself); the (N_i, Z) float32
        pieces are all-gathered, every rank returns the full host array."""
        import torch
        eng, W, r = self._engine, self._world(), self._rank()
        N, Z = len(mat), self.encoding_size
        per = (N + W - 1) // W
        lo, hi = min(N, r * per), min(N, (r + 1) * per)
        piece = torch.zeros((per, Z), dtype=torch.float32, device=eng.device)
        if hi > lo:
            self._encode_rows(mat, lo, hi, piece[:hi - lo])
        full = torch.empty((W * per, Z), dtype=torch.float32, device=eng.device)
        eng.dist.all_gather(full.view(-1), piece.view(-1))
        return full[:N].cpu().numpy()

    def _encode_rows(self, mat, lo, hi, out):
        """E.predict on rows [lo, hi) of a device-resident CellMatrix -> out (fp32, device)."""
        eng = self._engine
        if eng.device.type == "cuda" and os.environ.get("CELLCOMM_B200_ENCODE_STREAM", "1") != "0":
            rowptr, colidx, values = mat.device_csr(eng.device)
            eng.encode_stream(rowptr, colidx, values, lo, hi, out)
            return
        for s in range(lo, hi, self.PREDICT_TILE):
            m = min(self.PREDICT_TILE, hi - s)
            eng.encode(self._stage_cells(mat, s, m), out32=out[s - lo:s - lo + m])

    # ------------------------------------------------------------------ checkpoint / resume
    def save_checkpoint(self, path, extra=None):
        """Weights, RMSprop slots, BN moving statistics, the device RNG position and the host
        RNG states -> one .npz (the reference has no checkpointing; SURVEY.md 8f row f4).
        `extra`: additional scalars (e.g. the iteration number) stored as `meta/<key>`.
        Data parallel: rank 0 writes; the other ranks take part through serve() or by calling
        this too."""
        eng = self._require_engine()
        self._announce("state")
        state = eng.state_dict()
        state["meta/numpy_rng"] = _pack_numpy_state(np.random.get_state())
        state["meta/prior_rng"] = np.array(json.dumps(self._prior_rng.bit_generator.state))
        for k, v in (extra or {}).items():
            state[f"meta/{k}"] = v
        eng.write_checkpoint(path, state)

    def load_checkpoint(self, path):
        """-> dict of the checkpoint's `meta/*` entries (e.g. {'iteration': 7})."""
        state = self._require_engine().load_checkpoint(path)
        if "meta/numpy_rng" in state:
            np.random.set_state(_unpack_numpy_state(state["meta/numpy_rng"]))
        if "meta/prior_rng" in state:
            self._prior_rng.bit_generator.state = json.loads(str(state["meta/prior_rng"]))
        return {k[5:]: (v.item() if getattr(v, "ndim", 1) == 0 else v)
                for k, v in state.items() if k.startswith("meta/")}

    # ------------------------------------------------------------------ plumbing
    def _require_engine(self):
        if self._engine is None:
            raise RuntimeError("this BiGAN was built from non-NetModel components (mocks): the "
                               "CUDA engine is unavailable and there is no host fallback")
        return self._engine

    def _stage_cells(self, cells, row_start=0, rows=None):
        """[n, gene_size] bf16 device tile for `cells`: a CellBatch / CellMatrix is gathered
        from the device-resident CSR (cc_gather_rows); anything array-like (DataFrame, ndarray,
        list, torch tensor) is uploaded as float32 and cast on the device."""
        import torch
        ops = _engine.ops
        eng = self._engine
        dev = eng.device
        if isinstance(cells, (CellBatch, CellMatrix)):
            mat = cells.matrix if isinstance(cells, CellBatch) else cells
            rowptr, colidx, values = mat.device_csr(dev)
            if isinstance(cells, CellBatch):
                n = len(cells)
                idx = torch.from_numpy(cells.positions).to(dev, non_blocking=True)
                out = self._tile(n)
                ops.gather_rows(rowptr, colidx, values, mat.shape[1], row_idx=idx, out16=out)
            else:
                n = len(mat) - row_start if rows is None else rows
                out = self._tile(n)
                ops.gather_rows(rowptr, colidx, values, mat.shape[1], row_start=row_start,
                                n_rows=n, out16=out)
            return out
        if isinstance(cells, torch.Tensor):
            t = cells
        else:
            arr = cells.values if hasattr(cells, "values") and not isinstance(cells, np.ndarray) \
                else cells
            t = torch.as_tensor(np.ascontiguousarray(np.asarray(arr, dtype=np.float32)))
        if rows is not None:
            t = t[row_start:row_start + rows]
        t = t.to(dev, dtype=torch.float32, non_blocking=True)
        if t.dim() != 2 or t.shape[1] != self.gene_size:
            raise ValueError(f"expected cells of shape (n, {self.gene_size}), got {tuple(t.shape)}")
        out = self._tile(t.shape[0])
        ops.cast_f32_to_bf16(t, out)
        return out

    def _tile(self, n, name="_tile_buf"):
        buf = getattr(self, name, None)
        if buf is None or buf.shape[0] < n:
            buf = _engine.ops.alloc2d(max(n, 1), self.gene_size, device=self._engine.device)
            setattr(self, name, buf)
        return buf[:n]

    PREDICT_TILE = 4096

    def _predict(self, role, x):
        """Model.predict for G / E / D in inference mode -> float32 host array."""
        import torch
        eng = self._require_engine()
        dev = eng.device
        if role == "E":
            if isinstance(x, CellMatrix):
                # the encode-all-cells pass (src/intercepts/db_recorder.py:85)
                if self._world() > 1:
                    self._announce("encode_all")
                    return self._encode_all_sharded(x)
                out = torch.empty((len(x), self.encoding_size), dtype=torch.float32, device=dev)
                self._encode_rows(x, 0, len(x), out)
                return out.cpu().numpy()
            n = len(x)
            out = torch.empty((n, self.encoding_size), dtype=torch.float32, device=dev)
            for s in range(0, n, self.PREDICT_TILE):
                m = min(self.PREDICT_TILE, n - s)
                eng.encode(self._stage_cells(_rows(x, s, s + m)), out32=out[s:s + m])
            return out.cpu().numpy()
        enc, second = x
        z = torch.as_tensor(np.asarray(enc, dtype=np.float32)).to(dev)
        n = z.shape[0]
        if role == "G":
            r = torch.as_tensor(np.asarray(second, dtype=np.float32)).to(dev)
            out = torch.empty((n, self.gene_size), dtype=torch.float32, device=dev)
            for s in range(0, n, self.PREDICT_TILE):
                m = min(self.PREDICT_TILE, n - s)
                eng.set_latents(z[s:s + m], r[s:s + m], m)
                eng.generate(m, out32=out[s:s + m])
            return out.cpu().numpy()
        out = torch.empty((n, 1), dtype=torch.float32, device=dev)
        for s in range(0, n, self.PREDICT_TILE):
            m = min(self.PREDICT_TILE, n - s)
            tile = self._stage_cells(second, s, m) if isinstance(second, CellMatrix) \
                else self._stage_cells(_rows(second, s, s + m))
            eng.discriminate(z[s:s + m].contiguous(), tile, out[s:s + m])
        return out.cpu().numpy()

    def evaluate_discriminator_accuracy(self, sampled_batch):
        """(true-positives, true-negatives), reference src/bigan_basic.py:50-64 -- same draws in
        the same order (random encodings, then the generator noise), but G.predict -> round ->
        D.predict and E.predict -> D.predict stay on the device: the (B, genes) generated cells
        never visit the host.  Only the two counts are read back."""
        if self._engine is None:
            return super().evaluate_discriminator_accuracy(sampled_batch)
        import torch
        eng, ops = self._engine, _engine.ops
        n = len(sampled_batch)
        random_encodings = self.random_encoding_vector(n)
        noise = self.random_uniform_vector(n)           # generate_cells(encodings) draws it
        eng.set_latents(random_encodings, noise, n)
        fake = self._tile(n, "_fake_buf")
        ops.round_half_even(eng.generate(n), out16=fake)
        p = torch.empty((n, 1), dtype=torch.float32, device=eng.device)
        eng.discriminate(eng.z32[:n], fake, p)
        false_negatives = int(torch.count_nonzero(torch.round(p)))
        real = self._stage_cells(sampled_batch)
        eng.encode(real, out32=eng.gen_enc32[:n])
        eng.discriminate(eng.gen_enc32[:n], real, p)
        true_positives = int(torch.count_nonzero(torch.round(p)))
        return true_positives, n - false_negatives

    def _train_on_batch(self, substep, x, y):
        """Model.train_on_batch of one of the compiled graphs: runs that single sub-step and
        returns its loss (the target `y` is implied by the graph, as in the reference's calls
        :144-155)."""
        eng = self._require_engine()
        ops = _engine.ops
        if substep in (1, 4):
            enc, noise = x
            n = len(enc)
            eng.set_latents(enc, noise, n)
            cells = self._tile(n)
        elif substep == 2:
            cells_in, noise = x
            n = len(cells_in)
            eng.set_latents(np.zeros((n, self.encoding_size), np.float32), noise, n)
            cells = self._stage_cells(cells_in)
        else:
            n = len(x)
            eng.reserve(n)
            cells = self._stage_cells(x)
        ops.fill_f32(eng.loss_buf, 0.0)
        eng.substep(substep, cells)
        slot = {1: 0, 2: 1, 3: 2, 4: 3}[substep]
        return float(eng.loss_buf[slot])

    def _train_discriminator_on_batch(self, x, y):
        """`_discriminator.train_on_batch((encodings, cells), labels)`, reference :154-155.  The
        labels must be one constant vector (the reference only ever passes 0.95 * ones or
        zeros, :128-129): the loss kernel takes the label as a scalar."""
        import torch
        eng = self._require_engine()
        enc, cells = x
        labels = np.asarray(y, dtype=np.float32).reshape(-1)
        n = len(labels)
        if len(enc) != n or len(cells) != n:
            raise ValueError("train_on_batch: inputs and labels differ in length")
        if n and not np.all(labels == labels[0]):
            raise NotImplementedError("discriminator labels must be constant over the batch")
        eng.reserve(n)
        z = torch.as_tensor(np.asarray(enc, dtype=np.float32)).to(eng.device)
        ops = _engine.ops
        ops.fill_f32(eng.loss_buf, 0.0)
        eng.gen_enc32[:n].copy_(z)
        eng.train_discriminator(eng.gen_enc32[:n], self._stage_cells(cells), float(labels[0]), 5,
                                eng._drop_args(8, "D", None))
        ops.counter_add(eng.rng_counter, 1)
        return float(eng.loss_buf[5])


def _rows(x, lo, hi):
    """Rows [lo, hi) of a minibatch-like object (CellBatch, DataFrame, ndarray, tensor)."""
    if isinstance(x, CellBatch):
        return CellBatch(x.matrix, x.positions[lo:hi])
    if hasattr(x, "iloc"):
        return x.iloc[lo:hi]
    return x[lo:hi]


def _pack_numpy_state(st):
    """np.random.get_state() -> one uint32 array (npz-friendly, no pickle)."""
    name, keys, pos, has_gauss, cached = st
    assert name == "MT19937"
    tail = np.array([pos, has_gauss], dtype=np.uint32)
    g = np.frombuffer(np.float64(cached).tobytes(), dtype=np.uint32)
    return np.concatenate([np.asarray(keys, dtype=np.uint32), tail, g])


def _unpack_numpy_state(a):
    a = np.asarray(a, dtype=np.uint32)
    cached = float(np.frombuffer(a[626:628].tobytes(), dtype=np.float64)[0])
    return ("MT19937", a[:624].copy(), int(a[624]), int(a[625]), cached)


def _as_f32(a):
    import torch
    return torch.as_tensor(np.asarray(a, dtype=np.float32))


