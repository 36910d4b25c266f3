"""Deterministic mode on the GPU: the fixed-order column reductions and MSE loss are accurate
and bit-identical from launch to launch (also after a CUDA-graph replay), and a seeded
deterministic run -- engine steps, graph vs eager, checkpoint -> resume, bench.py
--dump-outputs, `python -m cellcomm_b200` -- repeats bit for bit."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

WIDTHS = [1, 3, 50, 256, 3369, 6738, 33694]
ROWS = [128, 2048]


def _ops():
    from cellcomm_b200 import ops
    return ops


def _rand(rows, cols, seed, dtype):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(rows, cols, generator=g, device="cuda").to(dtype)


def _ws(rows, cols):
    ops = _ops()
    return torch.zeros(ops.reduce_ws_floats(rows, cols), dtype=torch.float32, device="cuda")


def _repeatable(run):
    """run() -> tuple of tensors.  Two eager launches, then a CUDA-graph capture + replay, then
    another eager launch: all bit-identical (the graph replay leaves the tickets at zero)."""
    first = [t.clone() for t in run()]
    again = run()
    assert all(torch.equal(a, b) for a, b in zip(first, again))
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g):
        captured = run()
    g.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(first, captured))
    after = run()
    assert all(torch.equal(a, b) for a, b in zip(first, after))
    return first


def _close(got, ref, rows, scale=1.0):
    err = (got.double() - ref).abs()
    tol = 1e-4 * ref.abs() + 1e-5 * rows ** 0.5 * scale
    assert bool((err <= tol).all()), float(err.max())


def _layout(rows, cols):
    """(ticket counters, row slabs) of a column reduction: the launch geometry of
    tail_kernels.cu (column blocks of 128; slabs to fill 2 x SMs CTAs, at least 64 rows each)"""
    tickets = 2 * torch.cuda.get_device_properties(0).multi_processor_count
    gx = -(-cols // 128)
    gy = 1 if gx >= tickets else max(1, min(-(-tickets // gx), -(-rows // 64)))
    return tickets, gy


def _check_partials(ws, rows, cols, outs):
    """The fixed-order path ran: the workspace holds one row of per-column partials per slab
    (per output), they add up to the results, and every ticket counter is back at zero."""
    tickets, gy = _layout(rows, cols)
    assert gy > 1
    assert bool((ws[:tickets] == 0).all())
    part = ws[tickets:tickets + len(outs) * gy * cols].view(len(outs), gy, cols).double()
    for k, o in enumerate(outs):
        _close(o, part[k].sum(0), rows)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("rows", ROWS)
def test_colsum_bn_stats_bn_bwd_stats(rows, cols, dtype):
    ops = _ops()
    x = _rand(rows, cols, 1, dtype)
    dy = _rand(rows, cols, 2, dtype)
    mean = torch.randn(cols, device="cuda") * 0.1
    rstd = torch.rand(cols, device="cuda") + 0.5
    ws = _ws(rows, cols)
    xd, dyd = x.double(), dy.double()
    xhat = (xd - mean.double()) * rstd.double()

    cs, cs1 = torch.empty(cols, device="cuda"), torch.empty(cols, device="cuda")
    st, bw = torch.empty(2 * cols, device="cuda"), torch.empty(2 * cols, device="cuda")

    def run_colsum():
        ops.colsum(x, cs, ws=ws)
        cs1.fill_(1.0)
        ops.colsum(x, cs1, beta=1, ws=ws)
        return cs, cs1
    got = _repeatable(run_colsum)
    _close(got[0], xd.sum(0), rows)
    _close(got[1], 1.0 + xd.sum(0), rows)
    _check_partials(ws, rows, cols, [got[0]])

    def run_stats():
        ops.bn_stats(x, st, ws=ws)
        return (st,)
    got = _repeatable(run_stats)
    _close(got[0][:cols], xd.sum(0), rows)
    _close(got[0][cols:], (xd * xd).sum(0), rows)
    _check_partials(ws, rows, cols, [got[0][:cols], got[0][cols:]])

    def run_bwd():
        ops.bn_bwd_stats(dy, x, mean, rstd, bw, ws=ws)
        return (bw,)
    got = _repeatable(run_bwd)
    _close(got[0][:cols], dyd.sum(0), rows)
    _close(got[0][cols:], (dyd * xhat).sum(0), rows, scale=2.0)
    _check_partials(ws, rows, cols, [got[0][:cols], got[0][cols:]])

    # the atomic path agrees within the same tolerance
    ref = torch.empty(2 * cols, device="cuda")
    ops.bn_stats(x, ref)
    _close(ref[:cols], xd.sum(0), rows)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("rows", ROWS)
def test_bias_grad(rows, cols, dtype):
    ops = _ops()
    dy = _rand(rows, cols, 3, dtype)
    yr = _rand(rows, cols, 4, torch.float32)
    ws = _ws(rows, cols)
    for act in (0, 1, 2):
        y = (torch.sigmoid(yr) if act == 1 else yr).to(dtype)
        yd = y.double()
        d = {0: torch.ones_like(yd), 1: yd * (1 - yd), 2: (yd > 0).double()}[act]
        ref = (dy.double() * d).sum(0)
        for beta in (0, 1):
            out = torch.empty(cols, device="cuda")
            dz = torch.empty(rows, cols, device="cuda", dtype=torch.bfloat16)
            dz_lo = torch.empty_like(dz)

            def run(dz_lo_=dz_lo):
                out.fill_(0.25)
                ops.bias_grad(dy, y, act, out, dz=dz, beta=beta, dz_lo=dz_lo_, ws=ws)
                return out, dz, dz_lo
            got = _repeatable(run)
            _close(got[0], ref + (0.25 if beta else 0.0), rows)
            _check_partials(ws, rows, cols, [got[0] - (0.25 if beta else 0.0)])
            # dz / dz_lo are elementwise stores: identical to the atomic path's
            out_a = torch.full((cols,), 0.25, device="cuda")
            dz_a, dz_lo_a = torch.empty_like(dz), torch.empty_like(dz_lo)
            ops.bias_grad(dy, y, act, out_a, dz=dz_a, beta=beta, dz_lo=dz_lo_a)
            assert torch.equal(dz_a, got[1]) and torch.equal(dz_lo_a, got[2])
            _close(out_a, ref + (0.25 if beta else 0.0), rows)
        # fp32 dz without a low-order term, and a dz-only call (out = None): same dz
        dz32, dz32b = torch.empty(rows, cols, device="cuda"), torch.zeros(rows, cols, device="cuda")
        out = torch.empty(cols, device="cuda")
        ops.bias_grad(dy, y, act, out, dz=dz32, ws=ws)
        _close(out, ref, rows)
        ops.bias_grad(dy, y, act, None, dz=dz32b, ws=ws)
        assert torch.equal(dz32, dz32b)
        if act == 0:
            assert torch.equal(dz32, dy.float())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("rows", ROWS)
def test_mse(rows, cols, dtype):
    ops = _ops()
    pred = _rand(rows, cols, 5, dtype)
    target = _rand(rows, cols, 6, dtype)
    ws = _ws(rows, cols)
    loss = torch.empty(1, device="cuda")
    dp = torch.empty(rows, cols, device="cuda")

    def run():
        loss.fill_(0.5)
        ops.mse_fwd_bwd(pred, rows, loss, target=target, dpred=dp, ws=ws)
        return loss, dp
    got = _repeatable(run)
    ref = ((pred.double() - target.double()) ** 2).mean()
    assert abs(float(got[0]) - 0.5 - float(ref)) <= 1e-5 * float(ref) + 1e-6
    # the fixed-order path ran: per-block partial sums of squares after the ticket counters
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    work = rows * -(-cols // 8)                 # 8-column chunks, 256 per block, <= 8 x SMs
    blocks = max(1, min(-(-work // 256), 8 * sms))
    assert bool((ws[:2 * sms] == 0).all())
    total = float(ws[2 * sms:2 * sms + blocks].double().sum()) / (rows * cols)
    assert abs(total - float(ref)) <= 1e-5 * float(ref) + 1e-6
    loss_a, dp_a = torch.zeros(1, device="cuda"), torch.empty_like(dp)
    ops.mse_fwd_bwd(pred, rows, loss_a, target=target, dpred=dp_a)
    assert torch.equal(dp_a, got[1])


def test_workspace_too_small_is_an_error():
    ops = _ops()
    from cellcomm_b200._lib import CCError
    x = _rand(2048, 256, 7, torch.float32)
    need = ops.reduce_ws_floats(2048, 256)
    assert need > 0
    small = torch.zeros(need // 2, device="cuda")
    with pytest.raises(CCError, match="workspace"):
        ops.colsum(x, torch.empty(256, device="cuda"), ws=small)
    with pytest.raises(CCError, match="workspace"):
        ops.mse_fwd_bwd(x, 2048, torch.zeros(1, device="cuda"), target=x, ws=torch.zeros(4, device="cuda"))
    # a bound for a larger shape serves every smaller one
    big = _ws(2048, 33694)
    for cols in WIDTHS:
        out = torch.empty(2 * cols, device="cuda")
        ops.bn_stats(_rand(2048, cols, 8, torch.float32), out, ws=big)
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------- engine
def _csr(N, G, seed):
    from cellcomm_b200.cell_type_training import CellMatrix
    rng = np.random.default_rng(seed)
    dense = (rng.random((N, G)) < 0.06) * (rng.poisson(1.2, (N, G)) + 1)
    return CellMatrix.from_dense(dense.astype(np.float64)).device_csr("cuda")


def _state(e):
    out = {}
    for k, n in e.nets.items():
        n._rows()
        out[k + ".p32"], out[k + ".ms"], out[k + ".mom"] = n.p32, n.ms, n.mom
        out[k + ".p16"] = n.p16
        if n.p16lo is not None:
            out[k + ".p16lo"] = n.p16lo
        for i, L in enumerate(L for L in n.layers if L["kind"] == "bn"):
            out[f"{k}.bn{i}.mean"], out[f"{k}.bn{i}.var"] = L["moving_mean"], L["moving_var"]
    return {k: v.clone() for k, v in out.items()}


def _assert_same(a, b):
    assert a.keys() == b.keys()
    bad = [k for k in a if not torch.equal(a[k], b[k])]
    assert not bad, bad


def _run_engine(G, B, steps, csr, mode, fused=True):
    from cellcomm_b200 import engine as eng, ops
    e = eng.BiGanEngine("cont", 3, G, max_batch=B, device="cuda", seed=13, deterministic=True)
    e.set_fused_optimizer(fused)
    rs = np.random.RandomState(99)
    losses = []
    if mode == "graph":
        gs = e.capture_step(csr, G, B)
        for _ in range(steps):
            out = gs.replay(torch.from_numpy(rs.permutation(csr[0].numel() - 1)[:B]).cuda())
            losses.append([float(v) for v in out])
    else:
        idx = torch.zeros(B, dtype=torch.int64, device="cuda")
        x16 = ops.alloc2d(B, G, device="cuda")
        for _ in range(steps):
            idx.copy_(torch.from_numpy(rs.permutation(csr[0].numel() - 1)[:B]))
            ops.gather_rows(*csr, G, row_idx=idx, out16=x16)
            e.draw_latents(B)
            out = e.train_step(x16)
            e.join()
            losses.append([float(v) for v in out])
    x = ops.alloc2d(B, G, device="cuda")
    ops.gather_rows(*csr, G, row_idx=torch.arange(B, device="cuda"), out16=x)
    enc = torch.empty(B, 3, device="cuda")
    e.encode(x, out32=enc)
    torch.cuda.synchronize()
    st = _state(e)
    st["losses"] = torch.tensor(losses, dtype=torch.float64)
    st["encoding"] = enc.clone()
    # every reduction left its ticket counters at zero for the next step
    n_tickets = 2 * torch.cuda.get_device_properties(0).multi_processor_count
    assert bool((e.reduce_ws[:n_tickets] == 0).all())
    return st


@pytest.mark.parametrize("G,fused", [(6000, True), (6000, False), (33694, True)])
def test_engine_runs_are_bit_identical(G, fused):
    B, steps = 128, 3
    csr = _csr(300, G, seed=G)
    a = _run_engine(G, B, steps, csr, "graph", fused)
    b = _run_engine(G, B, steps, csr, "graph", fused)
    _assert_same(a, b)
    c = _run_engine(G, B, steps, csr, "eager", fused)
    _assert_same(a, c)                      # the captured step launches the same kernels
    assert np.isfinite(a["losses"].numpy()).all()


def test_reduction_on_the_optimiser_stream_is_refused():
    """One workspace serves a step only while every reduction runs on the main stream."""
    from cellcomm_b200 import engine as eng
    e = eng.BiGanEngine("cont", 3, 300, max_batch=8, device="cuda", seed=1, deterministic=True)
    side = e.G.opt_stream
    if side is None:
        pytest.skip("CELLCOMM_B200_ASYNC_OPT=0: no optimiser side stream")
    assert e.G._reduce_args()["ws"] is e.reduce_ws
    with torch.cuda.stream(side):
        with pytest.raises(AssertionError, match="side stream"):
            e.G._reduce_args()
        with pytest.raises(AssertionError, match="side stream"):
            e._reduce_args()


@pytest.mark.parametrize("G", [1000, 6000])
def test_checkpoint_resume_is_bit_identical(tmp_path, monkeypatch, G):
    monkeypatch.setenv("CELLCOMM_B200_DETERMINISTIC", "1")
    from cellcomm_b200 import intercepts
    from cellcomm_b200.cell_type_training import CellMatrix, CellTraining
    N, B = 180, 32
    rng = np.random.default_rng(6)
    dense = ((rng.random((N, G)) < 0.06) * (rng.poisson(1.2, (N, G)) + 1))
    data = CellMatrix.from_dense(dense.astype(np.float64))
    ck = intercepts.Checkpoints(str(tmp_path / "logs"))

    np.random.seed(21)
    a = CellTraining(data, batch_size=B, encoding_size=3, batches_per_iteration=2, seed=21)
    assert a.network._engine.deterministic
    seen_a = []
    a.run(2, intercepts.combined_interceptors((
        lambda it, l: seen_a.append((it, [float(v) for v in l])), ck.create_interceptor(a))))
    os.rename(ck.path, ck.path + ".keep")
    a.run(1, lambda it, l: seen_a.append((it, [float(v) for v in l])), start_iteration=2)
    os.rename(ck.path + ".keep", ck.path)
    enc_a = a.network.encoding_prediction(data)

    np.random.seed(12345)                   # everything below comes from the file
    b = CellTraining(data, batch_size=B, encoding_size=3, batches_per_iteration=2, seed=999)
    start = ck.resume(b)
    assert start == 2
    seen_b = []
    b.run(1, lambda it, l: seen_b.append((it, [float(v) for v in l])), start_iteration=start)
    assert seen_b == [seen_a[2]]
    _assert_same(_state(a.network._engine), _state(b.network._engine))
    assert np.array_equal(enc_a, b.network.encoding_prediction(data))


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "4",
           "--warmup", "3", "--cells", "600", "--genes", "1500", "--batch", "64",
           "--encode-tile", "256", "--small-batch", "0", "--dense-e2e-steps", "0",
           "--no-cpu-baseline", "--dump-outputs", out_dir]
    env = dict(os.environ, CELLCOMM_B200_DETERMINISTIC="1")
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]


def test_bench_dumps_are_bit_identical(tmp_path):
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    _bench(a)
    _bench(b)
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b)) and "losses.npy" in names
    for name in names:
        assert np.array_equal(np.load(os.path.join(a, name)), np.load(os.path.join(b, name))), name


def _entry_losses(tmp, cmd):
    from test_entry_point_gpu import _write_data_dir
    os.makedirs(tmp)
    _write_data_dir(tmp)
    env = dict(os.environ, CELLCOMM_DATA_DIR=tmp, CELLCOMM_ITERATIONS="2", CELLCOMM_BATCH_SIZE="16",
               CELLCOMM_SEED="7", CELLCOMM_B200_DETERMINISTIC="1",
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "src"), ROOT]))
    out = subprocess.run(cmd, cwd=tmp, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-3000:])
    runs = os.listdir(os.path.join(tmp, "logs"))
    assert len(runs) == 1
    with open(os.path.join(tmp, "logs", runs[0], "losses.csv"), "rb") as f:
        return f.read()


def test_entry_point_repeats_with_a_seed(tmp_path):
    cmd = [sys.executable, "-m", "cellcomm_b200"]
    a = _entry_losses(str(tmp_path / "a"), cmd)
    b = _entry_losses(str(tmp_path / "b"), cmd)
    assert a == b and a.count(b"\n") == 3


def test_entry_point_repeats_with_a_seed_under_torchrun(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29500 + (os.getpid() % 200)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(port), "-m", "cellcomm_b200"]
    a = _entry_losses(str(tmp_path / "a"), cmd)
    b = _entry_losses(str(tmp_path / "b"), cmd)
    assert a == b and a.count(b"\n") == 3
