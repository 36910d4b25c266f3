#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json): BiGAN train cells/sec and encode cells/sec on
synthetic 10x-shaped data, 30,000 cells x 33,694 genes, ContinuousCellBiGan, Z = 3.

    python bench.py --gpus N --steps K --warmup W [--batch B] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one `trainings_step` (six RMSprop updates + two predicts, reference
src/bigan_classify.py:126-155) on one batch of B cells per GPU.  Prints ONE JSON line.

  value     whole-job train cells/s with inputs resident in HBM (device CSR, device index and
            prior buffers), CUDA-event timed, max over ranks
  e2e       the same metric through the reference-facing Python API
            (`CellTraining.sample_cell_data` + `network.trainings_step`): host sampling,
            host->device copy of the batch indices and priors, device->host read of the losses
  roofline  dominant kernel (the tcgen05 GEMM family): algorithmic FLOPs of the step /
            summed GEMM kernel time, against the measured dense bf16 peak
  cpu_baseline / --impl reference   the oracle (torch-CPU restatement of the reference; TensorFlow
            is not installable here) on the host cores, bounded sample
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


class stdout_to_stderr:
    """stdout carries exactly one JSON line: while the process group / NCCL communicators come
    up, file descriptor 1 points at stderr, so the "NCCL version ..." banner that the library
    writes straight to stdout ends up there (measured: NCCL_DEBUG_FILE does not catch it)."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        try:                                     # C stdio buffers of the libraries as well
            import ctypes
            ctypes.CDLL(None).fflush(None)
        except Exception:
            pass
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def init_distributed(dev):
    """NCCL process group + first collective (creates the communicator) with stdout parked."""
    import torch
    import torch.distributed as dist
    with stdout_to_stderr():
        dist.init_process_group("nccl", device_id=dev)
        t = torch.zeros(1, device=dev)
        dist.all_reduce(t)
        torch.cuda.synchronize()


GENES, CELLS, Z = 33694, 30000, 3
FLOP_PER_CELL_TRAIN = 13.237e9      # SURVEY.md App. B (dense-equivalent 2*M*N*K, Continuous)
FLOP_PER_CELL_ENCODE = 0.3524e9
FLOP_PER_CELL_TRAIN_CLASSIFY = 8.057e9     # ClassifyCellBiGan (BASELINE.json configs[3])
FLOP_PER_CELL_ENCODE_CLASSIFY = 0.0684e9
Z_CLASSIFY = 10                     # synthetic cell types (SURVEY.md 8d config 4)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "hbm_gbs": p["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
                "source": "fallback (B200_PROFILING.md)"}


def gemm_traffic():
    """DRAM bytes per launch of the two GEMM sets, from the committed ncu pass over one step
    (profiles/r02_gemm_traffic.json, written by tools/summarize_traffic.py from
    profiles/r02_ncu_launches_b2048.csv)."""
    for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)
        except Exception:
            continue
    return {}


# ------------------------------------------------------------------------------ data
def synth_csr(n_cells, n_genes, seed, device):
    """10x-shaped synthetic counts as a CSR (SURVEY.md 8d config 2): nnz/cell ~
    clip(lognormal(ln 2000, 0.35), 200, 8000), Zipf-like gene popularity, counts
    1 + geometric(0.45), 1 % of entries x50; every gene gets >= 1 non-zero so the pivoted
    gene_size equals n_genes.  Built on the device (data synthesis is not timed)."""
    import numpy as np
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    rng = np.random.default_rng(seed)
    nnz_row = np.clip(np.round(rng.lognormal(np.log(2000.0), 0.35, n_cells)), 200,
                      min(8000, n_genes)).astype(np.int64)
    logp = -0.9 * torch.log(torch.arange(1, n_genes + 1, device=device, dtype=torch.float32))
    logp = logp[torch.randperm(n_genes, generator=g, device=device)]
    rowptr = np.zeros(n_cells + 1, dtype=np.int64)
    np.cumsum(nnz_row, out=rowptr[1:])
    kmax = int(nnz_row.max())
    nnz_dev = torch.from_numpy(nnz_row).to(device)
    parts = []
    chunk = 2048
    for s in range(0, n_cells, chunk):
        e = min(n_cells, s + chunk)
        u = torch.rand((e - s, n_genes), generator=g, device=device)
        keys = logp - torch.log(-torch.log(u.clamp_min(1e-20)))       # Gumbel top-k sampling
        # force gene j into cell j % n_cells so that no gene id is absent
        rows = torch.arange(s, e, device=device)
        for rep in range((n_genes + n_cells - 1) // n_cells):
            forced = rows + rep * n_cells
            ok = forced < n_genes
            keys[torch.nonzero(ok).flatten(), forced[ok]] = float("inf")
        top = torch.topk(keys, kmax, dim=1).indices
        keep = torch.arange(kmax, device=device)[None, :] < nnz_dev[s:e, None]
        top = torch.where(keep, top, torch.full_like(top, n_genes))   # drop the surplus picks
        top = torch.sort(top, dim=1).values                            # ascending, surplus last
        parts.append(top[keep.sum(1, keepdim=True) > torch.arange(kmax, device=device)[None, :]])
    colidx = torch.cat(parts).to(torch.int32)
    assert colidx.numel() == int(rowptr[-1])
    nnz = int(rowptr[-1])
    geo = torch.floor(torch.log(torch.rand(nnz, generator=g, device=device).clamp_min(1e-20)) /
                      float(np.log(1 - 0.45)))
    vals = 1.0 + geo
    big = torch.rand(nnz, generator=g, device=device) < 0.01
    vals = torch.where(big, vals * 50.0, vals)
    return rowptr, colidx.cpu().numpy(), vals.cpu().numpy().astype(np.float64)


def make_matrix(n_cells, n_genes, seed, device):
    import numpy as np
    from cellcomm_b200.cell_type_training import CellMatrix
    rowptr, colidx, vals = synth_csr(n_cells, n_genes, seed, device)
    return CellMatrix(rowptr, colidx, vals, np.arange(1, n_cells + 1), np.arange(1, n_genes + 1))


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                 "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------ CPU arm
def oracle_step_rate(batch, steps, warmup, genes, note, variant="cont", model=None):
    """cells/s of the oracle's trainings_step on the host cores (all threads)."""
    import torch
    from oracle import bigan_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    Z = Z_CLASSIFY if variant == "classify" else 3
    m = model if model is not None else O.OracleBiGan(variant, Z, genes, seed=0)
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(batch, genes, generator=g) < 0.06).float() * \
        (torch.poisson(torch.full((batch, genes), 1.2), generator=g) + 1)
    masks = O.make_masks(variant, Z, genes, batch, 1)
    times = []
    for i in range(warmup + steps):
        z, r = torch.rand(batch, Z, generator=g), torch.rand(batch, Z, generator=g)
        if variant == "classify":
            z = torch.nn.functional.one_hot(torch.randint(0, Z, (batch,), generator=g), Z).float()
        t0 = time.perf_counter()
        m.trainings_step(x, z, r, masks)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return {"value": batch / dt, "unit": "cells/s", "cores": torch.get_num_threads(),
            "kind": "port",
            "sample": f"{steps} trainings_step(s) of {batch} cells x {genes} genes, {note}; "
                      f"oracle = torch-CPU fp32 restatement of the reference's Keras step "
                      f"(TensorFlow 2.4 is not installable here)",
            "sec_per_step": dt}


def pick_sample_batch(batch, steps, genes, variant, budget_s, model=None):
    """The largest sample of the workload batch (batch, 1024, 512, 256, 128 cells) whose
    `steps` oracle steps fit the time budget, from one probe step at 128 cells (the oracle's
    time per step is affine in the batch: GEMMs scale with it, the optimiser sweep does not)."""
    probe = oracle_step_rate(min(128, batch), 1, 1, genes, "probe", variant, model)["sec_per_step"]
    for cand in (batch, 1024, 512, 256, 128):
        if cand <= batch and probe * max(1.0, cand / 128.0) * steps <= budget_s:
            return cand, probe
    return min(128, batch), probe


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  TensorFlow/Keras is
    not installed and cannot be (no network), so this times the oracle port on the host cores,
    rank 0 only.  Same `config` as the GPU arm (same matrix shape, networks and per-GPU batch);
    each timed step is a BOUNDED SAMPLE of that batch -- the largest of {batch, 1024, 512, 256,
    128} cells that keeps the whole run within --ref-budget seconds -- and the metric is the
    same cells/s.  (The oracle's cells/s grows slowly with the sample: its GEMMs are compute
    bound on the CPU at every one of these sizes and the batch-independent optimiser sweep is
    a few percent of a step.)"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "encode":
        return run_reference_encode(args)
    variant = "classify" if args.workload == "classify" else "cont"
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    from oracle import bigan_oracle as O
    model = O.OracleBiGan(variant, Z_CLASSIFY if variant == "classify" else 3, args.genes, seed=0)
    if args.ref_batch > 0:
        sample, probe = args.ref_batch, None
    else:
        sample, probe = pick_sample_batch(args.batch, steps + warmup, args.genes, variant,
                                          args.ref_budget, model)
    res = oracle_step_rate(sample, steps, warmup, args.genes,
                           f"a {sample}-cell sample of the GPU arm's {args.batch}-cell batch per "
                           f"step, same synthetic count model", variant, model)
    line = {
        "impl": "reference", "metric": "BiGAN train cells/sec", "value": res["value"],
        "unit": "cells/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": res["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.batch),
        "cpu_baseline": dict({k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
                             sample_cells_per_step=sample, probe_sec_per_128_cells=probe),
        "e2e": {"value": res["value"], "unit": "cells/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args, batch):
    classify = args.workload == "classify"
    return {"workload": (f"ClassifyCellBiGan trainings_step, {Z_CLASSIFY} synthetic cell types, "
                         if classify else "ContinuousCellBiGan trainings_step ") +
                        f"on synthetic 10x-shaped matrix {args.cells} cells x {args.genes} genes "
                        f"(BASELINE.json configs[{3 if classify else 1}])",
            "cells": args.cells, "genes": args.genes,
            "encoding_size": Z_CLASSIFY if classify else Z,
            "batch_per_gpu": batch, "l2_policy": "inputs larger than L2 (0.9-1.8 GB of bf16 "
            "weights streamed per update; every weight is rewritten between uses)"}


# ------------------------------------------------------------------------------ GPU arm
def dump_outputs(out_dir, losses, engine, rank, sample=1 << 20):
    """Write what the timed trainings_steps computed, for comparing two builds on the same
    inputs: `losses.npy`, the last step's (g, e, d) losses (float64), and `<G|E|D>_weights.npy`,
    each network's parameters after that step (float32) -- a fixed, seeded sample of `sample`
    entries of its weight arrays (Net.get_weights order) flattened and concatenated."""
    import numpy as np
    out = {"losses": np.asarray(losses, dtype=np.float64)}
    for name, n in engine.nets.items():
        ws = n.get_weights()          # collective in data-parallel runs: every rank calls it
        offs = np.cumsum([0] + [w.size for w in ws])
        pos = np.sort(np.random.default_rng(0).choice(offs[-1], min(sample, offs[-1]),
                                                      replace=False))
        which = np.searchsorted(offs, pos, side="right") - 1
        picked = np.empty(len(pos), dtype=np.float32)
        for i, w in enumerate(ws):
            m = which == i
            picked[m] = w.reshape(-1)[pos[m] - offs[i]]
        out[f"{name}_weights"] = picked
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for k, v in out.items():
            np.save(os.path.join(out_dir, k + ".npy"), v)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from cellcomm_b200 import engine as eng, ops
    from cellcomm_b200.cell_type_training import CellTraining

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_distributed(dev)
    # weak scaling (default): --batch cells per GPU; --strong: --batch is the global batch
    B = args.batch // world if args.strong else args.batch
    assert B >= 1 and (not args.strong or B * world == args.batch), "--strong: batch % gpus != 0"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    t_setup = time.time()
    data = make_matrix(args.cells, args.genes, 20260101, dev)
    assert data.shape == (args.cells, args.genes)
    classify = args.workload == "classify"
    Z = Z_CLASSIFY if classify else 3
    # the public API takes the GLOBAL batch: every rank draws the same permutation(N)[:B*world]
    # and trains on its contiguous B rows (CellTraining.run / trainings_step).  The trainer is
    # assembled here rather than by CellTraining(), which builds an unseeded Continuous variant
    # only: a fixed seed gives every run the same initial weights and device RNG key, so the
    # outputs of two builds can be compared (--dump-outputs).
    from cellcomm_b200.bigan_classify import ClassifyCellBiGan
    from cellcomm_b200.bigan_cont import ContinuousCellBiGan
    trainer = CellTraining.__new__(CellTraining)
    trainer.batch_size, trainer.data, trainer.batches_per_iteration = B * world, data, 10
    trainer.network = (ClassifyCellBiGan if classify else ContinuousCellBiGan)(
        Z, gene_size=args.genes, seed=0)
    net = trainer.network
    e = net._engine
    rowptr, colidx, values = data.device_csr(dev)
    setup_s = time.time() - t_setup

    # ---- device-resident loop: indices + priors already in HBM (each rank its own rows)
    n_pre = args.warmup + args.steps
    rs = np.random.RandomState(1000 + rank)
    idx_all = torch.stack([torch.from_numpy(rs.permutation(args.cells)[:B])
                           for _ in range(n_pre)]).to(dev)
    x16 = ops.alloc2d(B, args.genes, device=dev)
    e.reserve(B)

    graphed = None
    if args.graph and e.peer_graphable():     # one GPU, or the peer-memory data-parallel path
        graphed = e.capture_step((rowptr, colidx, values), args.genes, B,
                                 latents="host" if classify else "device")
    # classify prior: one-hot of a uniform category (src/bigan_classify.py:117-119), resident pool
    z_pool = None
    if classify:
        gz = torch.Generator(device=dev).manual_seed(7 + rank)
        z_pool = torch.nn.functional.one_hot(
            torch.randint(0, Z, (n_pre, B), generator=gz, device=dev), Z).float()
        r_pool = torch.rand((n_pre, B, Z), generator=gz, device=dev)

    def stage_latents(i):
        if classify:
            e.z32[:B].copy_(z_pool[i % n_pre], non_blocking=True)
            e.r32[:B].copy_(r_pool[i % n_pre], non_blocking=True)

    def eager_step(i):
        ops.gather_rows(rowptr, colidx, values, args.genes, row_idx=idx_all[i], out16=x16)
        if classify:
            stage_latents(i)
            ops.cast_f32_to_bf16(e.z32[:B], e.z16[:B])
            ops.cast_f32_to_bf16(e.r32[:B], e.r16[:B])
        else:
            e.draw_latents(B)
        return e.train_step(x16)

    def resident_step(i):
        if graphed is not None:
            graphed.idx.copy_(idx_all[i], non_blocking=True)
            stage_latents(i)
            return graphed.replay()
        return eager_step(i)

    for i in range(args.warmup):
        resident_step(i)
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    l0 = ops.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        losses = resident_step(args.warmup + i)
    e.join()                      # side-stream optimiser sweeps belong to the timed region
    ev1.record()
    barrier()
    launches = ops.launch_count() - l0
    if graphed is not None:
        launches = graphed.launches_per_replay * args.steps
    ms_resident = max_over_ranks(ev0.elapsed_time(ev1))
    last_losses = [float(v) for v in losses]
    if args.dump_outputs:         # before anything else trains the networks further
        dump_outputs(args.dump_outputs, last_losses, e, rank)

    # ---- the same step at the reference's default batch of 128 cells (src/__main__.py:44):
    # weight / optimiser streaming regime, HBM-bound; device-resident, same engine
    small = None
    if (world == 1 and args.small_batch and args.small_batch < B and graphed is not None
            and not classify):
        Bs = args.small_batch
        gs_small = e.capture_step((rowptr, colidx, values), args.genes, Bs, latents="device")
        idx_small = idx_all[:, :Bs].contiguous()
        for i in range(3):
            gs_small.idx.copy_(idx_small[i % n_pre], non_blocking=True)
            gs_small.replay()
        barrier()
        ev0.record()
        for i in range(args.steps):
            gs_small.idx.copy_(idx_small[i % n_pre], non_blocking=True)
            gs_small.replay()
        e.join()
        ev1.record()
        barrier()
        ms_small = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
        # ... and end to end through the public API at that batch (host sampling, H2D of the
        # indices + priors, three loss floats read back per step)
        for _ in range(2):
            [float(v) for v in net.trainings_step(data.sample(Bs))]
        barrier()
        ev0.record()
        for _ in range(args.steps):
            _ = [float(v) for v in net.trainings_step(data.sample(Bs))]
        e.join()
        ev1.record()
        barrier()
        ms_small_e2e = ev0.elapsed_time(ev1) / args.steps
        small = {"batch_per_gpu": Bs, "value": Bs * world / (ms_small / 1e3), "unit": "cells/s",
                 "ms_per_step": ms_small,
                 "e2e": {"value": Bs / (ms_small_e2e / 1e3), "unit": "cells/s",
                         "ms_per_step": ms_small_e2e, "h2d_bytes_per_step": Bs * 8 + 2 * Bs * 3 * 4,
                         "d2h_bytes_per_step": 12},
                 "note": "reference default batch; the step streams every weight and optimiser "
                         "slot once per update (26 B/parameter), so it is HBM-bound: "
                         f"{1.843e9 * 26 / 1e9:.1f} GB per step at the measured HBM peak = "
                         f"{1.843e9 * 26 / (peaks()['hbm_gbs'] * 1e9) * 1e3:.1f} ms"}

    # ---- end to end through the public API (host sampling, H2D indices+priors, D2H losses)
    np.random.seed(1000)
    net.sync_host_rng()           # data parallel: one global batch / prior stream on all ranks
    for _ in range(min(2, args.warmup)):
        [float(v) for v in net.trainings_step(trainer.sample_cell_data())]
    barrier()
    ev0.record()
    for _ in range(args.steps):
        g, el, d = net.trainings_step(trainer.sample_cell_data())
        _ = (float(g), float(el), float(d))           # the reference hands back host floats
    e.join()
    ev1.record()
    barrier()
    ms_e2e = max_over_ranks(ev0.elapsed_time(ev1))
    clock_info = clocks.stop() if rank == 0 else None

    # ---- the same call fed the way the reference feeds it: a dense float32 host batch (the
    # DataFrame.sample() rows, src/cell_type_training.py:37-38), 276 MB host->device per step
    dense_e2e = None
    if world == 1 and args.dense_e2e_steps > 0:
        xb = torch.empty((B, args.genes), dtype=torch.float32).pin_memory()
        xb.copy_(torch.from_numpy(trainer.sample_cell_data().to_numpy(np.float32)))
        xnp = xb.numpy()
        [float(v) for v in net.trainings_step(xnp)]
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.dense_e2e_steps):
            g, el, d = net.trainings_step(xnp)
            _ = (float(g), float(el), float(d))
        ev1.record()
        torch.cuda.synchronize()
        ms_dense = ev0.elapsed_time(ev1) / args.dense_e2e_steps
        dense_e2e = {"value": B / (ms_dense / 1e3), "unit": "cells/s", "ms_per_step": ms_dense,
                     "h2d_bytes_per_step": B * args.genes * 4 + 2 * B * Z * 4,
                     "d2h_bytes_per_step": 12, "steps": args.dense_e2e_steps,
                     "path": "network.trainings_step(float32 ndarray [B, genes]) from pinned host "
                             "memory: H2D copy of the dense batch + cast, eager step, losses read back"}

    if args.no_roofline:          # quick sweeps: the two train numbers only
        if rank == 0:
            print(json.dumps({
                "metric": "BiGAN train cells/sec", "unit": "cells/s", "n_gpus": world,
                "value": B * world * args.steps / (ms_resident / 1e3),
                "ms_per_step": ms_resident / args.steps, "steps": args.steps,
                "warmup": args.warmup, "clocks": clock_info,
                "e2e": {"value": B * world * args.steps / (ms_e2e / 1e3), "unit": "cells/s"},
                "config": workload_config(args, B), "partial": "--no-roofline"}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- encode-all-cells pass (E.predict over the whole matrix; each rank a row shard)
    shard = (args.cells + world - 1) // world
    r0, r1 = rank * shard, min(args.cells, (rank + 1) * shard)
    enc_out = torch.empty((r1 - r0, Z), dtype=torch.float32, device=dev)
    tile_rows = args.encode_tile

    def encode_shard():
        # cc_encode_stream: this rank's rows in one C call (gather + encoder forward per tile)
        e.encode_stream(rowptr, colidx, values, r0, r1, enc_out, tile_rows=tile_rows)

    encode_shard()
    barrier()
    ev0.record()
    for _ in range(args.encode_reps):
        encode_shard()
    ev1.record()
    barrier()
    ms_enc = max_over_ranks(ev0.elapsed_time(ev1)) / args.encode_reps
    def encode_e2e():
        # the DbRecorder's call, float32 host array; data parallel: rows sharded over the ranks,
        # (N_i, Z) pieces all-gathered (collective: every rank calls it)
        return net.encoding_prediction(data)

    encode_e2e()
    barrier()
    ev0.record()
    for _ in range(args.encode_reps):
        host_enc = encode_e2e()
    ev1.record()
    barrier()
    ms_enc_e2e = max_over_ranks(ev0.elapsed_time(ev1)) / args.encode_reps

    # ---- roofline of the dominant kernel family (tcgen05 GEMM).  One eager step is run with
    # every ops.gemm call recorded; the recorded launches (same descriptors, same buffers) are
    # then captured as a GEMM-only CUDA graph and its replay is timed with CUDA events: the
    # family's device time per step without the host launch gaps an eager event pair includes.
    # (All ranks run it: the eager step contains the data-parallel collectives.)
    real_gemm = ops.gemm
    calls, shapes = [], []

    def recording_gemm(*a, **k):
        calls.append((a, k))
        shapes.append((a[0], a[1], tuple(a[4]), a[5], a[6]))
        real_gemm(*a, **k)

    eager_step(0)                       # warm the eager path (the timed loop was a graph)
    e.join()
    torch.cuda.synchronize()
    ops.gemm = recording_gemm
    try:
        eager_step(1)
        e.join()
        torch.cuda.synchronize()
    finally:
        ops.gemm = real_gemm
    def time_calls(subset, reps=3):
        """CUDA-event time of `subset` re-issued as one CUDA graph (ms per replay)."""
        if not subset:
            return 0.0
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for a, k in subset:
                real_gemm(*a, **k)
        gr.replay()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            gr.replay()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / reps

    # launches whose epilogue applies RMSprop stream 26 B per parameter: HBM-bound, reported
    # against the HBM roofline; everything else is the tensor-bound set
    # (N > 128 selects the 256-wide, 8-epilogue-warp instantiation; the few tiny fused wgrads
    # stay in the first set, as in tools/summarize_traffic.py)
    is_fused = lambda c: c[1].get("rms") is not None and c[0][1] > 128
    fused_calls = [c for c in calls if is_fused(c)]
    plain_calls = [c for c in calls if not is_fused(c)]
    gemm_ms = [time_calls(calls), len(calls), time_calls(plain_calls), len(plain_calls),
               time_calls(fused_calls), len(fused_calls),
               sum(2.0 * a[0] * a[1] * a[4][0] for a, k in fused_calls),      # algorithmic FLOPs
               sum(26.0 * a[0] * a[1] for a, k in fused_calls)]               # algorithmic bytes
    # the same HBM roofline at the reference's batch: one recorded eager step of Bs cells, its
    # fused wgrad + RMSprop launches re-issued as a graph
    small_fused = None
    if small is not None:
        Bs = small["batch_per_gpu"]
        x16s = x16[:Bs]
        calls_s = []

        def small_step(i):
            ops.gather_rows(rowptr, colidx, values, args.genes, row_idx=idx_all[i][:Bs].contiguous(),
                            out16=x16s)
            e.draw_latents(Bs)
            return e.train_step(x16s)

        small_step(0)
        e.join()
        torch.cuda.synchronize()
        ops.gemm = lambda *a, **k: (calls_s.append((a, k)), real_gemm(*a, **k))[1]
        try:
            small_step(1)
            e.join()
            torch.cuda.synchronize()
        finally:
            ops.gemm = real_gemm
        fused_s = [c for c in calls_s if is_fused(c)]
        if fused_s:
            small_fused = (time_calls(fused_s), len(fused_s),
                           sum(26.0 * a[0] * a[1] for a, k in fused_s))
    table_path = os.environ.get("CELLCOMM_BENCH_GEMM_TABLE")
    if table_path and rank == 0:
        # per-shape table: each distinct launch replayed alone as a small graph
        agg = {}
        for c, sh in zip(calls, shapes):
            agg.setdefault(sh, []).append(c)
        rows = []
        for sh, cs in agg.items():
            gsh = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gsh):
                for a, k in cs:
                    real_gemm(*a, **k)
            gsh.replay()
            torch.cuda.synchronize()
            ev0.record()
            gsh.replay()
            gsh.replay()
            ev1.record()
            torch.cuda.synchronize()
            rows.append((ev0.elapsed_time(ev1) / 2, len(cs), sh))
        rows.sort(key=lambda r: -r[0])
        with open(table_path, "w") as f:
            for ms, n, (M_, N_, ks, am, bm) in rows:
                fl = 2.0 * M_ * N_ * sum(ks) * n
                f.write(f"{ms:8.3f} ms/step  n={n:3d}  M={M_:6d} N={N_:6d} K={ks} a_mn={am} "
                        f"b_mn={bm}  {fl / ms / 1e9:7.1f} TFLOP/s\n")
    if world > 1:
        barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    step_ms = ms_resident / args.steps
    value = B * world * args.steps / (ms_resident / 1e3)
    e2e_value = B * world * args.steps / (ms_e2e / 1e3)
    (gemm_total, gemm_launches, plain_ms, plain_launches, fused_ms, fused_launches, fused_flops,
     fused_bytes) = gemm_ms
    flops_step = (FLOP_PER_CELL_TRAIN_CLASSIFY if classify else FLOP_PER_CELL_TRAIN) * B
    flop_encode = FLOP_PER_CELL_ENCODE_CLASSIFY if classify else FLOP_PER_CELL_ENCODE
    # tensor-bound set: all Dense forward / dgrad GEMMs (+ the wgrads when the optimiser is not
    # fused); its algorithmic FLOPs are the step's minus the fused wgrads' share
    tensor_flops = flops_step - fused_flops
    achieved_tf = tensor_flops / (plain_ms / 1e3) / 1e12
    peak_tf = pk["bf16_tflops_sustained"]
    traffic = gemm_traffic()
    if small is not None and small_fused is not None:
        ms_f, n_f, bytes_f = small_fused
        small["roofline_hbm"] = {
            "bound": "hbm", "kernel": "wgrad GEMM with Keras RMSprop applied in the epilogue, "
            f"batch {small['batch_per_gpu']}",
            "achieved": bytes_f / (ms_f / 1e3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": bytes_f / (ms_f / 1e3) / 1e9 / pk["hbm_gbs"],
            "algorithmic_per_launch": bytes_f / n_f, "avg_launch_ms": ms_f / n_f,
            "ms_per_step": ms_f, "launches_per_step": n_f,
            "timing": "the fused launches of one step re-issued as a CUDA graph, CUDA events "
                      "around 3 replays"}
    line = {
        "metric": "BiGAN train cells/sec", "value": value, "unit": "cells/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
        "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": workload_config(args, B),
        "clocks": clock_info,
        "e2e": {"value": e2e_value, "unit": "cells/s",
                "h2d_bytes_per_step": B * 8 + 2 * B * Z * 4, "d2h_bytes_per_step": 12,
                "ms_per_step": ms_e2e / args.steps,
                "path": "CellTraining.sample_cell_data() + network.trainings_step(batch): host "
                        "numpy sampling, pageable->device copy of the batch indices and priors, "
                        "three loss floats read back per step"},
        "e2e_dense_host_batch": dense_e2e,
        "reference_batch": small,
        "gpu_launches": int(launches),
        "roofline": {
            "bound": "tensor",
            "kernel": "gemm_tcgen05_persistent_kernel (Dense fwd / dgrad GEMMs"
                      + ("" if fused_launches else " / wgrad") + ")",
            "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": achieved_tf / peak_tf,
            "traffic": traffic.get("tensor_bytes_per_launch"),
            "traffic_note": traffic.get("note"),
            "algorithmic_per_launch": tensor_flops / max(plain_launches, 1),
            "avg_launch_ms": plain_ms / max(plain_launches, 1),
            "peak_source": pk["source"] + ", sustained cuBLAS bf16 (kernel timed inside a long step)",
            "frac_of_burst_peak": achieved_tf / pk["bf16_tflops"],
            "flops_per_step_algorithmic": flops_step,
            "flops_per_step_in_these_launches": tensor_flops,
            "ms_per_step": plain_ms, "launches_per_step": plain_launches,
            "gemm_ms_per_step": gemm_total, "gemm_launches_per_step": gemm_launches,
            "gemm_share_of_step": gemm_total / step_ms,
            "timing": "all GEMM launches of one step re-issued as a GEMM-only CUDA graph, "
                      "CUDA events around 3 replays",
            "whole_step_tflops": flops_step / (step_ms / 1e3) / 1e12,
            "whole_step_frac": flops_step / (step_ms / 1e3) / 1e12 / peak_tf,
        },
        "roofline_hbm": None if not fused_launches else {
            "bound": "hbm",
            "kernel": "gemm_tcgen05_persistent_kernel<..., 8 epilogue warps> (wgrad GEMM with Keras "
                      "RMSprop applied in the epilogue)",
            "achieved": fused_bytes / (fused_ms / 1e3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": fused_bytes / (fused_ms / 1e3) / 1e9 / pk["hbm_gbs"],
            "traffic": traffic.get("fused_bytes_per_launch"),
            "algorithmic_per_launch": fused_bytes / fused_launches,
            "avg_launch_ms": fused_ms / fused_launches,
            "algorithmic_bytes_per_parameter": 26, "ms_per_step": fused_ms,
            "launches_per_step": fused_launches, "flops_per_step_in_these_launches": fused_flops,
            "peak_source": pk["source"] + ", HBM copy bandwidth"},
        "encode": {
            "metric": "encode cells/sec (E.predict over all cells)",
            "value": args.cells / (ms_enc / 1e3), "unit": "cells/s",
            "e2e": args.cells / (ms_enc_e2e / 1e3), "cells": args.cells,
            "tensor_frac": args.cells * flop_encode / (ms_enc / 1e3) / 1e12 /
            (peak_tf * world), "d2h_bytes": args.cells * Z * 4,
        },
        "losses_last_step": last_losses, "setup_seconds": setup_s,
        "cuda_graph": bool(graphed is not None),
        "precision_policy": "bf16 GEMM operands, fp32 accumulate; fp32 master weights + RMSprop "
                            "slots; CELLCOMM_B200_SPLIT=" + os.environ.get("CELLCOMM_B200_SPLIT", "auto"),
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = {k: v for k, v in oracle_step_rate(
            args.small_batch or 128, 3, 1, args.genes, "1 warm-up + 3 timed steps",
            "classify" if classify else "cont").items()
            if k != "sec_per_step"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------ train + record
def run_record(args):
    """BASELINE.json configs[2]: ContinuousCellBiGan training with the per-iteration
    encode-all-cells pass feeding `DbRecorder.intercept`, data parallel, through the product
    entry point `CellTraining.run` (what `python3 src` / `torchrun -m cellcomm_b200` executes;
    reference src/__main__.py:44-66, src/cell_type_training.py:40-50,
    src/intercepts/db_recorder.py:82-108).

    One "step" = one ITERATION of the reference loop: 10 `trainings_step`s on global batches of
    batch x gpus cells, then the interceptor on rank 0 -- encode all cells (rows sharded over
    the ranks), x255, duplicate groups, one `encits` document into the in-memory Mongo."""
    import tempfile
    import numpy as np
    import torch
    import torch.distributed as dist
    from cellcomm_b200 import intercepts, ops
    from cellcomm_b200.cell_type_training import CellTraining
    from cellcomm_b200.intercepts import db_recorder as dbr
    from cellcomm_b200.intercepts.fake_mongo import MongoClient as FakeMongo

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_distributed(dev)
    B = args.batch // world if args.strong else args.batch

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    data = make_matrix(args.cells, args.genes, 20260101, dev)
    np.random.seed(1000)
    trainer = CellTraining(data, batch_size=B * world, encoding_size=Z)
    net, bpi = trainer.network, trainer.batches_per_iteration
    icpt, spent = None, {"s": 0.0}
    if rank == 0:
        tmp = tempfile.mkdtemp(prefix="cellcomm_record_")
        src = {}
        for kind in dbr.SOURCE_KINDS:
            src[kind] = os.path.join(tmp, f"synthetic_{kind}.{'mtx' if kind == 'matrix' else 'tsv'}")
            open(src[kind], "w").close()
        FakeMongo(dbr.MONGO_URL).drop_database(dbr.MONGO_DB)
        rec = dbr.DbRecorder("bench-record", src, client_factory=FakeMongo)
        rec.store_encoding_run()
        rec.barcodes = [f"CELL{i:07d}-1" for i in range(args.cells)]   # (cells imported before)
        rec.cell_ids = list(range(1, args.cells + 1))
        record = rec.create_interceptor(trainer)

        def icpt(it, losses):
            torch.cuda.synchronize()          # the 10 queued steps are not interceptor time
            t0 = time.perf_counter()
            _ = [float(v) for v in losses]
            record(it, losses)
            spent["s"] += time.perf_counter() - t0

    it = 0
    for _ in range(max(1, min(args.warmup, 2))):
        trainer.run(1, icpt, start_iteration=it)
        it += 1
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    spent["s"] = 0.0
    l0 = ops.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        trainer.run(1, icpt, start_iteration=it)
        it += 1
    net._engine.join()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    launches = ops.launch_count() - l0
    gs = [g for g in net._engine._graphs.values()]
    if gs:
        launches += gs[0].launches_per_replay * bpi * args.steps
    if rank == 0:
        clock_info = clocks.stop()
        docs = FakeMongo(dbr.MONGO_URL)[dbr.MONGO_DB][dbr.ITERATIONS_COLLECTION].find(
            {"eid": "bench-record"}, {"_id": 0, "it": 1})
        cells_per_step = B * world * bpi
        value = cells_per_step * args.steps / (ms / 1e3)
        cfg = workload_config(args, B)
        cfg["workload"] = (f"ContinuousCellBiGan CellTraining.run: {bpi} trainings_steps + "
                           f"encode-all-cells + DbRecorder.intercept per iteration, "
                           f"{args.cells} cells x {args.genes} genes (BASELINE.json configs[2])")
        line = {
            "metric": "BiGAN train cells/sec", "value": value, "unit": "cells/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg,
            "clocks": clock_info, "gpu_launches": int(launches),
            "e2e": {"value": value, "unit": "cells/s",
                    "h2d_bytes_per_step": bpi * (B * 8 + 2 * B * world * Z * 4),
                    "d2h_bytes_per_step": bpi * 12 + args.cells * Z * 4,
                    "path": "CellTraining.run(1, DbRecorder interceptor): the whole timed region "
                            "IS the public API (host sampling, index/prior uploads, losses and "
                            "all encodings read back, documents built and stored)"},
            "record": {"iterations_recorded": len(docs), "cells_encoded_per_iteration": args.cells,
                       "interceptor_seconds_per_iteration": spent["s"] / args.steps,
                       "interceptor_share_of_step": spent["s"] * 1e3 / ms,
                       "store": "in-memory Mongo stand-in (mongod / pymongo are not in the image)"},
            "roofline": None, "cpu_baseline": None,
            "note": "configs[2] composite; the kernel rooflines are reported by the train and "
                    "encode workloads",
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------ encode-only
def run_encode(args):
    """BASELINE.json configs[4]: encode-only pass (E.predict, src/bigan_basic.py:29-30, the
    DbRecorder's call src/intercepts/db_recorder.py:85) over --encode-cells synthetic cells x
    33,694 genes, rows sharded contiguously over the GPUs, no communication.  A step = one pass
    over this rank's shard.  The 10x-shaped CSR is the 30k-cell synthetic matrix repeated."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from cellcomm_b200 import ops
    from cellcomm_b200.bigan_cont import ContinuousCellBiGan
    from cellcomm_b200.cell_type_training import CellMatrix

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_distributed(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    total = args.encode_cells
    shard = (total + world - 1) // world
    n_local = max(0, min(total, (rank + 1) * shard) - rank * shard)
    base_cells = min(args.cells, n_local)
    rp, ci, va = synth_csr(base_cells, args.genes, 20260102, dev)
    reps = (n_local + base_cells - 1) // base_cells
    nnz = int(rp[-1])
    rowptr = np.concatenate([rp[:-1] + k * nnz for k in range(reps)] + [[reps * nnz]])
    rowptr = rowptr[:n_local + 1].astype(np.int64)
    colidx = np.tile(ci, reps)[:rowptr[-1]]
    values = np.tile(va, reps)[:rowptr[-1]]
    data = CellMatrix(rowptr, colidx, values, np.arange(1, n_local + 1), np.arange(1, args.genes + 1))
    # every rank holds (only) its own row shard: the network is built without a process group,
    # so encoding_prediction(data) is this rank's pass over its shard -- no communication
    from cellcomm_b200 import engine as eng
    net = ContinuousCellBiGan(Z, gene_size=args.genes, dist=eng._NoDist())
    e = net._engine
    d_rowptr, d_colidx, d_values = data.device_csr(dev)
    tile_rows = args.encode_tile
    out = torch.empty((n_local, Z), dtype=torch.float32, device=dev)

    def one_pass():
        # cc_encode_stream: gather + encoder forward, tile by tile, ONE C call per pass
        e.encode_stream(d_rowptr, d_colidx, d_values, 0, n_local, out, tile_rows=tile_rows)

    steps, warm = max(1, args.steps), max(3, args.warmup)
    one_pass()
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    l0 = ops.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warm - 1):
        one_pass()
    barrier()
    ev0.record()
    for _ in range(steps):
        one_pass()
    ev1.record()
    barrier()
    launches = (ops.launch_count() - l0) * steps // (steps + warm - 1)
    ms = ev0.elapsed_time(ev1)
    # end to end: the public call, float32 host array back (12 B per cell D2H)
    net.encoding_prediction(data)
    barrier()
    ev0.record()
    for _ in range(steps):
        host = net.encoding_prediction(data)
    ev1.record()
    barrier()
    ms_e2e = ev0.elapsed_time(ev1)
    clock_info = clocks.stop() if rank == 0 else None
    assert host.shape == (n_local, Z) and np.isfinite(host).all()
    if world > 1:
        t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    if rank == 0:
        pk = peaks()
        value = total * steps / (ms / 1e3)
        tf = value * FLOP_PER_CELL_ENCODE / 1e12 / world
        line = {
            "metric": "encode cells/sec", "value": value, "unit": "cells/s", "n_gpus": world,
            "steps": steps, "warmup": warm, "ms_per_step": ms / steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"encode-only pass, {total} synthetic cells x {args.genes} genes, "
                                   f"ContinuousCellBiGan encoder (BASELINE.json configs[4])",
                       "cells": total, "genes": args.genes, "encoding_size": Z,
                       "tile_rows": tile_rows, "nnz_per_rank": int(rowptr[-1]),
                       "l2_policy": "inputs larger than L2 (CSR shard %.1f GB, bf16 tiles 276 MB, "
                                    "227 MB of encoder weights per tile)" % (rowptr[-1] * 8 / 1e9)},
            "clocks": clock_info,
            "e2e": {"value": total * steps / (ms_e2e / 1e3), "unit": "cells/s",
                    "h2d_bytes_per_step": 0, "d2h_bytes_per_step": n_local * Z * 4,
                    "path": "network.encoding_prediction(CellMatrix): device-resident CSR -> "
                            "float32 host array (the DbRecorder's call)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_persistent_kernel (encoder "
                         "forward GEMMs)", "achieved": tf, "peak": pk["bf16_tflops_sustained"],
                         "unit": "TFLOP/s", "frac": tf / pk["bf16_tflops_sustained"],
                         "traffic": None, "note": "whole-pass rate (gather + 5 GEMMs + BN); "
                         "0.3524 GFLOP per cell (SURVEY.md App. B)"},
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = oracle_encode_rate(args.genes)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def oracle_encode_rate(genes, cells=2048):
    """Oracle E.predict on the host cores: the reference's Keras predict batches 32 rows
    (SURVEY.md A.7); rows are independent in inference, so the port runs 256-row tiles."""
    import torch
    from oracle import bigan_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    m = O.OracleBiGan("cont", Z, genes, seed=0)
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(cells, genes, generator=g) < 0.06).float() * \
        (torch.poisson(torch.full((cells, genes), 1.2), generator=g) + 1)
    m.encoding_prediction(x[:256])
    t0 = time.perf_counter()
    for s_ in range(0, cells, 256):
        m.encoding_prediction(x[s_:s_ + 256])
    dt = time.perf_counter() - t0
    return {"value": cells / dt, "unit": "cells/s", "cores": torch.get_num_threads(),
            "kind": "port", "sample": f"{cells} cells x {genes} genes through the oracle's "
            f"encoding_prediction in 256-row tiles (torch-CPU fp32 restatement of E.predict)"}


def run_reference_encode(args):
    res = oracle_encode_rate(args.genes, cells=4096)
    print(json.dumps({
        "impl": "reference", "metric": "encode cells/sec", "value": res["value"],
        "unit": "cells/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": "encode-only pass (bounded sample)",
                                        "genes": args.genes},
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": "cells/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0}}), flush=True)


# ------------------------------------------------------------------------------ loader
def write_synthetic_mtx(path, n_cells, n_genes, seed):
    """10x-shaped MatrixMarket text (3 header lines, `gene barcode count`, barcode-major,
    genes ascending inside a barcode): ~2,000 non-zeros per cell.  Host only."""
    import numpy as np
    rng = np.random.default_rng(seed)
    nnz_row = np.clip(np.round(rng.lognormal(np.log(2000.0), 0.35, n_cells)), 200,
                      min(8000, n_genes)).astype(np.int64)
    rows = []
    for c in range(n_cells):
        g = np.sort(rng.choice(n_genes, nnz_row[c], replace=False)) + 1
        v = 1 + rng.geometric(0.45, nnz_row[c])
        rows.append(np.stack([g, np.full_like(g, c + 1), v], 1))
    coo = np.concatenate(rows)
    with open(path, "w") as f:
        f.write("%%MatrixMarket matrix coordinate integer general\n%\n")
        f.write(f"{n_genes} {n_cells} {len(coo)}\n")
        np.savetxt(f, coo, fmt="%d %d %d")
    return len(coo)


def run_loader(args):
    """SURVEY.md 8a row a1: `load_matrix` (src/cell_type_training.py:9-17) on a synthetic 10x
    .mtx: the C++ parser + compact-index CSR builder behind the C ABI (cc_mtx_load_csr) against
    the reference's own pandas body (oracle/loader_oracle.load_matrix_pandas) on the same file,
    results compared (bit-exact).  Host code: no GPU involved, no roofline."""
    import tempfile
    import numpy as np
    from cellcomm_b200.cell_type_training import load_matrix
    from oracle import loader_oracle as LO
    n_cells = args.loader_cells
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "matrix.mtx")
        nnz = write_synthetic_mtx(path, n_cells, args.genes, 20260103)
        size = os.path.getsize(path)
        load_matrix(path)
        times = []
        for _ in range(max(1, args.steps)):
            t0 = time.perf_counter()
            m = load_matrix(path)
            times.append(time.perf_counter() - t0)
        t_ours = min(times)
        t0 = time.perf_counter()
        ref = LO.load_matrix_pandas(path)
        t_ref = time.perf_counter() - t0
        same = (m.shape == ref.shape and
                np.array_equal(m.dense_rows(np.arange(min(64, n_cells))),
                               ref.values[:min(64, n_cells)].astype(np.float64)))
    print(json.dumps({
        "metric": "load_matrix nnz/sec", "value": nnz / t_ours, "unit": "nnz/s", "n_gpus": 0,
        "steps": args.steps, "warmup": 1, "ms_per_step": t_ours * 1e3, "higher_is_better": True,
        "scaling": "n/a", "vs_baseline": None, "dtype": "int64/f64", "data": "synthetic",
        "config": {"workload": f"load_matrix on a synthetic 10x .mtx, {n_cells} cells x "
                               f"{args.genes} genes, {nnz} non-zeros, {size / 1e6:.0f} MB of text",
                   "cells": n_cells, "genes": args.genes},
        "file_MB_per_s": size / t_ours / 1e6, "matches_reference_pandas_body": bool(same),
        "cpu_baseline": {"value": nnz / t_ref, "unit": "nnz/s", "cores": 1, "kind": "reference",
                         "sample": "the reference's pandas read_csv + pivot_table body on the same "
                                   "file (oracle/loader_oracle.load_matrix_pandas), one pass",
                         "seconds": t_ref},
        "roofline": None, "gpu_launches": 0}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("CELLCOMM_BENCH_BATCH", "2048")),
                    help="cells per GPU per trainings_step (reference default 128; 2048 saturates "
                         "the tensor cores)")
    ap.add_argument("--ref-budget", type=float, default=240.0,
                    help="--impl reference: seconds of oracle work the whole run may take")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: --batch is the GLOBAL batch, split over the GPUs")
    ap.add_argument("--ref-batch", type=int, default=0,
                    help="batch of the CPU arm's bounded sample (the reference's default)")
    ap.add_argument("--cells", type=int, default=CELLS)
    ap.add_argument("--genes", type=int, default=GENES)
    ap.add_argument("--encode-tile", type=int, default=4096)
    ap.add_argument("--encode-reps", type=int, default=2)
    ap.add_argument("--loader-cells", type=int, default=2000)
    ap.add_argument("--workload", default="train", choices=["train", "classify", "encode", "loader", "record"],
                    help="train: ContinuousCellBiGan trainings_step (BASELINE configs[1], the "
                         "headline); classify: ClassifyCellBiGan (configs[3]); encode: the "
                         "encode-only pass over --encode-cells cells (configs[4]); loader: "
                         "load_matrix on a synthetic .mtx (host C++ vs the reference's pandas)")
    ap.add_argument("--encode-cells", type=int, default=1_000_000)
    ap.add_argument("--small-batch", type=int, default=128,
                    help="also time the step at this (the reference's default) batch; 0: skip")
    ap.add_argument("--dense-e2e-steps", type=int, default=3,
                    help="steps of the dense-host-batch end-to-end variant (0: skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true",
                    help="train numbers only (tuning sweeps); the driver's runs never pass this")
    ap.add_argument("--graph", type=int, default=int(os.environ.get("CELLCOMM_BENCH_GRAPH", "1")),
                    help="1: run the device-resident loop as one CUDA graph per step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="train / classify: after the timed steps, write the last step's losses "
                         "and a seeded sample of the updated weights to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("train", "classify")):
        ap.error("--dump-outputs needs --impl ours and --workload train or classify")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload == "loader":
        run_loader(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.workload == "encode":
        run_encode(args)
    elif args.workload == "record":
        run_record(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
