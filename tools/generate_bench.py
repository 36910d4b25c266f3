"""Streamed generation on one GPU: the device pass of BiGanEngine.generate_csr and an end-to-end
A/B of generate_cell_matrix (sparse, streamed) against generate_cells (dense), at 33,694 genes
on a seeded ContinuousCellBiGan (Z = 3).  Writes one JSON file with the card's name and power
limit read in the same run.

    python tools/generate_bench.py --out profiles/r04_generate_stream.json

Device pass (--cells, default 2^20): generator forward + cc_round_csr_count + cc_round_csr_fill
+ cudaMemcpyAsync into reused pinned staging, per 4096-cell tile, nothing accumulated on the
host; host clock around a synchronised pass.  Separately, with CUDA events over repeated
launches on one 4096-row tile: the generator forward (GEMM FLOPs from the graph's Dense shapes,
against bench.peaks()) and the two compaction kernels (algorithmic bytes 8*rows*cols read +
8*nnz + 8*rows written, against the measured 6.47 TB/s copy bandwidth).

End to end (--e2e-cells, default 32,768): each arm runs in a fresh process, alternating; wall
time of the call, and its peak host bytes = the largest RSS sampled every millisecond during the
call minus the RSS just before it.
"""
import argparse
import json
import os
import resource
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

G, Z, TILE = 33694, 3, 4096
COPY_GBS = 6472.1       # measured B200 HBM copy bandwidth (SURVEY.md, profiles/README.md)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def network(expressed=0.0, seed=0):
    """seeded, untrained ContinuousCellBiGan.  Its rounded output is almost all zeros (about 40
    non-zeros per cell); expressed > 0 raises the output bias of that fraction of the genes
    (a seeded choice) by 2, so that about expressed * genes entries per cell are non-zero, the
    density of a 10x matrix at expressed = 0.06."""
    import numpy as np
    from cellcomm_b200.bigan_cont import ContinuousCellBiGan
    net = ContinuousCellBiGan(Z, G, seed=seed)
    if expressed > 0:
        gen = net._engine.G
        w = gen.get_weights()
        w[-1] = w[-1] + 2.0 * (np.random.default_rng(seed).random(G) < expressed)
        gen.set_weights(w)
    return net


def priors(n, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    return rng.random((n, Z), dtype=np.float32), rng.random((n, Z), dtype=np.float32)


def graph_flops_per_cell(eng):
    """2 * K * N of every Dense layer of the generator graph (hi + lo operand terms are extra
    tensor-core work that this count leaves out)"""
    g = eng.G.g
    total = 0
    for node in g.nodes:
        if node["kind"] == "dense":
            total += 2 * sum(g.widths[i] for i in node["ins"]) * g.widths[node["out"]]
    return total


def events_ms(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def device_pass(args, expressed):
    import torch
    import bench
    from cellcomm_b200 import ops
    net = network(expressed)
    eng = net._engine
    # one 4096-row tile: generator forward and compaction kernels on their own
    z, r = priors(TILE, 1)
    eng.set_latents(z, r, TILE)
    tile = ops.alloc2d(TILE, G, dtype=torch.float32, device="cuda", zero=False)
    fwd_ms = events_ms(lambda: eng.generate(TILE, out32=tile), args.reps)
    rowptr = torch.zeros(TILE + 1, dtype=torch.int64, device="cuda")
    ops.round_csr_count(tile, rowptr)
    nnz_tile = int(rowptr[-1])
    col = torch.empty(max(nnz_tile, 1), dtype=torch.int32, device="cuda")
    val = torch.empty(max(nnz_tile, 1), dtype=torch.float32, device="cuda")
    count_ms = events_ms(lambda: ops.round_csr_count(tile, rowptr), args.reps)
    fill_ms = events_ms(lambda: ops.round_csr_fill(tile, rowptr, col[:nnz_tile],
                                                   val[:nnz_tile]), args.reps)
    del tile, col, val
    flops = graph_flops_per_cell(eng) * TILE
    pk = bench.peaks()
    compact_bytes = 8 * TILE * G + 8 * nnz_tile + 8 * TILE
    compact_ms = count_ms + fill_ms

    # the whole streamed pass, nothing kept on the host
    z, r = priors(args.cells, 2)
    seen = {"nnz": 0}

    def consume(row0, rp, colidx, values):
        seen["nnz"] += int(rp[-1])

    eng.generate_csr(z[:2 * TILE], r[:2 * TILE], consume=lambda *a: None)     # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.generate_csr(z, r, consume=consume)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return {
        "expressed_genes_raised": expressed,
        "cells": args.cells,
        "cells_per_s": args.cells / wall,
        "wall_s": wall,
        "nnz_per_cell": seen["nnz"] / args.cells,
        "tile_4096": {
            "generator_forward_ms": fwd_ms,
            "gemm_graph_flops": flops,
            "gemm_tflops": flops / fwd_ms / 1e9,
            "bf16_peak_tflops": pk["bf16_tflops"],
            "gemm_fraction_of_bf16_peak": flops / fwd_ms / 1e9 / pk["bf16_tflops"],
            "peaks_source": pk["source"],
            "nnz": nnz_tile,
            "count_ms": count_ms,
            "fill_ms": fill_ms,
            "compaction_bytes": compact_bytes,
            "compaction_gbs": compact_bytes / compact_ms / 1e6,
            "compaction_fraction_of_copy_bw": compact_bytes / compact_ms / 1e6 / COPY_GBS,
            "compaction_fraction_of_forward": compact_ms / fwd_ms,
        },
    }


def _rss():
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


def arm(name, cells, expressed):
    """one end-to-end call in this process -> JSON on stdout"""
    import numpy as np
    import torch
    net = network(expressed)
    z, r = priors(cells, 3)
    net.generate_cells(z[:TILE], r[:TILE])                     # warm-up (both arms alike)
    torch.cuda.synchronize()
    before = _rss()
    peak, done = [before], threading.Event()

    def sample():                    # RSS every millisecond while the call runs
        while not done.is_set():
            peak[0] = max(peak[0], _rss())
            time.sleep(0.001)

    th = threading.Thread(target=sample)
    th.start()
    t0 = time.perf_counter()
    if name == "sparse":
        out = net.generate_cell_matrix(z, r)
    else:
        out = net.generate_cells(z, r)
    wall = time.perf_counter() - t0
    done.set()
    th.join()
    peak[0] = max(peak[0], _rss())
    nnz = out.nnz if name == "sparse" else int(np.count_nonzero(out))
    print(json.dumps({"arm": name, "wall_s": wall, "peak_host_bytes": peak[0] - before,
                      "nnz": nnz}))


def e2e(args):
    rows = []
    for rep in range(args.e2e_reps):
        for name in ("sparse", "dense") if rep % 2 == 0 else ("dense", "sparse"):
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--arm", name,
                                "--e2e-cells", str(args.e2e_cells), "--expressed",
                                str(args.expressed)], capture_output=True,
                               text=True, cwd=ROOT, timeout=900)
            if p.returncode != 0:
                raise SystemExit(f"arm {name} failed:\n{p.stderr[-3000:]}")
            rows.append(json.loads(p.stdout.strip().splitlines()[-1]))

    def med(name, key):
        v = sorted(x[key] for x in rows if x["arm"] == name)
        return v[len(v) // 2]

    return {"cells": args.e2e_cells, "expressed_genes_raised": args.expressed, "runs": rows,
            "median_wall_s": {a: med(a, "wall_s") for a in ("sparse", "dense")},
            "median_peak_host_bytes": {a: med(a, "peak_host_bytes") for a in ("sparse", "dense")},
            "speedup_sparse_over_dense": med("dense", "wall_s") / med("sparse", "wall_s")}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--cells", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--e2e-cells", type=int, default=32768)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_generate_stream.json"))
    ap.add_argument("--expressed", type=float, default=0.06,
                    help="end to end: fraction of genes with a raised output bias")
    ap.add_argument("--arm", choices=("sparse", "dense"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.arm:
        arm(args.arm, args.e2e_cells, args.expressed)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("generate_bench.py measures on a CUDA device; none is present")
    gpu = card()
    res = {"gpu (name, power limit, max SM clock)": gpu, "genes": G, "encoding_size": Z,
           "network": "ContinuousCellBiGan, seed 0 (untrained); *_expressed: with the output "
                      "bias of a seeded fraction of the genes raised by 2", "tile_rows": TILE,
           "copy_bandwidth_gbs": COPY_GBS}
    import gc
    res["device_pass"] = device_pass(args, 0.0)
    gc.collect()
    res["device_pass_expressed"] = device_pass(args, args.expressed)
    gc.collect()                     # the device passes' networks, before the children start
    torch.cuda.empty_cache()
    res["end_to_end"] = e2e(args)
    res["maxrss_parent_bytes"] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
