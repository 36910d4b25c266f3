"""The score pass on one GPU: BiGanEngine.score_stream over a synthetic 10x-shaped matrix, the
cost of each stage of one 4096-cell tile, and an end-to-end A/B of score_cells (streamed)
against its composed definition (BasicBiGan.score_cells: dense G.predict output on the host,
the error in numpy), at 33,694 genes on a seeded ContinuousCellBiGan (Z = 3).  Writes one JSON
file with the card's name and power limit read in the same run.

    python tools/score_bench.py --out profiles/r05_score_stream.json

Device pass (--cells, default 2^18): a CSR with about 2,000 stored genes per cell
(bench.synth_csr: 16,384 distinct cells, repeated on the device to --cells rows, so the CSR
alone is ~4 GB and every tile's 552 MB fp32 generator output is far beyond the 126 MB L2);
host clock around a synchronised pass; cells/s and graph FLOP/s at 1.842 GFLOP per cell
(E 0.352 + G 0.501 + D 0.989, SURVEY.md 8a).  Per 4096-cell tile, CUDA events over repeated
launches: the encoder (cc_encode_stream: gather + E forward), the generator forward, the
discriminator (cc_gather_rows + D forward) and cc_recon_sqerr, whose bytes
rows*cols*4 + nnz*8 + rows*12 are reported as TB/s and as a fraction of bench.peaks()'s HBM
copy bandwidth.

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
GFLOP_PER_CELL = {"E": 0.352, "G": 0.501, "D": 0.989}    # SURVEY.md 8a


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def network(seed=0):
    from cellcomm_b200.bigan_cont import ContinuousCellBiGan
    return ContinuousCellBiGan(Z, G, seed=seed)


def device_csr(cells, distinct=16384, seed=0):
    """(rowptr, colidx, values) on the device: `distinct` synthetic cells repeated to `cells`"""
    import numpy as np
    import torch
    import bench
    rowptr, colidx, values = bench.synth_csr(distinct, G, seed, "cuda")
    reps = (cells + distinct - 1) // distinct
    nnz = int(rowptr[-1])
    rp = torch.from_numpy(rowptr).cuda()
    rp_all = torch.cat([rp[:-1] + k * nnz for k in range(reps)] + [rp[-1:] + (reps - 1) * nnz])
    ci = torch.from_numpy(colidx).cuda().repeat(reps)
    va = torch.from_numpy(values.astype(np.float32)).cuda().repeat(reps)
    end = int(rp_all[cells])
    return rp_all[:cells + 1].contiguous(), ci[:end].contiguous(), va[:end].contiguous()


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


def device_pass(args):
    import numpy as np
    import torch
    import bench
    from cellcomm_b200 import ops
    net = network()
    eng = net._engine
    rowptr, colidx, values = device_csr(args.cells)
    n = args.cells
    nnz = int(rowptr[-1])
    r = np.random.default_rng(1).random((n, Z), dtype=np.float32)
    enc = torch.empty((n, Z), dtype=torch.float32, device="cuda")
    mse = torch.empty(n, dtype=torch.float32, device="cuda")
    d = torch.empty(n, dtype=torch.float32, device="cuda")
    eng.score_stream(rowptr, colidx, values, 0, 2 * TILE, r[:2 * TILE], enc[:2 * TILE],
                     mse[:2 * TILE], d[:2 * TILE])                       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.score_stream(rowptr, colidx, values, 0, n, r, enc, mse, d)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    flops = sum(GFLOP_PER_CELL.values()) * 1e9 * n

    # one tile in the middle of the matrix, each stage on its own
    s = (n // 2) // TILE * TILE
    z = enc[s:s + TILE]
    pred = ops.alloc2d(TILE, G, dtype=torch.float32, device="cuda", zero=False)
    cells = ops.alloc2d(TILE, G, device="cuda")
    eng.set_latents(z, r[s:s + TILE], TILE)
    stages = {
        "encoder_ms": lambda: eng.encode_stream(rowptr, colidx, values, s, s + TILE, z),
        "generator_ms": lambda: eng.generate(TILE, out32=pred),
        "recon_sqerr_ms": lambda: ops.recon_sqerr(pred, rowptr, colidx, values, s,
                                                  mse[s:s + TILE], scale=1.0 / G),
        "discriminator_ms": lambda: (ops.gather_rows(rowptr, colidx, values, G, row_start=s,
                                                     n_rows=TILE, out16=cells),
                                     eng.discriminate(z, cells, d[s:s + TILE].view(TILE, 1))),
    }
    tile = {k: events_ms(fn, args.reps) for k, fn in stages.items()}
    tile_nnz = int(rowptr[s + TILE] - rowptr[s])
    kbytes = TILE * G * 4 + tile_nnz * 8 + TILE * 12
    pk = bench.peaks()
    k_gbs = kbytes / tile["recon_sqerr_ms"] / 1e6
    stage_sum = sum(tile.values())
    tile.update({
        "nnz": tile_nnz,
        "recon_sqerr_bytes": kbytes,
        "recon_sqerr_tbs": k_gbs / 1e3,
        "copy_bandwidth_gbs": pk["hbm_gbs"],
        "peaks_source": pk["source"],
        "recon_sqerr_fraction_of_copy_bw": k_gbs / pk["hbm_gbs"],
        "recon_sqerr_fraction_of_tile": tile["recon_sqerr_ms"] / stage_sum,
        "stages_sum_ms": stage_sum,
    })
    return {"cells": n, "nnz_per_cell": nnz / n, "wall_s": wall, "cells_per_s": n / wall,
            "graph_gflop_per_cell": sum(GFLOP_PER_CELL.values()),
            "graph_tflops": flops / wall / 1e12,
            "mse_mean": float(mse.double().mean()), "d_real_mean": float(d.double().mean()),
            "tile_4096": tile}


def _rss():
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


def arm(name, cells):
    """one end-to-end call in this process -> JSON on stdout"""
    import numpy as np
    import torch
    import bench
    from cellcomm_b200.bigan_basic import BasicBiGan
    net = network()
    mat = bench.make_matrix(cells, G, 5, "cuda")
    r = np.random.default_rng(3).random((cells, Z), dtype=np.float32)
    score = net.score_cells if name == "streamed" else \
        (lambda m, x: BasicBiGan.score_cells(net, m, x))
    warm = bench.make_matrix(TILE, G, 6, "cuda")
    score(warm, r[:TILE])                                    # warm-up (both arms alike)
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
    out = score(mat, r)
    wall = time.perf_counter() - t0
    done.set()
    th.join()
    peak[0] = max(peak[0], _rss())
    print(json.dumps({"arm": name, "wall_s": wall, "peak_host_bytes": peak[0] - before,
                      "mse_mean": float(np.mean(out.mse, dtype=np.float64))}))


def e2e(args):
    rows = []
    for rep in range(args.e2e_reps):
        for name in ("streamed", "composed") if rep % 2 == 0 else ("composed", "streamed"):
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--arm", name,
                                "--e2e-cells", str(args.e2e_cells)], capture_output=True,
                               text=True, cwd=ROOT, timeout=1800)
            if p.returncode != 0:
                rows.append({"arm": name, "failed": p.stderr[-2000:]})
                continue
            rows.append(json.loads(p.stdout.strip().splitlines()[-1]))

    def med(name, key):
        v = sorted(x[key] for x in rows if x["arm"] == name and key in x)
        return v[len(v) // 2] if v else None

    res = {"cells": args.e2e_cells, "runs": rows,
           "median_wall_s": {a: med(a, "wall_s") for a in ("streamed", "composed")},
           "median_peak_host_bytes": {a: med(a, "peak_host_bytes")
                                      for a in ("streamed", "composed")}}
    if res["median_wall_s"]["streamed"] and res["median_wall_s"]["composed"]:
        res["speedup_streamed_over_composed"] = (res["median_wall_s"]["composed"] /
                                                 res["median_wall_s"]["streamed"])
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--cells", type=int, default=1 << 18)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--e2e-cells", type=int, default=32768)
    ap.add_argument("--e2e-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_score_stream.json"))
    ap.add_argument("--arm", choices=("streamed", "composed"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.arm:
        arm(args.arm, args.e2e_cells)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("score_bench.py measures on a CUDA device; none is present")
    res = {"gpu (name, power limit, max SM clock)": card(), "genes": G, "encoding_size": Z,
           "network": "ContinuousCellBiGan, seed 0 (untrained)", "tile_rows": TILE}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    import gc
    res["device_pass"] = device_pass(args)
    gc.collect()
    torch.cuda.empty_cache()
    with open(args.out, "w") as f:               # the device numbers survive a failed A/B
        json.dump(res, f, indent=1)
    res["end_to_end"] = e2e(args)
    res["maxrss_parent_bytes"] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
