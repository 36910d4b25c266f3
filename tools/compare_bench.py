"""The compare pass on one GPU: BiGanEngine.moments_stream over real cells (a synthetic
10x-shaped matrix) and over generated cells, the cost of cc_col_moments on one 4096-cell
generator tile, and an end-to-end A/B of compare_cells (streamed) against its composed numpy
definition, at 33,694 genes on a seeded ContinuousCellBiGan (Z = 3).  Writes one JSON file with
the card's name and power limit read in the same run.

    python tools/compare_bench.py --out profiles/r06_compare_stream.json

Network: seeded and untrained, with the output bias of 6 % of the genes raised by 2
(generate_bench.network), so a generated cell holds about 2,100 non-zeros, like a real one.

Device pass (--cells, default 2^18, three groups of random labels): real cells from a CSR with
about 2,100 stored genes per cell (score_bench.device_csr), grouped by a stable argsort of the
labels; generated cells from seeded priors.  Host clock around each synchronised pass.

Kernel (one 4096-cell tile of generator output, 552 MB of fp32: far beyond the 126 MB L2):
CUDA events over --reps launches of cc_col_moments with and without rounding, and of the
generator forward.  Bytes = rows * cols * 4 + the workspace partials written and read
(2 * slabs * cols * 24), reported as TB/s and against the device-to-device copy bandwidth
measured in this run (a 2 GiB copy, read + write bytes).

End to end (--e2e-cells, default 32,768): each arm runs in a fresh process, alternating; wall
time of compare_cells and its peak host bytes = the largest RSS sampled every millisecond during
the call minus the RSS just before it.
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

from tools.generate_bench import network                      # noqa: E402
from tools.score_bench import card, device_csr, events_ms      # noqa: E402

G, Z, TILE, K = 33694, 3, 4096, 3
EXPRESSED = 0.06


def copy_gbs(reps=20):
    """device-to-device copy bandwidth: (read + write bytes) / time of a 2 GiB copy"""
    import torch
    n = 1 << 29
    src = torch.ones(n, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    ms = events_ms(lambda: dst.copy_(src), reps)
    return 2 * n * 4 / ms / 1e6


def groups(n, seed=0):
    """K random labels -> (bounds, stable argsort order)"""
    import numpy as np
    labels = np.random.default_rng(seed).integers(0, K, n)
    counts = np.bincount(labels, minlength=K)
    return (np.concatenate([[0], np.cumsum(counts)]),
            np.argsort(labels, kind="stable").astype(np.int64))


def device_pass(args):
    import numpy as np
    import torch
    from cellcomm_b200 import ops
    net = network(EXPRESSED)
    eng = net._engine
    n = args.cells
    bounds, order = groups(n)
    csr = device_csr(n)
    rng = np.random.default_rng(1)
    z = rng.random((n, Z), dtype=np.float32)
    r = rng.random((n, Z), dtype=np.float32)
    warm = [0, TILE, 2 * TILE]
    eng.moments_stream(warm, csr=csr, order=order[:2 * TILE])               # warm-up
    eng.moments_stream(warm, z32=z[:2 * TILE], r32=r[:2 * TILE])
    torch.cuda.synchronize()
    out = {"cells": n, "groups": K, "nnz_per_real_cell": int(csr[0][-1]) / n}
    for side, kw in (("real", {"csr": csr, "order": order}), ("generated", {"z32": z, "r32": r})):
        t0 = time.perf_counter()
        s1, _, nz = eng.moments_stream(bounds, **kw)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        out[side] = {"wall_s": wall, "cells_per_s": n / wall,
                     "mean_library_size": float(s1.sum() / n),
                     "mean_genes_detected": float(nz.sum() / n)}

    # one generator tile, each stage on its own
    eng.set_latents(z[:TILE], r[:TILE], TILE)
    tile = ops.alloc2d(TILE, G, dtype=torch.float32, device="cuda", zero=False)
    acc = (torch.zeros(G, dtype=torch.float64, device="cuda"),
           torch.zeros(G, dtype=torch.float64, device="cuda"),
           torch.zeros(G, dtype=torch.int64, device="cuda"))
    ws_bytes = ops.col_moments_ws_bytes(TILE, G)
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    gen_ms = events_ms(lambda: eng.generate(TILE, out32=tile), args.reps)
    rnd_ms = events_ms(lambda: ops.col_moments(tile, *acc, round=True, ws=ws), args.reps)
    raw_ms = events_ms(lambda: ops.col_moments(tile, *acc, round=False, ws=ws), args.reps)
    slabs = (TILE + 255) // 256
    kbytes = TILE * G * 4 + 2 * slabs * G * 24
    copy = copy_gbs()
    out["tile_4096"] = {
        "generator_ms": gen_ms,
        "col_moments_round_ms": rnd_ms,
        "col_moments_ms": raw_ms,
        "col_moments_bytes": kbytes,
        "workspace_bytes": ws_bytes,
        "col_moments_round_tbs": kbytes / rnd_ms / 1e9,
        "col_moments_tbs": kbytes / raw_ms / 1e9,
        "copy_bandwidth_gbs": copy,
        "copy_bandwidth_source": "measured in this run: 2 GiB device-to-device copy",
        "col_moments_round_fraction_of_copy_bw": kbytes / rnd_ms / 1e6 / copy,
        "col_moments_fraction_of_copy_bw": kbytes / raw_ms / 1e6 / copy,
        "col_moments_round_fraction_of_generated_tile": rnd_ms / (gen_ms + rnd_ms),
        "col_moments_round_vs_generator_forward": rnd_ms / gen_ms,
    }
    return out


def _rss():
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


def composed(net, mat):
    """compare_cells from the definitions: dense numpy statistics of the real cells and of
    generate_cells' dense output (same groups, same draws as compare_cells)"""
    import numpy as np
    from cellcomm_b200.bigan_basic import BasicBiGan, CellComparison
    labels, k = net._comparison_groups(mat)
    real = BasicBiGan.gene_statistics(net, mat, labels, k)
    enc = net._comparison_encodings(real.cells)
    noise = net.random_uniform_vector(len(enc))
    cells = net.generate_cells(enc, noise)
    gen = BasicBiGan.gene_statistics(net, cells, np.repeat(np.arange(k), real.cells), k)
    return CellComparison(real, gen)


def arm(name, cells):
    """one end-to-end call in this process -> JSON on stdout"""
    import numpy as np
    import torch
    import bench
    net = network(EXPRESSED)
    mat = bench.make_matrix(cells, G, 5, "cuda")
    compare = net.compare_cells if name == "streamed" else (lambda m: composed(net, m))
    state = net._prior_rng.bit_generator.state
    compare(bench.make_matrix(TILE, G, 6, "cuda"))          # warm-up (both arms alike)
    net._prior_rng.bit_generator.state = state
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
    out = compare(mat)
    wall = time.perf_counter() - t0
    done.set()
    th.join()
    peak[0] = max(peak[0], _rss())
    digest = float(np.nansum(out.real.mean) + np.nansum(out.generated.mean) +
                   np.nansum(out.generated.var) + np.nansum(out.generated.detected))
    print(json.dumps({"arm": name, "wall_s": wall, "peak_host_bytes": peak[0] - before,
                      "digest": digest}))


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
                                      for a in ("streamed", "composed")},
           "digests_equal": len({x["digest"] for x in rows if "digest" in x}) == 1}
    if res["median_wall_s"]["streamed"] and res["median_wall_s"]["composed"]:
        res["speedup_streamed_over_composed"] = (res["median_wall_s"]["composed"] /
                                                 res["median_wall_s"]["streamed"])
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--cells", type=int, default=1 << 18)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--e2e-cells", type=int, default=32768)
    ap.add_argument("--e2e-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_compare_stream.json"))
    ap.add_argument("--arm", choices=("streamed", "composed"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.arm:
        arm(args.arm, args.e2e_cells)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("compare_bench.py measures on a CUDA device; none is present")
    res = {"gpu (name, power limit, max SM clock)": card(), "genes": G, "encoding_size": Z,
           "network": f"ContinuousCellBiGan, seed 0 (untrained), output bias of {EXPRESSED:.0%} "
                      "of the genes raised by 2", "tile_rows": TILE}
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
