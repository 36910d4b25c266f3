"""The two-sample pass on one GPU at 33,694 genes: cc_log1p_features on one 4096-cell generator
tile against the copy bandwidth measured in the same run, the Gram GEMM and cc_mmd_sums at
N = 8192 (n = 4096 per side, 1,001 labellings, three bandwidths), the full device pass of one
group (features of both sides, Gram, median, sums), and an end-to-end A/B of two_sample_test
(streamed) against its numpy definition at a size the host can do.  Writes one JSON file with
the card's name and power limit read in the same run.

    python tools/twosample_bench.py --out profiles/r07_twosample.json

Network: generate_bench.network(0.06), seeded and untrained, about 2,100 non-zeros per
generated cell.  Real cells: score_bench.device_csr, about 2,100 stored genes per cell.

Kernel times are CUDA events over --reps launches after a warm-up.  The feature kernel reads
4096 x 33,694 fp32 (552 MB, beyond the 126 MB L2) and writes 4096 x 33,728 bf16; its bytes over
time is compared with a 2 GiB device-to-device copy (read + write bytes).  Gram FLOP = three
n x n x genes products (XX, XY, YY quadrants) x 2.

End to end (--e2e-cells real cells, one group, 200 permutations): each arm runs in a fresh
process, alternating, twice; wall time of two_sample_test and its peak host bytes (largest RSS
sampled every millisecond during the call minus the RSS before it).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.generate_bench import network                      # noqa: E402
from tools.score_bench import card, device_csr, events_ms      # noqa: E402

G, Z, TILE = 33694, 3, 4096
EXPRESSED = 0.06


def copy_gbs(reps=20):
    import torch
    n = 1 << 29
    src = torch.ones(n, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    ms = events_ms(lambda: dst.copy_(src), reps)
    return 2 * n * 4 / ms / 1e6


def device_numbers(args):
    import numpy as np
    import torch
    from cellcomm_b200 import ops
    from cellcomm_b200.bigan_basic import MMD_SCALES, pack_labellings, two_sample_labellings
    net = network(EXPRESSED)
    eng = net._engine
    out = {"genes": G}
    copy = copy_gbs()
    out["copy_gbs"] = copy
    rng = np.random.default_rng(1)
    z = rng.random((TILE, Z), dtype=np.float32)
    r = rng.random((TILE, Z), dtype=np.float32)
    tile = ops.alloc2d(TILE, G, dtype=torch.float32, zero=False)
    eng.set_latents(z, r, TILE)
    eng.generate(TILE, out32=tile)
    feats = ops.alloc2d(TILE, G, dtype=torch.bfloat16, zero=False)
    lib = torch.empty(TILE, dtype=torch.float64, device="cuda")
    det = torch.empty(TILE, dtype=torch.int32, device="cuda")
    nbytes = TILE * G * 4 + TILE * ops.pad_ld(G) * 2 + TILE * 12
    for rnd in (True, False):
        ms = events_ms(lambda: ops.log1p_features(tile, feats, lib, det, round=rnd), args.reps)
        key = "features_round" if rnd else "features_exact"
        out[key + "_ms_per_tile"] = ms
        out[key + "_gbs"] = nbytes / ms / 1e6
        out[key + "_of_copy"] = nbytes / ms / 1e6 / copy
    gen_ms = events_ms(lambda: eng.generate(TILE, out32=tile), 5)
    out["generator_tile_ms"] = gen_ms
    # Gram and sums at N = 8192
    n = TILE
    fx = feats
    fy = ops.alloc2d(n, G, dtype=torch.bfloat16, zero=False)
    eng.set_latents(rng.random((n, Z), dtype=np.float32), rng.random((n, Z), dtype=np.float32), n)
    eng.generate(n, out32=tile)
    ops.log1p_features(tile, fy, lib, det, round=True)
    N = 2 * n
    gram = ops.alloc2d(N, N, dtype=torch.float32, zero=False)

    def gram_fn():
        ops.gemm(n, n, [fx], [fx], [G], 0, 0, out32=gram[:n, :n])
        ops.gemm(n, n, [fx], [fy], [G], 0, 0, out32=gram[:n, n:])
        ops.gemm(n, n, [fy], [fy], [G], 0, 0, out32=gram[n:, n:])

    ms = events_ms(gram_fn, args.reps)
    out["gram_ms"] = ms
    out["gram_tflops"] = 3 * n * n * G * 2 / ms / 1e9
    masks = pack_labellings(two_sample_labellings(n, 1000, 0, 0))
    m_dev = torch.from_numpy(masks.view(np.int32)).cuda()
    sums = torch.empty((1001, 3, 3), dtype=torch.float64, device="cuda")
    ws = torch.empty(ops.mmd_sums_ws_bytes(N, 3, 1001), dtype=torch.uint8, device="cuda")
    med, _ = eng.mmd_sums(fx, fy, MMD_SCALES, masks)
    inv = [1.0 / (s * med) for s in MMD_SCALES]
    ms = events_ms(lambda: ops.mmd_sums(gram, inv, m_dev, sums, ws=ws), max(3, args.reps // 4))
    out["mmd_sums_ms"] = ms
    out["mmd_sums_over_gram"] = ms / out["gram_ms"]
    # the full device pass of one group: both sides' features, Gram, median, sums
    csr = device_csr(n)
    order = np.arange(n)
    zz, rr = rng.random((n, Z), dtype=np.float32), rng.random((n, Z), dtype=np.float32)

    def group():
        a = eng.features_stream(csr=csr, order=order)[0]
        b = eng.features_stream(z32=zz, r32=rr)[0]
        eng.mmd_sums(a, b, MMD_SCALES, masks)

    group()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(3):
        group()
    torch.cuda.synchronize()
    out["group_pass_s"] = (time.perf_counter() - t) / 3
    out["group_cells_per_side"] = n
    out["labellings"] = 1001
    return out


def e2e_arm(arm, cells):
    """one arm in this process -> (seconds, peak host bytes)"""
    import numpy as np
    from cellcomm_b200.bigan_basic import BasicBiGan
    from cellcomm_b200.cell_type_training import CellMatrix
    net = network(EXPRESSED)
    rng = np.random.default_rng(3)
    k = 60
    cols = (np.arange(k) * (G // k) + rng.integers(0, G // k, (cells, k))).astype(np.int32)
    mat = CellMatrix(np.arange(cells + 1, dtype=np.int64) * k, cols.reshape(-1),
                     rng.geometric(0.3, cells * k).astype(np.float64), np.arange(1, cells + 1),
                     np.arange(1, G + 1))
    net.two_sample_test(CellMatrix.from_dense(np.ones((4, G))), permutations=2)   # warm-up

    def rss():
        with open("/proc/self/statm") as f:
            return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")

    peak, stop = [0], threading.Event()

    def sample():
        while not stop.is_set():
            peak[0] = max(peak[0], rss())
            time.sleep(0.001)

    base = rss()
    th = threading.Thread(target=sample)
    th.start()
    t = time.perf_counter()
    if arm == "device":
        res = net.two_sample_test(mat, permutations=200)
    else:
        res = BasicBiGan.two_sample_test(net, mat, permutations=200)
    sec = time.perf_counter() - t
    stop.set()
    th.join()
    return {"seconds": sec, "peak_host_bytes": max(0, peak[0] - base),
            "mmd2": [float(v) for v in res.mmd2[0]], "p": [float(v) for v in res.p_value[0]]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_twosample.json"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--e2e-cells", type=int, default=2048)
    ap.add_argument("--arm", choices=["device", "numpy"])
    args = ap.parse_args()
    if args.arm:
        print(json.dumps(e2e_arm(args.arm, args.e2e_cells)))
        return
    res = {"card": card(), "device": device_numbers(args)}
    runs = []
    for _ in range(2):
        for arm in ("device", "numpy"):
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--arm", arm,
                                "--e2e-cells", str(args.e2e_cells)], capture_output=True,
                               text=True, check=True)
            runs.append({"arm": arm, **json.loads(p.stdout.strip().splitlines()[-1])})
    res["end_to_end"] = {"cells": args.e2e_cells, "permutations": 200, "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
