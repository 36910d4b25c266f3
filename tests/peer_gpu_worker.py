"""Worker of tests/test_peer_exact_gpu.py::test_real_fabric (one process per GPU under
torchrun).  Not collected by pytest.

    torchrun --nproc-per-node N tests/peer_gpu_worker.py

Buffers come from engine.TorchDist.symmetric_zeros.  Every rank builds all ranks' gradients
from one seed, so each computes the full reference locally.  It runs the protocol replay of
test_peer_exact_gpu (Replay) with real peer pointers, once with P2P stores and once with the
NVLS multicast address when the fabric has one, then three peer_allreduce calls in the
engine's epoch-counter form.  Each rank asserts bit identity with its local reference, and
the bf16 copies and all-reduce results must agree across ranks.  Rank 0 prints
`peer_check ok: {...}` naming the store paths that ran, or `peer_check skip: <reason>`.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


class Unavailable(Exception):
    pass


def main():
    from cellcomm_b200 import engine as eng, ops
    import peer_ref as P
    import test_peer_exact_gpu as T
    from dp_gpu_worker import _init, _same_on_all_ranks
    rank, world = _init()
    td = eng.TorchDist()
    keep, mc_of = [], {}

    def alloc(n, dtype):
        got = td.symmetric_zeros(n + 2 * T.PAD, dtype, "cuda")
        if got is None:
            raise Unavailable("symmetric memory unavailable")
        t, ptrs, h = got
        keep.append(h)
        esz = t.element_size()
        try:
            mc = int(h.multicast_ptr or 0)
        except Exception:
            mc = 0
        f = T.Flat(n, dtype, raw=t)
        mc_of[f.ptr] = mc + T.PAD * esz if mc else 0
        return {rank: f}, [p + T.PAD * esz for p in ptrs]

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()

    res = {"world": world}
    try:
        for path in ("p2p", "multicast"):
            rp = T.Replay(ops, world, [rank], alloc, 2 ** 32 - 2, seed=[world, 7], barrier=barrier)
            if path == "multicast":
                rp.mc = (mc_of[rp.p16[rank].ptr], mc_of[rp.p16lo[rank].ptr])
                if not rp.mc[0]:
                    res[path] = "no multicast address"
                    break
            for u in range(3):
                rp.update(u)
                # as bytes: NCCL has no int16, and a bf16 view would compare the NaN padding
                # as unequal
                _same_on_all_ranks(rp.p16[rank].raw.view(torch.uint8), f"{path} update {u} p16")
                _same_on_all_ranks(rp.p16lo[rank].raw.view(torch.uint8),
                                   f"{path} update {u} p16lo")
            res[path] = "3 updates bit-exact"
        # three all-reduces: epoch = 1 + *ctr, as TorchDist.all_reduce calls it
        n, cap = 13476, T.AR_CAP
        slots, s_p = alloc(2 * world * cap, T.F32)
        flags, f_p = alloc(world, T.I32)
        flags[rank].t.zero_()
        ctr = torch.zeros(1, dtype=torch.int32, device="cuda")
        rng = np.random.default_rng([world, 11])
        barrier()
        for call in range(3):
            D, _ = P.order_terms(rng, world, n)
            data = T._dev(D[rank]).clone()
            ops.peer_allreduce(data, world, rank, s_p, f_p, cap, 1, epoch_ctr=ctr)
            torch.cuda.synchronize()
            want = T._dev(P.rank_order_sum(D))
            assert torch.equal(data.view(torch.int32), want.view(torch.int32)), f"all-reduce {call}"
            assert T.ctr_value(ctr) == call + 1
            _same_on_all_ranks(data, f"all-reduce {call}")
        res["allreduce"] = "3 calls bit-exact"
    except Unavailable as exc:
        if rank == 0:
            print(f"peer_check skip: {exc}", flush=True)
        res = None
    barrier()
    if res is not None and rank == 0:
        print("peer_check ok:", json.dumps(res), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
