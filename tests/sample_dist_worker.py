"""Worker of tests/test_gpu_sample.py::test_sample_one_process_per_gpu, launched by torchrun with one rank per GPU:
qipb200_state_sample on a sharded state (collective) against the serial scan of the gathered state on rank 0.
K = 100 000 draws: the cross-rank sum of the drawn indices runs in several reduction-slot batches."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    from oracle import qip_oracle as qo
    from rustqip_b200 import circuits
    from rustqip_b200.dist import gather_state, init_sharded_state
    from rustqip_b200.state import Context

    local_rank = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local_rank)
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    g = (world - 1).bit_length()
    ctx = Context(local_rank)
    failures = 0
    K = 100000
    for n, dtype in [(18, np.complex128), (17, np.complex64)]:
        draws = np.concatenate([[0.0, 1.0 - 2.0 ** -53, 1.0, 0.5], np.random.default_rng(n).random(K)])
        st = init_sharded_state(n, dtype, ctx)
        st.set_basis(5)
        st.apply_schedule(circuits.sharded_parity_circuit(n, g))
        got = st.sample(list(range(n))[::-1], draws)    # before any download: the layout is still permuted
        few = [st.soft_measure([0, 2, n - 1], float(r)) for r in draws[:8]]
        psi = gather_state(st)
        gathered = [None] * world
        dist.all_gather_object(gathered, (got.tobytes(), few))
        st.free()
        if rank == 0:
            psi = psi.astype(np.complex128)
            cdf = np.cumsum(np.abs(psi) ** 2)
            i = np.searchsorted(cdf, draws, side="left")
            want = np.where(i < len(cdf), i, 0).astype(np.uint64)
            near = np.array([np.min(np.abs(cdf[max(k - 1, 0):k + 1] - r)) <= 1e-10 for k, r in zip(np.minimum(i, len(cdf) - 1), draws)])
            checks = {
                "ranks_agree": all(x == gathered[0] for x in gathered),
                "per_draw": bool(np.all((got == want) | near)),
                "few_excluded": int(near.sum()) <= 8,
                "soft_measure": few == [qo.soft_measure(n, [0, 2, n - 1], psi, float(r)) for r in draws[:8]],
            }
            ok = all(checks.values())
            print("sample n=%d %s world=%d: %d draws, %d at a boundary -> %s %s" % (
                n, np.dtype(dtype).name, world, len(draws), int(near.sum()), "OK" if ok else "FAIL",
                "" if ok else [k for k, v in checks.items() if not v]), flush=True)
            failures += 0 if ok else 1
    flag = [failures]
    dist.broadcast_object_list(flag, src=0)
    ctx.close()
    dist.destroy_process_group()
    sys.exit(1 if flag[0] else 0)


if __name__ == "__main__":
    main()
