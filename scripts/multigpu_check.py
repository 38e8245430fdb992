"""Multi-GPU parity check (run under torch.distributed.run, one rank per GPU):
sharded greedy IVAR (scalar noise and a heteroscedastic noise function) and greedy max-variance must pick exactly the
indices of the single-process CPU oracle."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp, kernels
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device
    from gpexp_b200.engine import GreedyVarEngine, Shard
    ed.VERBOSE = False
    shard = Shard()
    rng = np.random.default_rng(42)
    ok = True
    # --- greedy IVAR, candidates sharded -----------------------------------------------------------
    cand, mc = rng.uniform(-1, 1, (4001, 2)), rng.uniform(-1, 1, (3000, 2))
    kern = kernels.KernelSquaredExponential([0.2, 0.3], 1.0, 2)
    cf = ed.costFunctionGP_IVAR(gp.GP(kern, 1e-6), 1, Space(2, None, None), mcPoints=mc)
    idx = ed.performGreedyIVARExperimentalDesign(cf, cand, 12, returnIndices=True, shard=shard)

    # --- the same with a noise function: each rank evaluates it on its own block, nu(p) travels in the pivot record -----
    def nu(p):
        return 1e-4 + 1e-3 * p[:, 0] ** 2
    cfh = ed.costFunctionGP_IVAR(gp.GP(kern, 1e-6), 1, Space(2, None, None, noise=nu), mcPoints=mc)
    hidx = ed.performGreedyIVARExperimentalDesign(cfh, cand, 12, returnIndices=True, shard=shard)
    # --- greedy max variance, pool sharded ----------------------------------------------------------
    pool = rng.uniform(-1, 1, (10007, 5))
    mk = kernels.KernelIsoMatern(1.0, 1.0, 5)
    dev = mk._bind()
    vpts = ed.performGreedyVarExperimentalDesign(mk, pool, 25, 5, shard=shard)   # public API, pool sharded inside
    vidx = [int(np.where(np.all(pool == p, axis=1))[0][0]) for p in vpts]
    # --- greedy mutual information, |V| x |V| matrices sharded by column blocks ------------------------
    from gpexp_b200.engine import ShardedMIEngine
    vpool = rng.standard_normal((1500, 3))
    hk = kernels.KernelMehlerND([0.9, 0.9, 0.9], 3)
    hk._bind(dev)
    meng = ShardedMIEngine(dev, vpool, 14, 1e-2, shard=shard)
    midx = meng.run(14, start=0)
    minfo = int(meng.info.item())
    torch.cuda.synchronize()
    if rank == 0:
        from oracle import gpexp_oracle as orc
        mref, _ = orc.fast_greedy_mi(orc.KernelSpec.mehler([0.9, 0.9, 0.9], 3), vpool, 1e-2, 14, start=0)
        mi_ok = [int(i) for i in midx] == mref and minfo == 0
        print("multigpu_check world=%d mi=%s -> %s" % (world, [int(i) for i in midx][:8], "OK" if mi_ok else "MISMATCH"), flush=True)
        if not mi_ok:
            print("ref mi", mref, "got", [int(i) for i in midx], "info", minfo)
        ref, _ = orc.fast_greedy_ivar(orc.KernelSpec.se([0.2, 0.3], 1.0, 2), cand, mc, 12, 1e-6)
        vref, _ = orc.fast_greedy_var(orc.KernelSpec.matern32(1.0, 1.0, 5), pool, 25)
        from tests.hetero_oracle import fast_greedy_ivar_nu
        href, _ = fast_greedy_ivar_nu(orc.KernelSpec.se([0.2, 0.3], 1.0, 2), cand, mc, 12, nu(cand))
        h_ok = [int(i) for i in hidx] == href
        print("multigpu_check world=%d hetero ivar=%s -> %s" % (world, [int(i) for i in hidx][:6], "OK" if h_ok else "MISMATCH"),
              flush=True)
        if not h_ok:
            print("ref hetero ivar", href, "got", [int(i) for i in hidx])
        ok = [int(i) for i in idx] == ref and [int(i) for i in vidx] == vref and mi_ok and h_ok
        print("multigpu_check world=%d ivar=%s var=%s -> %s" % (world, [int(i) for i in idx][:6], [int(i) for i in vidx][:6],
                                                                 "OK" if ok else "MISMATCH"), flush=True)
        if not ok:
            print("ref ivar", ref, "got", [int(i) for i in idx]); print("ref var", vref, "got", [int(i) for i in vidx])
    # every rank must hold the same picks
    t = torch.tensor([int(i) for i in idx] + [int(i) for i in hidx] + [int(i) for i in vidx] + [int(i) for i in midx],
                     device="cuda")
    g = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(g, t)
    same = all(bool((x == t).all()) for x in g)
    if rank == 0:
        print("all ranks agree:", same, flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if (ok and same) else 1)


if __name__ == "__main__":
    main()
