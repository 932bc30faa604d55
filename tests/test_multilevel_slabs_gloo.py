"""World-size-2 (and 3) gloo tests of the multilevel driver's host path on slabs, on CPU: the level-to-level warm
start gathers this rank's coarse l, y into the reference's global order and resamples them globally, which must give
exactly what `interpolate_y_l` gives for the global vectors; and a level with fewer z planes than ranks is refused
before anything is built."""
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, n):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sip_b200 as sip
    from sip_b200 import distributed as dd
    from sip_b200 import multilevel as ml
    dd._state.update(active=True, rank=rank, world=world)      # host logic only: no NCCL communicator on CPU
    TF = np.float64
    d = (25.0, 20.0, 10.0)
    cg = sip.compgrid(d, n)
    cons = [sip.set_definitions("bounds", "identity", 1500.0, 4500.0, ("tensor", "")),
            sip.set_definitions("bounds", "D_x", -1.0, 1.0, ("tensor", "")),
            sip.set_definitions("bounds", "D_z", 0.0, 1e6, ("tensor", "")),
            sip.set_definitions("l1", "TV", 0.0, 1e3, ("tensor", ""))]
    opt = sip.PARSDMM_options()
    opt.FL = TF
    m = np.zeros(int(np.prod(n)), dtype=TF)
    TD_OP_levels, _, _, set_Prop_levels, grids, _ = sip.setup_multi_level_PARSDMM(m, 2, 2, cg, cons, opt)
    coarse = tuple(grids[1].n)
    assert coarse[2] >= world and (coarse[2] % world or n[2] % world), "uneven slabs expected"
    rng = np.random.default_rng(11 + world)
    xg = rng.standard_normal(int(np.prod(coarse))).astype(TF)
    lg = [rng.standard_normal(A.rows).astype(TF) for A in TD_OP_levels[1]]
    yg = [rng.standard_normal(A.rows).astype(TF) for A in TD_OP_levels[1]]
    kinds = {A.kind for A in TD_OP_levels[1]}
    assert {"identity", "D_x", "D_z", "TV"} <= kinds, kinds
    slab = dd.slab_range(coarse[2])
    l_loc = [dd.scatter_td(v, A, *slab) for v, A in zip(lg, TD_OP_levels[1])]
    y_loc = [dd.scatter_td(v, A, *slab) for v, A in zip(yg, TD_OP_levels[1])]
    x, l, y = ml._host_warm_start(xg.copy(), l_loc, y_loc, TD_OP_levels[1], set_Prop_levels, grids, True, 0)
    l_ref, y_ref = sip.interpolate_y_l([v.copy() for v in lg], [v.copy() for v in yg], set_Prop_levels, grids, True, 0)
    assert np.array_equal(x, sip.resample_nn(xg, coarse, n))
    assert len(l) == len(l_ref) == len(TD_OP_levels[0])
    for j, A in enumerate(TD_OP_levels[0]):
        assert l[j].size == A.rows and np.array_equal(l[j], l_ref[j]), j
        assert y[j].size == A.rows and np.array_equal(y[j], y_ref[j]), j
    # 3 levels of a grid with 3 z planes: 3 -> 2 -> 1 planes; the first level with fewer planes than ranks is named
    bad = r"level 2 \(grid \(2, 2, 1\)\)" if world == 2 else r"level 1 \(grid \(3, 3, 2\)\)"
    with pytest.raises(ValueError, match=bad):
        sip.setup_multi_level_PARSDMM(np.zeros(6 * 6 * 3, dtype=TF), 3, 2, sip.compgrid(d, (6, 6, 3)), cons, opt)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, (7, 6, 11)), (3, (8, 6, 14))])
def test_multilevel_host_warm_start_gloo(world, n):
    port = 29640 + world
    mp.spawn(_worker, args=(world, port, n), nprocs=world, join=True)
