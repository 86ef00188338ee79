"""Multi-GPU check of per-frame weights under frame sharding (run under torchrun, one rank per GPU, NCCL):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29513 tests/dist_weights_check.py

Every rank owns a ragged slice of the same trajectory and passes the weights of its own frames; the fitted
map and the weighted residual must equal the single-GPU weighted fit on all frames.  Weights that vanish on
one rank's whole slice still fit, and weights that vanish everywhere raise ValueError on every rank (the
check passes one exchange, so no rank is left waiting in a collective).
"""
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import aggforce_b200 as agf  # noqa: E402
from aggforce_b200.synth import chignolin_topology, synth_trajectory_device  # noqa: E402


def main() -> None:
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    topo = chignolin_topology()
    T = 20_000
    cmap = agf.LinearMap([[i] for i in topo.bead_atoms], n_fg_sites=topo.n_sites)
    bounds = np.linspace(0, T, world + 1).astype(int)
    bounds[1:-1] += 3  # ragged, unaligned shards
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    ac, af = synth_trajectory_device(topo, T, seed=99, frame0=0)
    rng = np.random.default_rng(7)
    w_all = 10.0 ** rng.uniform(-2, 2, size=T)
    kw = dict(coord_map=cmap, constrained_inds=topo.xh_constraints, l2_regularization=1e3)
    ok = True
    rels = []
    for case in ("ragged", "zero slice"):
        w = w_all.copy()
        if case == "zero slice":
            w[bounds[1]:bounds[2]] = 0.0  # rank 1 contributes nothing
        with agf.frame_sharding():
            res = agf.project_forces(coords=ac[lo:hi], forces=af[lo:hi], frame_weights=w[lo:hi], **kw)
        ref = agf.project_forces(coords=ac, forces=af, frame_weights=w, **kw)
        m, mr = res["tmap"].force_map.standard_matrix, ref["tmap"].force_map.standard_matrix
        rel_w = np.linalg.norm(m - mr) / np.linalg.norm(mr)
        rel_r = abs(res["residual"] / ref["residual"] - 1)
        rels.append((rel_w, rel_r))
        ok = ok and rel_w < 1e-9 and rel_r < 1e-9
    raised = 0
    try:
        with agf.frame_sharding():
            agf.project_forces(coords=ac[lo:hi], forces=af[lo:hi], frame_weights=np.zeros(hi - lo), **kw)
    except ValueError as exc:
        raised = int("frame_weights" in str(exc))
    ok = ok and raised == 1
    flag = torch.tensor([int(ok)], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"dist_weights_check world={world}: ragged rel_w={rels[0][0]:.2e} rel_res={rels[0][1]:.2e}; "
              f"zero slice rel_w={rels[1][0]:.2e} rel_res={rels[1][1]:.2e}; all-zero raised on every rank "
              f"-> {'OK' if flag.item() else 'FAILED'}")
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
