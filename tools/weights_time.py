"""Cost of per-frame weights: each case timed weighted and unweighted in the same process.

Weighted Grams run on the FP64 DMMA kernels; the unweighted call takes the default path (int8 tensor cores
where it applies) and, for comparison, the DMMA path (``_GRAM_I8`` off).  At w = 1 the weighted Gram must
equal the unweighted DMMA Gram to 1e-9 relative Frobenius.

    python tools/weights_time.py [--out FILE]

Cases (synthetic data, device-resident float32):
  * config 2: qp_linear_map on cln025, 1 M frames (whole fit: Gram + device solve) and its Gram alone;
  * config 4: linear Gram at n_red 2 600 (protein_like_topology(500)), 20 k frames;
  * config 3: featurised Grams on cln025 (id + gb, n_feat 769, 10 beads), 50 k frames.
Prints one JSON line with the card name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import aggforce_b200 as agf  # noqa: E402
from aggforce_b200 import _engine  # noqa: E402
from aggforce_b200.qp import Multifeaturize, gb_feat, id_feat, qp_linear_map  # noqa: E402
from aggforce_b200.qp.featlinearmap import _FusedContext, _fusable  # noqa: E402
from aggforce_b200.qp.qplinear import reduced_columns  # noqa: E402
from aggforce_b200.synth import chignolin_topology, protein_like_topology, synth_trajectory_device  # noqa: E402
from aggforce_b200.util import Curry  # noqa: E402


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = (s.strip() for s in out.split(","))
    except Exception as exc:  # noqa: BLE001
        name, limit = torch.cuda.get_device_name(0), f"unknown ({type(exc).__name__})"
    return {"gpu": name, "power_limit": limit}


def timeit(fn, reps: int = 5) -> float:
    """Median milliseconds of ``reps`` calls, each bracketed by CUDA events and a synchronise."""
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times))


def rel(a: torch.Tensor, b: torch.Tensor) -> float:
    return float((a - b).norm() / b.norm())


def with_i8(on: bool, fn):
    prev = _engine._GRAM_I8[0]
    _engine._GRAM_I8[0] = on
    try:
        return fn()
    finally:
        _engine._GRAM_I8[0] = prev


def gram_case(topo, n_frames: int, seed: int) -> dict:
    _, forces = synth_trajectory_device(topo, n_frames, seed=seed, want_coords=False)
    cols = reduced_columns(topo.n_sites, topo.xh_constraints)
    n_red = int(cols.max()) + 1
    fr = _engine.Frames(forces)
    ones = _engine.frame_weights_dev(torch.ones(n_frames, dtype=torch.float64, device="cuda"), n_frames)
    w = _engine.frame_weights_dev(10.0 ** torch.empty(n_frames, dtype=torch.float64, device="cuda").uniform_(-3, 3),
                                  n_frames)
    out = {"frames": n_frames, "n_red": n_red,
           "unweighted_default_ms": timeit(lambda: _engine.gram_linear(fr, cols, n_red)),
           "unweighted_dmma_ms": with_i8(False, lambda: timeit(lambda: _engine.gram_linear(fr, cols, n_red))),
           "weighted_ms": timeit(lambda: _engine.gram_linear(fr, cols, n_red, weights=w))}
    g1 = _engine.gram_linear(fr, cols, n_red, weights=ones)
    g0 = with_i8(False, lambda: _engine.gram_linear(fr, cols, n_red))
    out["rel_fro_w1_vs_unweighted_dmma"] = rel(g1, g0)
    return out


def fit_case(topo, n_frames: int) -> dict:
    coords, forces = synth_trajectory_device(topo, n_frames, seed=1)
    traj = agf.Trajectory(coords=coords, forces=forces)
    cmap = agf.LinearMap([[i] for i in topo.bead_atoms], n_fg_sites=topo.n_sites)
    w = torch.rand(n_frames, dtype=torch.float64, device="cuda") * 2.0

    def fit(**kw):
        return qp_linear_map(traj, cmap, topo.xh_constraints, l2_regularization=1e3, **kw).force_map.standard_matrix

    ones = np.ones(n_frames)
    m1 = fit(frame_weights=ones)
    m0 = with_i8(False, lambda: fit())
    return {"frames": n_frames,
            "unweighted_default_ms": timeit(fit),
            "unweighted_dmma_ms": with_i8(False, lambda: timeit(fit)),
            "weighted_ms": timeit(lambda: fit(frame_weights=w)),
            "rel_map_w1_vs_unweighted_dmma": float(np.linalg.norm(m1 - m0) / np.linalg.norm(m0))}


def feat_case(topo, n_frames: int) -> dict:
    c, f = synth_trajectory_device(topo, n_frames, seed=2)
    cmap = agf.LinearMap([[i] for i in topo.bead_atoms], n_fg_sites=topo.n_sites)
    feat = Multifeaturize([id_feat, Curry(gb_feat, inner=0, outer=8, width=1, n_basis=7)])
    ctx = _FusedContext(cmap, topo.xh_constraints, _fusable(feat))
    fc, ff = _engine.Frames(c), _engine.Frames(f)
    kbt = 0.6955215
    ones = _engine.frame_weights_dev(torch.ones(n_frames, dtype=torch.float64, device="cuda"), n_frames)
    w = _engine.frame_weights_dev(torch.rand(n_frames, dtype=torch.float64, device="cuda") * 2.0, n_frames)

    def grams(**kw):
        return ctx.grams(fc, ff, kbt, on_device=True, **kw)

    out = {"frames": n_frames, "n_feat": int(ctx.n_feat_kernel),
           "unweighted_default_ms": timeit(grams, 3),
           "unweighted_dmma_ms": with_i8(False, lambda: timeit(grams, 3)),
           "weighted_ms": timeit(lambda: grams(weights=w), 3)}
    g1 = grams(weights=ones)
    g0 = with_i8(False, grams)
    out["rel_fro_w1_vs_unweighted_dmma"] = max(rel(g1[b], g0[b]) for b in range(g0.shape[0]))
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "weights_time.py measures on a CUDA device"
    torch.cuda.set_device(0)
    cln = chignolin_topology()
    res = {"card": card()}
    res["config2_fit"] = fit_case(cln, 1_000_000)
    res["config2_gram"] = gram_case(cln, 1_000_000, seed=1)
    res["config4_gram"] = gram_case(protein_like_topology(500), 20_000, seed=3)
    res["config3_feat_gram"] = feat_case(cln, 50_000)
    ok = (res["config2_gram"]["rel_fro_w1_vs_unweighted_dmma"] < 1e-9
          and res["config4_gram"]["rel_fro_w1_vs_unweighted_dmma"] < 1e-9
          and res["config3_feat_gram"]["rel_fro_w1_vs_unweighted_dmma"] < 1e-9)
    res["w1_parity_ok"] = bool(ok)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
