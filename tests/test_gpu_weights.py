"""Per-frame weights (``frame_weights``): weighted Grams of the FP64 DMMA kernels against the float64
oracle on sqrt(w)-scaled arrays, the repetition identity (integer weights == repeated frames) end to end,
the weighted residual and the validation of the weights.  Tolerances as in test_gpu_parity.py: Grams
<= 1e-9 relative Frobenius, maps <= 1e-6."""
import functools

import numpy as np
import pytest
import torch

import oracle
from conftest import pairs_to_set, rel_fro

pytestmark = pytest.mark.gpu

GRAM_TOL = 1e-9
MAP_TOL = 1e-6
KBT = 0.6955215
GB = dict(outer=8.0, inner=0.0, n_basis=7, width=1.0)


@pytest.fixture(scope="module")
def topo():
    from aggforce_b200.synth import chignolin_topology

    return chignolin_topology()


@pytest.fixture(scope="module")
def wide():
    from aggforce_b200.synth import protein_like_topology

    return protein_like_topology(30)  # 300 sites, 156 reduced columns: the n_red > 128 kernels


def _cmap(topo):
    from aggforce_b200 import LinearMap

    return LinearMap([[i] for i in topo.bead_atoms], n_fg_sites=topo.n_sites)


def _weights(n, seed):
    """Weights spanning six orders of magnitude, with zeros."""
    rng = np.random.default_rng(seed)
    w = 10.0 ** rng.uniform(-3, 3, size=n)
    w[rng.choice(n, size=max(1, n // 10), replace=False)] = 0.0
    return w


def _no_workspace(monkeypatch):
    """A zero-byte workspace: the ws entry points fall back to their fused / gather kernels."""
    from aggforce_b200 import _engine

    monkeypatch.setattr(_engine, "workspace", lambda nbytes: torch.empty(0, dtype=torch.uint8, device="cuda"))


# ------------------------------------------------------------------ linear Gram
@pytest.mark.parametrize("system", ["cln", "wide", "wide_gather"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("where", ["host", "device"])
def test_weighted_gram_linear(topo, wide, system, dtype, where, monkeypatch):
    from aggforce_b200 import _engine
    from aggforce_b200.qp.qplinear import reduced_columns
    from aggforce_b200.synth import synth_trajectory_host

    t = topo if system == "cln" else wide
    if system == "wide_gather":
        _no_workspace(monkeypatch)
    _, forces = synth_trajectory_host(t, 203, seed=31)
    forces = forces.astype(dtype)
    w = _weights(len(forces), 5)
    cols = reduced_columns(t.n_sites, t.xh_constraints)
    n_red = int(cols.max()) + 1
    assert (n_red <= 128) == (system == "cln")
    src = forces if where == "host" else torch.as_tensor(forces, device="cuda")[1:]
    ref_f = forces if where == "host" else forces[1:]
    ww = w if where == "host" else w[1:]
    wd = _engine.frame_weights_dev(ww, len(ref_f))
    got = _engine.to_host(_engine.gram_linear(_engine.Frames(src), cols, n_red, weights=wd))
    ref = oracle.gram_linear(ref_f.astype(np.float64) * np.sqrt(ww)[:, None, None], t.xh_constraints)
    assert np.array_equal(got, got.T)
    assert rel_fro(got, ref) < GRAM_TOL


@pytest.mark.parametrize("system", ["cln", "wide"])
def test_weighted_gram_linear_host_pieces(topo, wide, system, monkeypatch):
    """A host array cut into several upload pieces: every piece reads its own slice of the weights."""
    from aggforce_b200 import _engine
    from aggforce_b200.qp.qplinear import reduced_columns
    from aggforce_b200.synth import synth_trajectory_host

    t = topo if system == "cln" else wide
    _, forces = synth_trajectory_host(t, 150, seed=8)
    monkeypatch.setattr(_engine, "_PIECE_BYTES", 36 * t.n_sites * 3 * 4)  # 36 frames per piece
    frames = _engine.Frames(forces)
    assert frames.piece_frames() == 36
    w = _weights(len(forces), 9)
    cols = reduced_columns(t.n_sites, t.xh_constraints)
    n_red = int(cols.max()) + 1
    got = _engine.to_host(_engine.gram_linear(frames, cols, n_red, weights=_engine.frame_weights_dev(w, 150)))
    ref = oracle.gram_linear(forces.astype(np.float64) * np.sqrt(w)[:, None, None], t.xh_constraints)
    assert rel_fro(got, ref) < GRAM_TOL


# ------------------------------------------------------------------ featurised Gram
@pytest.mark.parametrize("drop", [True, False])
@pytest.mark.parametrize("kernel", ["packed", "fused"])
def test_weighted_feat_grams(topo, drop, kernel, monkeypatch):
    from aggforce_b200 import _engine
    from aggforce_b200.qp import Multifeaturize, gb_feat, id_feat
    from aggforce_b200.qp.featlinearmap import _FusedContext, _fusable
    from aggforce_b200.synth import synth_trajectory_host

    if kernel == "fused":
        _no_workspace(monkeypatch)
    coords, forces = synth_trajectory_host(topo, 37, seed=71)
    w = _weights(len(forces), 3)
    cmap, cons = _cmap(topo), topo.xh_constraints
    feat = Multifeaturize([id_feat, functools.partial(gb_feat, drop_last_channel=drop, **GB)])
    ctx = _FusedContext(cmap, cons, _fusable(feat))
    grams = ctx.grams(_engine.Frames(coords), _engine.Frames(forces), KBT,
                      weights=_engine.frame_weights_dev(w, len(w)))
    for bead in (0, 5, 9):
        idf, idd = oracle.id_features(len(coords), ctx.labels)
        gf, gd = oracle.gb_features(coords, cmap.standard_matrix, cons, ctx.labels, bead, drop_last_channel=drop, **GB)
        rows = oracle.feat_regressor_rows(forces, np.concatenate([idf, gf], axis=2), np.concatenate([idd, gd], axis=1),
                                          KBT)
        rows = rows.reshape(len(w), 3, -1) * np.sqrt(w)[:, None, None]
        rows = rows.reshape(-1, rows.shape[2])
        assert rel_fro(grams[bead], rows.T @ rows) < GRAM_TOL


# ------------------------------------------------------------------ repetition identity
def _repeat_case(topo, n_frames, seed):
    from aggforce_b200.synth import synth_trajectory_host

    coords, forces = synth_trajectory_host(topo, n_frames, seed=seed)
    counts = np.random.default_rng(seed).integers(0, 4, size=n_frames)
    return coords, forces, counts, np.repeat(coords, counts, axis=0), np.repeat(forces, counts, axis=0)


def test_integer_weights_equal_repeated_frames_linear(topo):
    from aggforce_b200 import project_forces

    coords, forces, n, rc, rf = _repeat_case(topo, 300, 12)
    cmap, cons = _cmap(topo), topo.xh_constraints
    got = project_forces(coords=coords, forces=forces, coord_map=cmap, constrained_inds=cons,
                         l2_regularization=1e3, frame_weights=n)
    ref = project_forces(coords=rc, forces=rf, coord_map=cmap, constrained_inds=cons, l2_regularization=1e3)
    w, wr = got["tmap"].force_map.standard_matrix, ref["tmap"].force_map.standard_matrix
    assert rel_fro(w, wr) < MAP_TOL
    assert abs(got["residual"] / ref["residual"] - 1) < 1e-9
    assert got["mapped_forces"].shape == forces.shape[:1] + (10, 3)  # per-frame outputs, not repeated
    assert rel_fro(got["mapped_coords"], oracle.apply_map(coords, cmap.standard_matrix)) < 1e-12


def test_integer_weights_equal_repeated_frames_featurised(topo):
    from aggforce_b200 import project_forces
    from aggforce_b200.qp import Multifeaturize, gb_feat, id_feat, qp_feat_linear_map

    coords, forces, n, rc, rf = _repeat_case(topo, 40, 21)
    cmap, cons = _cmap(topo), topo.xh_constraints
    feat = Multifeaturize([id_feat, functools.partial(gb_feat, **GB)])
    live = np.nonzero(n > 0)[0]
    frames = np.random.default_rng(5).choice(live, size=15, replace=False)
    first_copy = np.cumsum(n) - n  # index of frame t's first copy in the repeated arrays
    kw = dict(coord_map=cmap, constrained_inds=cons, method=qp_feat_linear_map, featurizer=feat, kbt=KBT,
              l2_regularization=1e3)
    got = project_forces(coords=coords, forces=forces, constraint_frames=frames, frame_weights=n, **kw)
    ref = project_forces(coords=rc, forces=rf, constraint_frames=first_copy[frames], **kw)
    cg = np.stack(got["tmap"].force_map.tags["coef_list"])
    cr = np.stack(ref["tmap"].force_map.tags["coef_list"])
    assert rel_fro(cg, cr) < MAP_TOL
    # the featurised QP is ill-conditioned: coefficients that agree to the map bar move the residual to first order
    # (l2 > 0), so the residual is held to the same bar as in test_gpu_feat.py
    assert abs(got["residual"] / ref["residual"] - 1) < MAP_TOL


# ------------------------------------------------------------------ scale invariances
def test_unit_weights_give_the_unweighted_fit(topo):
    """w = 1 runs the weighted DMMA kernel where the unweighted call of 10 000 float32 frames takes the int8 path."""
    from aggforce_b200 import Trajectory, _engine
    from aggforce_b200.qp import qp_linear_map
    from aggforce_b200.qp.qplinear import reduced_columns
    from aggforce_b200.synth import synth_trajectory_host

    coords, forces = synth_trajectory_host(topo, 10_000, seed=4)
    cmap, cons = _cmap(topo), topo.xh_constraints
    cols = reduced_columns(topo.n_sites, cons)
    n_red = int(cols.max()) + 1
    ones = np.ones(len(forces))
    g1 = _engine.to_host(_engine.gram_linear(_engine.Frames(forces), cols, n_red,
                                             weights=_engine.frame_weights_dev(ones, len(ones))))
    g0 = _engine.to_host(_engine.gram_linear(_engine.Frames(forces), cols, n_red))
    assert rel_fro(g1, g0) < GRAM_TOL
    traj = Trajectory(coords=coords, forces=forces)
    a = qp_linear_map(traj, cmap, cons, l2_regularization=1e3, frame_weights=ones).force_map.standard_matrix
    b = qp_linear_map(traj, cmap, cons, l2_regularization=1e3).force_map.standard_matrix
    assert rel_fro(a, b) < GRAM_TOL


@pytest.mark.parametrize("system", ["cln", "wide"])
def test_scaled_weights_with_scaled_l2_give_the_same_map(topo, wide, system):
    from aggforce_b200 import Trajectory
    from aggforce_b200.qp import qp_linear_map
    from aggforce_b200.synth import synth_trajectory_host

    t = topo if system == "cln" else wide
    coords, forces = synth_trajectory_host(t, 500, seed=17)
    w = _weights(len(forces), 2)
    traj, cmap = Trajectory(coords=coords, forces=forces), _cmap(t)
    a = qp_linear_map(traj, cmap, t.xh_constraints, l2_regularization=10.0, frame_weights=w)
    b = qp_linear_map(traj, cmap, t.xh_constraints, l2_regularization=10.0 * 37.5, frame_weights=37.5 * w)
    assert rel_fro(a.force_map.standard_matrix, b.force_map.standard_matrix) < GRAM_TOL


# ------------------------------------------------------------------ generic featurizer
def test_weighted_generic_featurizer_path_equals_fused(small_cln, golden, topo):
    from aggforce_b200 import Trajectory
    from aggforce_b200.qp import id_feat, qp_feat_linear_map

    ref = np.load(golden / "ref_idfeat.npz")
    cons = pairs_to_set(small_cln["cons10"])
    traj = Trajectory(coords=small_cln["coords"], forces=small_cln["forces"])
    w = _weights(len(small_cln["forces"]), 13)
    w[ref["frame_choice"]] = 1.0

    def custom(points, cmap, constraints):  # not recognised -> generic device path
        return id_feat(points, cmap, constraints)

    kw = dict(kbt=0.7, constraints=cons, l2_regularization=5.0, constraint_frames=ref["frame_choice"],
              frame_weights=w)
    a = qp_feat_linear_map(traj, _cmap(topo), custom, **kw)
    b = qp_feat_linear_map(traj, _cmap(topo), id_feat, **kw)
    ca, cb = np.stack(a.force_map.tags["coef_list"]), np.stack(b.force_map.tags["coef_list"])
    assert rel_fro(ca, cb) < 1e-9
    kw.pop("frame_weights")
    c = np.stack(qp_feat_linear_map(traj, _cmap(topo), id_feat, **kw).force_map.tags["coef_list"])
    assert rel_fro(ca, c) > 1e-6  # the weights changed the fit


# ------------------------------------------------------------------ weighted residual
@pytest.mark.parametrize("method", ["uni", "qp"])
@pytest.mark.parametrize("where", ["host", "device"])
def test_weighted_residual_matches_numpy(topo, method, where):
    from aggforce_b200 import project_forces
    from aggforce_b200.qp import constraint_aware_uni_map, qp_linear_map
    from aggforce_b200.synth import synth_trajectory_host

    coords, forces = synth_trajectory_host(topo, 400, seed=41)
    w = _weights(len(forces), 1)
    if where == "device":
        coords, forces = torch.as_tensor(coords, device="cuda"), torch.as_tensor(forces, device="cuda")
        w = torch.as_tensor(w, device="cuda", dtype=torch.float32)
    res = project_forces(coords=coords, forces=forces, coord_map=_cmap(topo), constrained_inds=topo.xh_constraints,
                         method=constraint_aware_uni_map if method == "uni" else qp_linear_map, frame_weights=w)
    mf = res["mapped_forces"]
    mf = mf.cpu().numpy() if isinstance(mf, torch.Tensor) else mf
    wn = w.double().cpu().numpy() if isinstance(w, torch.Tensor) else w
    ref = float(np.sum(wn * np.sum(mf.astype(np.float64) ** 2, axis=(1, 2))) / (3 * mf.shape[1] * wn.sum()))
    assert abs(res["residual"] / ref - 1) < 1e-12


# ------------------------------------------------------------------ validation
@pytest.mark.parametrize("bad", ["short", "2d", "negative", "nan", "inf", "zeros"])
def test_invalid_weights_raise(topo, bad):
    from aggforce_b200 import Trajectory, project_forces
    from aggforce_b200.qp import qp_feat_linear_map, qp_linear_map
    from aggforce_b200.synth import synth_trajectory_host

    coords, forces = synth_trajectory_host(topo, 30, seed=2)
    w = np.ones(30)
    w = {"short": w[:29], "2d": w.reshape(30, 1), "negative": np.where(np.arange(30) == 7, -1e-3, w),
         "nan": np.where(np.arange(30) == 3, np.nan, w), "inf": np.where(np.arange(30) == 3, np.inf, w),
         "zeros": np.zeros(30)}[bad]
    traj, cmap = Trajectory(coords=coords, forces=forces), _cmap(topo)
    with pytest.raises(ValueError, match="frame_weights"):
        qp_linear_map(traj, cmap, topo.xh_constraints, frame_weights=w)
    with pytest.raises(ValueError, match="frame_weights"):
        qp_feat_linear_map(traj, cmap, None, kbt=KBT, frame_weights=w)
    with pytest.raises(ValueError, match="frame_weights"):
        project_forces(coords=coords, forces=forces, coord_map=cmap, constrained_inds=topo.xh_constraints,
                       frame_weights=torch.as_tensor(w, device="cuda"))


def test_grid_cv_rejects_weights(topo):
    from aggforce_b200 import project_forces_grid_cv
    from aggforce_b200.synth import synth_trajectory_host

    coords, forces = synth_trajectory_host(topo, 30, seed=2)
    with pytest.raises(ValueError, match="frame_weights"):
        project_forces_grid_cv({"l2_regularization": [1.0]}, coords, forces, n_folds=2, coord_map=_cmap(topo),
                               constrained_inds=topo.xh_constraints, frame_weights=np.ones(30))


# ------------------------------------------------------------------ frame sharding
def test_nccl_sharded_weighted_fit_equals_single_gpu_fit():
    import socket
    import subprocess
    import sys
    from pathlib import Path

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = Path(__file__).resolve().parent / "dist_weights_check.py"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(n, 8)}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)]
    run = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert run.returncode == 0, run.stdout[-3000:] + run.stderr[-3000:]
    assert "-> OK" in run.stdout
