"""Orchestration: fit a force map and apply it (reference ``src/aggforce/agg.py``).

``project_forces`` keeps the reference's signature and result dictionary.  Every per-frame
reduction behind it runs on the GPU:
  constraint detection (kernel c) -> fit (kernel a + host QP, or kernel b) -> apply coords and
  forces (kernel d, the residual ``mean(F_mapped**2)`` fused into the force application).
Under ``aggforce_b200.frame_sharding()`` the arrays are this rank's frame slice; the fit
all-reduces its accumulators and the residual is the global mean.
"""
from __future__ import annotations

from gc import collect
from itertools import product
from typing import Any, Callable, Collection, Dict, Final, List, Mapping, NamedTuple, Optional, Tuple, Union

import numpy as np
import torch

from . import _engine
from .constraints import Constraints, guess_pairwise_constraints
from .map import LinearMap, SeperableTMap, TMap
from .qp import constraint_aware_uni_map, qp_linear_map
from .trajectory import Trajectory

PROJECT_FORCES_CNSTR_AUTO: Final = "auto"

SCORES_KNAME: Final = "scores"
SDS_KNAME: Final = "sds"
NRUNS_KNAME: Final = "n_runs"

PROJFORCES_KNAME: Final = "mapped_forces"
PROJCOORDS_KNAME: Final = "mapped_coords"
TMAP_KNAME: Final = "tmap"
RESIDUAL_KNAME: Final = "residual"
CONSTRAINTS_KNAME: Final = "constraints"


def force_smoothness(array) -> float:
    """Mean squared element of ``array`` (reference agg.py:291-297)."""
    if isinstance(array, torch.Tensor):
        return float((array.double() ** 2).mean().item())
    return float(np.mean(np.asarray(array) ** 2))


def _global_mean_sq(sumsq: float, shape) -> float:
    local = np.array([sumsq, float(np.prod(shape))])
    tot = np.sum(_engine.allgather_host(local), axis=0)
    return float(tot[0] / tot[1])


def _weighted_residual(mapped_forces, weights: torch.Tensor) -> float:
    """``sum_t w_t sum F_t**2 / (size of one frame * sum_t w_t)`` over all ranks (maps applied as a whole)."""
    dev = mapped_forces if isinstance(mapped_forces, torch.Tensor) else torch.as_tensor(mapped_forces)
    dev = dev.to(_engine.device())
    num = torch.zeros(1, dtype=torch.float64, device=dev.device)
    _engine.weighted_sumsq(dev, weights, num)
    per_frame = float(np.prod(tuple(dev.shape[1:])))
    local = _engine.to_host(torch.cat([num, (weights.sum() * per_frame).reshape(1)]))
    tot = np.sum(_engine.allgather_host(local), axis=0)
    return float(tot[0] / tot[1])


def project_forces(
    coords,
    forces,
    coord_map: LinearMap,
    constrained_inds: Union[Constraints, str, None] = PROJECT_FORCES_CNSTR_AUTO,
    method: Callable[..., TMap] = qp_linear_map,
    **kwargs,
) -> Dict[str, Any]:
    """Produce an optimised force map and the mapped trajectory.

    Arguments as in the reference: ``coords``/``forces`` of shape ``(n_steps, n_sites, 3)``
    (numpy arrays, or torch CUDA tensors for device-resident data), ``coord_map`` the
    configurational ``LinearMap``, ``constrained_inds`` a set of frozensets or ``"auto"``
    (``guess_pairwise_constraints`` on all of ``coords``), ``method`` any callable
    ``(traj, coord_map, constraints, **kwargs) -> TMap``.

    Returns a dict with keys ``mapped_coords``, ``mapped_forces``, ``tmap``, ``residual``
    (mean squared mapped force, not held out) and ``constraints``.

    ``frame_weights`` (extension, keyword): one non-negative weight per frame (numpy or CUDA tensor; under
    ``frame_sharding`` the weights of this rank's frames), for trajectories that are not samples of the
    target ensemble (reweighted biased runs, pooled or bootstrapped datasets).  It is forwarded to
    ``method`` (``qp_linear_map`` and ``qp_feat_linear_map`` fit the weighted objective,
    ``constraint_aware_uni_map`` ignores it) and the residual becomes the weighted mean
    ``sum_t w_t sum F_t**2 / (3 n_cg sum_t w_t)``.  ``mapped_coords`` / ``mapped_forces`` are the per-frame
    mapped arrays as without weights.  Constraint detection (``constrained_inds="auto"``) stays
    unweighted: a rigid pair is rigid in every frame, whatever its weight.
    """
    auto = isinstance(constrained_inds, str) and constrained_inds == PROJECT_FORCES_CNSTR_AUTO
    if auto and coords is None:
        raise ValueError(f"If constrained_inds is {PROJECT_FORCES_CNSTR_AUTO}, coords cannot be None.")
    t = Trajectory(coords=coords, forces=forces)
    # one device upload per array, shared by constraint detection, the fit and the application: while
    # this context is open Frames(coords) / Frames(forces) anywhere below resolve to the same upload,
    # and every method (also user callables and generic featurizers) receives the caller's own arrays
    with _engine.shared_uploads(coords, forces):
        return _project_forces(t, coords, forces, coord_map, constrained_inds, auto, method, kwargs)


def _project_forces(t, coords, forces, coord_map, constrained_inds, auto, method, kwargs) -> Dict[str, Any]:
    coords_in, forces_in = _engine.Frames(coords), _engine.Frames(forces)
    weights = _engine.frame_weights_dev(kwargs.get("frame_weights"), forces_in.n_frames)
    if weights is not None:
        kwargs = dict(kwargs, frame_weights=weights)  # checked and uploaded once: the method reuses it
    if auto:
        constrained_inds = guess_pairwise_constraints(coords_in)
    # ONE status buffer for both applications: [sum(out_c^2), sum(out_f^2), n_elements, flags_c, flags_f]
    # (each flag slot holds two int32: saw_nan, nan_violation).  Under frame sharding the first three are
    # summed and the flag slots max-ed over the ranks by one exchange -- as float64 bit patterns two small
    # non-negative int32 order like the pair (violation, saw), so a violation on any rank survives.
    stat = torch.zeros(5, dtype=torch.float64, device=_engine.device())
    slots_c, slots_f = (stat[0:1], stat[3:4]), (stat[1:2], stat[4:5])
    # The coordinate map does not depend on the fit: its application is deferred to the moment the
    # fit has enqueued its last kernel (or launched right here when the fit never asks), so it runs
    # on the GPU while the host builds / solves the map.
    early: Dict[str, Any] = {}
    dl_c: list = []  # pinned copies of the mapped arrays whose download has been started (host input only)
    dl_f: list = []
    if isinstance(coord_map, LinearMap) and coords is not None:
        if method is qp_linear_map and not coords_in.on_host and coord_map.n_fg_sites > 1024:
            # large fits go through cuSOLVER with host-side checks: [Gram][coordinate map] | solve
            _engine.defer(lambda: early.update(launch=coord_map._launch(coords_in, slots=slots_c)))
        elif method is qp_linear_map or method is constraint_aware_uni_map:
            # runs while the host builds the uniform map or prepares the fit's launches (small fits are solved on
            # the device: nothing later in the call would hide it better); for host arrays its download (started
            # inside) leaves over PCIe while the forces arrive and the fit runs
            early["launch"] = coord_map._launch(coords_in, slots=slots_c, download=dl_c)
        # other methods return maps that are applied as a whole (featurised / augmented): nothing to hoist
    try:
        with _engine.deferred_fits():  # a device-side fit reports through the read below
            traj_map: TMap = method(
                traj=t,
                coord_map=coord_map,
                constraints=constrained_inds,
                **kwargs,
            )
    except BaseException:
        _engine.clear_deferred()
        raise
    if (isinstance(traj_map, SeperableTMap) and isinstance(traj_map.force_map, LinearMap)
            and isinstance(traj_map.coord_map, LinearMap)):
        # both applications are enqueued back to back; one read returns the NaN flags, the residual
        # sum and -- for a fit solved on the device -- the solver status and the fitted coefficients
        cm, fm = traj_map.coord_map, traj_map.force_map
        if cm is not coord_map:
            _engine.clear_deferred()
            if "launch" in early:
                early.clear()
                dl_c.clear()
                stat.zero_()
        _engine.run_deferred()
        fc, oc, _ = early["launch"] if "launch" in early else cm._launch(coords_in, slots=slots_c, download=dl_c)
        ff, of, _ = fm._launch(forces_in, want_sumsq=weights is None, slots=slots_f, download=dl_f)
        host_c = dl_c[0] if dl_c else None  # downloads overlap the force upload, piece by piece
        host_f = dl_f[0] if dl_f else None
        pend = fm._pending if fm._matrix is None else None
        n_elem = float(np.prod(of.shape))
        if weights is not None:  # weighted residual: numerator and denominator 3 n_cg sum(w) in the same slots
            _engine.weighted_sumsq(of, weights, stat[1:2])
            stat[2:3].copy_((weights.sum() * float(np.prod(of.shape[1:]))).reshape(1))
        if _engine.sharded():
            # residual numerator / denominator are summed over ranks and the NaN flags max-ed, so that a
            # violated NaN protocol raises on every rank (a lone raiser would leave the others in the next
            # collective): ONE message
            if weights is None:
                stat[2:3].copy_(_engine.dev_f64([n_elem]))
            _engine.allreduce_sum_max_(stat, 3)
        if pend is not None and pend.buf is None:
            pend = None  # a large device fit: checked when it was solved, downloaded only on request
        got = _engine.read_many([stat] + ([pend.buf] if pend is not None else []))
        st = got[0]
        if _engine.sharded() or weights is not None:
            n_elem = float(st[2])
        status = np.array([st[0], st[1], st[3], st[4]])
        if pend is not None:
            fm._matrix = pend.resolve(got[1])  # raises ValueError("Map optimization failed.") like the host path
            fm._adopt_device_fit()
        if pend is not None and pend.fell_back:
            # the device solve declined (P or the Schur complement not positive definite): the host
            # solution replaces the map and the force application is redone with it
            fm = LinearMap(pend.expanded, handle_nans=fm.handle_nans, nan_check_threshold=fm.nan_check_threshold)
            fm._column_labels = pend.cols
            traj_map = SeperableTMap(coord_map=cm, force_map=fm)
            mapped_coords = cm._finish(fc, oc, status[2:3], host_c)
            mapped_forces = fm(forces_in)
            if weights is not None:
                residual = _weighted_residual(mapped_forces, weights)
            else:
                residual = _global_mean_sq(float((torch.as_tensor(mapped_forces).double() ** 2).sum()),
                                           mapped_forces.shape)
        else:
            mapped_coords = cm._finish(fc, oc, status[2:3], host_c)
            mapped_forces = fm._finish(ff, of, status[3:4], host_f)
            residual = float(status[1] / n_elem)
    else:
        _engine.clear_deferred()
        mapped = traj_map(t)
        mapped_coords, mapped_forces = mapped.coords, mapped.forces
        residual = force_smoothness(mapped_forces) if weights is None else _weighted_residual(mapped_forces, weights)
    return {
        PROJCOORDS_KNAME: mapped_coords,
        PROJFORCES_KNAME: mapped_forces,
        TMAP_KNAME: traj_map,
        RESIDUAL_KNAME: residual,
        CONSTRAINTS_KNAME: constrained_inds,
    }


def project_forces_grid_cv(
    cv_arg_dict: Mapping[str, List[Any]],
    coords,
    forces,
    n_folds: int = 5,
    rng: Optional[np.random.Generator] = None,
    **kwargs,
) -> Dict[str, Dict[Any, Any]]:
    """K-fold cross validation of ``project_forces`` over a grid of arguments (reference
    ``agg.py:142-235``): for every parameter combination, ``scores`` holds the hold-out
    ``force_smoothness`` averaged over folds, ``sds`` its sample standard deviation and ``n_runs``
    the number of folds whose optimisation succeeded.  ``rng`` (extension) seeds the fold
    shuffle, which the reference leaves unseeded (``agg.py:188``).

    Fast path (SURVEY 8f-3) when the method is ``qp_linear_map``, the constraints are given and the
    grid only varies ``l2_regularization``: ONE pass over the data accumulates a Gram per fold
    (kernel (a)); the training Gram of a fold is the total minus its own, and the hold-out score
    is ``trace(W G_fold W') / (3 T_fold n_cg)`` -- no further pass over the frames for any grid
    point.  Everything else runs ``project_forces`` per fold and grid point as the reference does
    (it calls ``tmap.from_arrays``, which no TMap defines; ``map_arrays`` is used here).

    ``frame_weights`` are not supported here: per-fold fits would need the weights of each fold's frames.
    Passing them raises ``ValueError``.
    """
    if kwargs.get("frame_weights") is not None:
        raise ValueError("project_forces_grid_cv does not take frame_weights: the full-length weights do not match "
                         "the frames of a fold's fit")
    n_frames = forces.shape[0]
    frames = np.arange(n_frames)
    (np.random.default_rng() if rng is None else rng).shuffle(frames)
    folds = np.array_split(frames, n_folds, axis=0)
    grid = process_cvargs(cv_arg_dict)
    results: Dict[str, Dict[Any, Any]] = {SCORES_KNAME: {}, SDS_KNAME: {}, NRUNS_KNAME: {}}

    fast = (kwargs.get("method", qp_linear_map) is qp_linear_map and set(cv_arg_dict) <= {"l2_regularization"}
            and not isinstance(kwargs.get("constrained_inds", PROJECT_FORCES_CNSTR_AUTO), str)
            and dict(kwargs.get("solver_args") or {}).get("backend", "exact") == "exact"
            and isinstance(kwargs.get("coord_map"), LinearMap) and not _engine.sharded())
    fold_scores: Dict[Any, List[float]] = {label: [] for label, _ in grid}
    if fast:
        from .qp.qplinear import reduced_columns
        from .qp.solver import solve_equality_qp

        coord_map, cons = kwargs["coord_map"], kwargs.get("constrained_inds") or set()
        n_fg, n_cg = coord_map.n_fg_sites, coord_map.n_cg_sites
        cols = reduced_columns(n_fg, cons)
        n_red = int(cols.max()) + 1
        src = _engine.Frames(forces)
        grams = [_engine.to_host(_engine.gram_linear(_engine.Frames(src.gather(np.sort(idx))), cols, n_red))
                 for idx in folds]
        total = np.sum(grams, axis=0)
        group_size = np.bincount(cols, minlength=n_red).astype(np.float64)
        cmat = np.asarray(coord_map.standard_matrix, dtype=np.float64)
        a_mat = np.zeros((n_cg, n_red))
        np.add.at(a_mat.T, cols, cmat.T)
        for label, args in grid:
            l2 = float(args.get("l2_regularization", kwargs.get("l2_regularization", 0.0)))
            for fold, g_val in zip(folds, grams):
                p_train = total - g_val
                if l2 > 0.0:
                    p_train[np.diag_indices(n_red)] += l2 * group_size
                sol = solve_equality_qp(p_train, a_mat, np.eye(n_cg))
                if sol is None:
                    print("Map optimization failed.")
                    continue
                w = sol.T  # (n_cg, n_red) reduced weights
                fold_scores[label].append(float(np.einsum("cr,rs,cs->", w, g_val, w) / (3.0 * len(fold) * n_cg)))
    else:
        is_dev = isinstance(forces, torch.Tensor)
        take = (lambda arr, idx: arr[torch.as_tensor(idx, device=arr.device)]) if is_dev else (lambda arr, idx: arr[idx])
        outside = [np.concatenate([f for j, f in enumerate(folds) if j != i]) for i in range(len(folds))]
        for label, args in grid:
            combined = dict(kwargs, **args)
            for train_inds, val_inds in zip(outside, folds):
                try:
                    tmap = project_forces(coords=None if coords is None else take(coords, train_inds),
                                          forces=take(forces, train_inds), **combined)[TMAP_KNAME]
                    _, val_forces = tmap.map_arrays(None if coords is None else take(coords, val_inds),
                                                    take(forces, val_inds))
                    fold_scores[label].append(force_smoothness(val_forces))
                    del tmap
                except ValueError as e:  # failed optimisation: the fold is skipped, as in the reference
                    print(e)
                collect()
    for label, _ in grid:
        results[SCORES_KNAME][label] = mean(fold_scores[label])
        results[SDS_KNAME][label] = sample_sd(fold_scores[label])
        results[NRUNS_KNAME][label] = len(fold_scores[label])
    return results


def process_cvargs(arg_dict: Mapping[str, List[Any]]) -> List[Tuple[Any, Dict[str, Any]]]:
    """Grid of parameter combinations: ``[(CVArgs(key1=v, key2=w, ...), {key1: v, key2: w, ...}), ...]``
    for every element of the product of the value lists (reference ``agg.py:238-288``)."""
    names = list(arg_dict.keys())
    cv_args = NamedTuple("CVArgs", [(n, Any) for n in names])  # type: ignore[misc]
    out = []
    for values in product(*[arg_dict[n] for n in names]):
        key = cv_args(**dict(zip(names, values)))
        out.append((key, {n: getattr(key, n) for n in names}))
    return out


def mean(s: Collection[float]) -> Union[float, None]:
    """Arithmetic mean, ``None`` for an empty collection (reference ``agg.py:300-318``)."""
    return None if len(s) == 0 else sum(s) / len(s)


def sample_sd(s: Collection[float]) -> Union[float, None]:
    """Sample standard deviation, ``None`` for an empty collection (reference ``agg.py:321-343``;
    a single element divides by zero there -- NaN here)."""
    m = mean(s)
    if m is None:
        return None
    if len(s) < 2:
        return float("nan")
    return (sum((o - m) ** 2 for o in s) / (len(s) - 1)) ** 0.5
