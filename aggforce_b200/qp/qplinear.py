"""Optimal static linear force map -- kernel (a) plus the host QP.

Drop-in for the reference's ``src/aggforce/qp/qplinear.py``.
"""
from __future__ import annotations

import functools
import hashlib
from typing import Union

import numpy as np
import scipy.sparse as ss
import torch

from .. import _engine, _lib
from ..constraints import Constraints, constraint_lookup_dict, merged_groups
from ..map import LinearMap, SeperableTMap
from ..trajectory import ForcesTrajectory
from .solver import (DEFAULT_SOLVER_OPTIONS, SolverOptions, solve, solve_equality_qp_device,
                     warn_if_solver_ignored)


def reduced_columns(n_sites: int, constraints: Constraints) -> np.ndarray:
    """Reduced-coefficient column of every site (``int64[n_sites]``).

    Sites constrained together share one coefficient.  Column order follows the reference
    (``qplinear.py:157-163``): walking the sites in increasing order, every site that is not a
    dependent member of a merged constraint group opens the next column; dependents reuse
    their anchor's (the smallest index of their group).  Pure index bookkeeping: memoised on the
    constraint set (a fit, the uniform map and the CV folds all ask for the same table).
    """
    try:
        key = frozenset(constraints)
    except TypeError:  # unhashable members: compute directly
        return _reduced_columns(n_sites, constraints)
    return _reduced_columns_cached(n_sites, key).copy()


@functools.lru_cache(maxsize=16)
def _reduced_columns_cached(n_sites: int, constraints: frozenset) -> np.ndarray:
    cols = _reduced_columns(n_sites, constraints)
    cols.setflags(write=False)
    return cols


def _reduced_columns(n_sites: int, constraints: Constraints) -> np.ndarray:
    anchor_of = constraint_lookup_dict(merged_groups(constraints))
    cols = np.full(n_sites, -1, dtype=np.int64)
    free = [s for s in range(n_sites) if s not in anchor_of]
    cols[free] = np.arange(len(free))
    for site, anchor in anchor_of.items():
        cols[site] = cols[anchor]
    return cols


def make_bond_constraint_matrix(n_sites: int, constraints: Constraints) -> np.ndarray:
    """One-hot ``(n_sites, n_reduced)`` matrix expanding reduced coefficients to all sites."""
    cols = reduced_columns(n_sites, constraints)
    mat = np.zeros((n_sites, int(cols.max()) + 1 if n_sites else 0))
    mat[np.arange(n_sites), cols] = 1
    return mat


def qp_form(target: np.ndarray) -> np.ndarray:
    """``(n_steps, n_sites, 3) -> (n_steps*3, n_sites)`` with rows ordered (step, dim)."""
    mixed = np.swapaxes(target, 1, 2)
    return np.reshape(mixed, (mixed.shape[0] * mixed.shape[1], -1))


def force_gram(forces, n_sites: int, constraints: Constraints, weights=None):
    """``(gram (n_red, n_red) float64 on the host, columns)`` -- the QP objective of
    ``qplinear.py:66-71``, accumulated on the GPU and all-reduced across frame shards
    (``weights``: per-frame weights from ``_engine.frame_weights_dev``)."""
    cols = reduced_columns(n_sites, constraints)
    n_red = int(cols.max()) + 1
    gram = _engine.gram_linear(_engine.Frames(forces), cols, n_red, weights=weights)
    return _engine.to_host_overlapped(gram), cols


# reduced problems at least this large are solved on the device by cuSOLVER (through torch.linalg);
# small ones (n_red <= 128, n_cg <= 32) by the one-CTA kernel agf_qp_equality_small, so that
# Gram -> solve -> force application never stops at the host; what lies between goes to the host
_DEVICE_SOLVE_MIN = 512


class _DeviceFit:
    """Result of ``agf_qp_equality_small`` that still lives on the device.

    ``buf`` is ONE float64 device buffer ``[qp status | apply status slots | X (n_cg x n_red)]`` so that
    ``project_forces`` gets the solver status, both applications' NaN flags, the residual sum and the
    fitted coefficients with a single read.  ``matrix()`` is what ``LinearMap.standard_matrix`` calls
    on first access when nobody resolved the fit before."""

    N_HEAD = 6  # [0] qp status (int32), [1:3] coordinate-map status, [3:5] force-map status, [5] spare

    def __init__(self, buf, gram, order, cols, n_red, n_cg, diag, a_mat, solver_args) -> None:
        self.buf, self.gram, self.order, self.cols = buf, gram, order, cols
        self.n_red, self.n_cg, self.diag, self.a_mat, self.solver_args = n_red, n_cg, diag, a_mat, solver_args
        self.expanded: Union[None, np.ndarray] = None
        self.fell_back = False

    def resolve(self, host_buf: np.ndarray) -> np.ndarray:
        """Check the solver status in a downloaded copy of ``buf`` and return the expanded matrix
        (host fallback -- exact solve with its null-space branch -- when the device solve failed)."""
        if self.expanded is None:
            status = int(np.ascontiguousarray(host_buf[0:1]).view(np.int32)[0])
            if status == 0:
                reduced = host_buf[self.N_HEAD:].reshape(self.n_cg, self.n_red)
            else:
                self.fell_back = True
                gram = self.gram.clone()
                _lib.call("agf_symmetrize", _engine.ptr(gram), self.n_red, _engine.stream_ptr())
                qp_mat = _engine.to_host(gram)
                back = np.empty(self.n_red, dtype=np.int64)
                back[self.order] = np.arange(self.n_red)
                qp_mat = qp_mat[back][:, back]
                qp_mat[np.diag_indices(self.n_red)] += self.diag
                sol = solve(qp_mat, self.a_mat, np.eye(self.n_cg), self.solver_args)
                if sol is None:
                    raise ValueError("Map optimization failed.")
                reduced = sol.T
            self.expanded = np.ascontiguousarray(reduced[:, self.cols])
            self.gram = None
        return self.expanded

    def matrix(self) -> np.ndarray:
        if self.expanded is None:
            self.resolve(_engine.to_host(self.buf))
        return self.expanded


class _LargeDeviceFit:
    """Result of the cuSOLVER path (n_red >= 512) that stays on the device: ``x_dev`` is the float64
    ``(n_red, n_cg)`` solution, already checked (finite, equality rows met) when it was computed, so nothing
    has to be read before the map is applied; ``matrix()`` downloads and expands it on first host access."""

    buf = None  # no status to read: project_forces does not resolve this fit eagerly
    fell_back = False

    def __init__(self, x_dev, cols: np.ndarray) -> None:
        self.x_dev, self.cols = x_dev, cols
        self.expanded: Union[None, np.ndarray] = None

    def matrix(self) -> np.ndarray:
        if self.expanded is None:
            reduced = _engine.to_host(self.x_dev).T
            self.expanded = np.ascontiguousarray(reduced[:, self.cols])
            self.x_dev = None
        return self.expanded

    def resolve(self, _host_buf=None) -> np.ndarray:
        return self.matrix()


def _equality_rows(coord_map: LinearMap, cols: np.ndarray, n_red: int) -> np.ndarray:
    """``A = coord_map @ C``: the coordinate-map columns of every group summed (qplinear.py:82)."""
    n_fg = coord_map.n_fg_sites
    cmat = np.asarray(coord_map.standard_matrix, dtype=np.float64)
    if n_fg * coord_map.n_cg_sites <= (1 << 16):  # small: a scatter-add beats building a sparse one-hot
        a_mat = np.zeros((coord_map.n_cg_sites, n_red))
        np.add.at(a_mat.T, cols, cmat.T)
        return a_mat
    onehot = ss.csr_matrix((np.ones(n_fg), (np.arange(n_fg), cols)), shape=(n_fg, n_red))
    return np.asarray((onehot.T @ cmat.T).T)


_EQ_ROWS_CACHE: dict = {}


def _equality_rows_cached(coord_map: LinearMap, cols: np.ndarray, n_red: int, want_device: bool):
    """``(A, A on the device or None)`` for large fits: building ``A = cmap C`` (a sparse product over a 500 x 5 000
    map) and uploading its 10 MB cost 8 ms per call at the config-4 shape; both are functions of the coordinate
    map's content and the column table only.  The key reuses the content digest the map's own compile step took
    a moment ago (``LinearMap._compile``), so an edited map misses."""
    compiled = getattr(coord_map, "_compiled", None)
    digest = compiled[0] if compiled is not None and isinstance(compiled[0], bytes) and compiled[0] != b"device-fit" else None
    if digest is None or not isinstance(coord_map, LinearMap):
        a_mat = _equality_rows(coord_map, cols, n_red)
        return a_mat, (_engine.dev_f64(a_mat) if want_device else None)
    key = (digest, hash(np.ascontiguousarray(cols).tobytes()), int(n_red), _engine.device().index)
    hit = _EQ_ROWS_CACHE.get(key)
    if hit is None:
        if len(_EQ_ROWS_CACHE) > 8:
            _EQ_ROWS_CACHE.clear()
        a_mat = _equality_rows(coord_map, cols, n_red)
        hit = _EQ_ROWS_CACHE[key] = [a_mat, None]
    if want_device and hit[1] is None:
        hit[1] = torch.as_tensor(hit[0], device=_engine.device())
    return hit[0], hit[1]


class _SmallFitPlan:
    """Everything about a small device-side fit that depends only on (coordinate map, constraints, l2):
    column order, CSR of the groups, equality rows, index maps of the QP kernel's outputs and the
    structure of the fitted map -- host bookkeeping and small device tables, built once and reused."""

    cache: dict = {}

    def __init__(self, coord_map: LinearMap, cols: np.ndarray, n_red: int, l2: float) -> None:
        self.cols, self.n_red, self.n_cg = cols, n_red, coord_map.n_cg_sites
        self.gram_plan = _engine.GramPlan(cols, n_red)
        order = self.gram_plan.order
        group_size = np.bincount(cols, minlength=n_red).astype(np.float64)
        self.diag = (l2 if l2 > 0.0 else 0.0) * group_size
        self.a_mat = _equality_rows(coord_map, cols, n_red)
        self.compiled_structure, ucol_of_col = _engine.CompiledMap.from_labels(cols, self.n_cg, n_red)
        self.d_diag = _engine.dev_f64(self.diag[order]) if l2 > 0.0 else None
        self.d_a = _engine.dev_f64(self.a_mat[:, order])
        self.d_x_index = _engine.dev_i32(order)
        self.d_u_index = _engine.dev_i32(ucol_of_col[order])

    @classmethod
    def get(cls, coord_map: LinearMap, constraints, cols: np.ndarray, n_red: int, l2: float) -> "_SmallFitPlan":
        try:
            m = np.asarray(coord_map.standard_matrix)
            key = (m.shape, hashlib.blake2b(np.ascontiguousarray(m, dtype=np.float64).tobytes(), digest_size=16).digest(),
                   frozenset(constraints), float(l2), _engine.device().index)
        except TypeError:
            return cls(coord_map, cols, n_red, l2)
        plan = cls.cache.get(key)
        if plan is None:
            if len(cls.cache) > 16:
                cls.cache.clear()
            plan = cls.cache[key] = cls(coord_map, cols, n_red, l2)
        return plan


def _fit_small_on_device(traj, coord_map: LinearMap, constraints, cols: np.ndarray, n_red: int, l2: float,
                         solver_args, weights=None) -> SeperableTMap:
    """Gram (kernel a) -> ``agf_qp_equality_small`` -> a ``LinearMap`` whose coefficients are already
    where kernel (d) reads them.  Nothing synchronises here when called through ``project_forces``
    (which reads status + coefficients once, after the applications); a direct call resolves the fit
    before returning, as the reference raises at fit time."""
    plan = _SmallFitPlan.get(coord_map, constraints, cols, n_red, l2)
    n_cg = plan.n_cg
    gram, order = _engine.gram_linear_raw(_engine.Frames(traj.forces), cols, n_red, plan=plan.gram_plan, weights=weights)
    _engine.run_deferred()
    compiled = plan.compiled_structure.with_values(torch.empty((n_red, n_cg), dtype=torch.float64, device=gram.device))
    buf = torch.zeros(_DeviceFit.N_HEAD + n_cg * n_red, dtype=torch.float64, device=gram.device)
    p = _engine.ptr
    _lib.call("agf_qp_equality_small", p(gram), n_red, p(plan.d_diag), p(plan.d_a), n_cg, p(plan.d_x_index),
              p(buf[_DeviceFit.N_HEAD:]), p(plan.d_u_index), p(compiled.umat_t), p(buf[0:1]), _engine.stream_ptr())
    fit = _DeviceFit(buf, gram, order, cols, n_red, n_cg, plan.diag, plan.a_mat, solver_args)
    force_map = LinearMap.from_device_fit(fit, n_cg, cols, compiled)
    if not _engine.fits_deferred():
        fit.matrix()  # direct call: synchronise, check the solver status (ValueError on failure)
        if fit.fell_back:
            force_map = LinearMap(fit.expanded)
            force_map._column_labels = cols
    return SeperableTMap(coord_map=coord_map, force_map=force_map)


def qp_linear_map(
    traj: ForcesTrajectory,
    coord_map: LinearMap,
    constraints: Union[None, Constraints] = None,
    l2_regularization: float = 0.0,
    solver_args: SolverOptions = DEFAULT_SOLVER_OPTIONS,
    frame_weights=None,
) -> SeperableTMap:
    """Linear force map minimising the mean squared mapped force.

    Same contract as the reference: constrained sites share coefficients, the map satisfies
    ``coord_map @ W.T = I`` on the reduced coefficients, ``l2_regularization`` penalises the
    expanded coefficient vector and is relative to the *unnormalised* frame sum.

    ``solver_args``: the reference hands them to ``qpsolvers.solve_qp`` (OSQP by default).  Here the
    problem is solved exactly (closed form, on the device for small and for large reduced problems)
    unless ``solver_args={"backend": "qpsolvers", ...}``; other keys given without that backend are
    reported once with a warning and not used.

    ``frame_weights`` (extension): one non-negative weight per frame (numpy or CUDA tensor; under
    ``frame_sharding`` the weights of this rank's frames).  The objective becomes the raw weighted sum
    ``P = sum_t w_t r_t r_t^T`` -- not normalised, so ``l2_regularization`` stays relative to that sum and
    scaling both by ``c`` gives the same map.  Integer weights equal repeating frames.
    """
    if constraints is None:
        constraints = set()
    warn_if_solver_ignored(solver_args)
    n_fg = coord_map.n_fg_sites
    if traj.forces.shape[1] != n_fg:
        raise ValueError("coord_map and forces disagree on the number of fine-grained sites.")
    weights = _engine.frame_weights_dev(frame_weights, traj.forces.shape[0])
    backend = dict(solver_args or {}).get("backend", "exact")
    cols = reduced_columns(n_fg, constraints)
    n_red = int(cols.max()) + 1
    on_device = backend == "exact" and n_red >= _DEVICE_SOLVE_MIN
    n_cg = coord_map.n_cg_sites
    if (backend == "exact" and not on_device and isinstance(coord_map, LinearMap)
            and _lib.lib().agf_qp_equality_small_supported(n_red, n_cg)):
        return _fit_small_on_device(traj, coord_map, constraints, cols, n_red, l2_regularization, solver_args,
                                    weights)
    if on_device:
        qp_mat = _engine.gram_linear(_engine.Frames(traj.forces), cols, n_red, weights=weights)  # stays on the device
        _engine.run_deferred()
    else:
        qp_mat, cols = force_gram(traj.forces, n_fg, constraints, weights)
    group_size = np.bincount(cols, minlength=n_red).astype(np.float64)
    if l2_regularization > 0.0:  # l2 * C'C
        if on_device:
            qp_mat.diagonal().add_(torch.as_tensor(l2_regularization * group_size, device=qp_mat.device))
        else:
            qp_mat[np.diag_indices(n_red)] += l2_regularization * group_size
    a_mat, a_dev = _equality_rows_cached(coord_map, cols, n_red, on_device)
    if backend == "exact":
        sol = None
        if on_device:
            sol = solve_equality_qp_device(qp_mat, a_dev, np.eye(coord_map.n_cg_sites), keep_on_device=True)
            if sol is not None:
                # the solution is the coefficient operand of kernel (d) up to a row permutation: the fitted map
                # is applied from the device, its 20 MB host form (500 x 5 000) only exists if somebody asks
                structure, ucol_of_col = _engine.CompiledMap.from_labels(cols, n_cg, n_red)
                pos = _engine._dev_cached(np.ascontiguousarray(np.argsort(ucol_of_col), dtype=np.int64))
                compiled = structure.with_values(sol.index_select(0, pos).contiguous())
                force_map = LinearMap.from_device_fit(_LargeDeviceFit(sol, cols), n_cg, cols, compiled)
                return SeperableTMap(coord_map=coord_map, force_map=force_map)
            qp_mat = _engine.to_host(qp_mat)  # not numerically positive definite: host path, null-space fallback
        if sol is None:
            sol = solve(qp_mat, a_mat, np.eye(coord_map.n_cg_sites), solver_args)
        if sol is None:
            raise ValueError("Map optimization failed.")
        reduced = sol.T
    else:
        rows = []
        for bead in range(coord_map.n_cg_sites):
            target = np.zeros(coord_map.n_cg_sites)
            target[bead] = 1
            x = solve(qp_mat, a_mat, target, solver_args)
            if x is None:
                raise ValueError("Map optimization failed.")
            rows.append(x)
        reduced = np.stack(rows)
    force_map = LinearMap(reduced[:, cols])
    force_map._column_labels = cols  # sites of one reduced column share their matrix column by construction
    return SeperableTMap(coord_map=coord_map, force_map=force_map)
