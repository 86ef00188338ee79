"""Featurised (configuration dependent) force maps.

API of the reference's ``src/aggforce/qp/featlinearmap.py``: featurizer protocol
``(points, cmap, constraints) -> {"feats", "divs", "names"}``, ``FeatZipper`` / ``Multifeaturize``
to combine featurizers, ``id_feat``, and ``qp_feat_linear_map``.

Two execution paths behind ``qp_feat_linear_map``:

* **fused** -- the featurizer is (a ``Multifeaturize`` of) ``id_feat`` and/or ``gb_feat`` (plain,
  ``Curry`` or ``functools.partial``).  The per-bead Gram, the equality rows and the application of
  the fitted map run in ``csrc/featgram.cu``; features are never materialised.
* **generic** -- any other featurizer callable: its arrays are uploaded bead by bead and the
  regression rows / Gram are formed on the device with library contractions (float64).  This keeps
  user-defined featurizers working; it is not the optimised path.
"""
from __future__ import annotations

import functools
from copy import deepcopy
from queue import Empty, SimpleQueue
from typing import Any, Callable, ClassVar, Dict, Final, Generator, Iterable, List, Optional, Tuple, Union

import ctypes as C

import numpy as np
import scipy.sparse as ss
import torch
from numpy.random import default_rng

from .. import _engine, _lib
from ..constraints import Constraints, reduce_constraint_sets
from ..map import CLAFTMap, CLAMap, LinearMap
from ..trajectory import Trajectory
from ..util import Curry
from .gbfeat import GbSpec, gb_feat
from .solver import (DEFAULT_SOLVER_OPTIONS, SolverOptions, solve, solve_equality_qp_device,
                     solve_equality_qp_device_batched, warn_if_solver_ignored)

_DEVICE_SOLVE_MIN = 512  # feature counts from which the per-bead QP is solved on the device

KNAME_FEATS: Final = "feats"
KNAME_DIVS: Final = "divs"
KNAME_NAMES: Final = "names"

Features = Dict[str, Any]
Featurizer = Callable[[Any, LinearMap, Constraints], Features]
GeneralizedFeatures = Union[Features, "FeatZipper"]
GeneralizedFeaturizer = Callable[[Any, LinearMap, Constraints], GeneralizedFeatures]


def _cat(arrays, axis: int):
    if any(isinstance(a, torch.Tensor) for a in arrays):
        return torch.cat([torch.as_tensor(a) for a in arrays], dim=axis)
    return np.concatenate(arrays, axis=axis)


class FeatZipper:
    """Lazily concatenates the outputs of several featurizers, bead by bead.

    Indexing with ``"feats"`` / ``"divs"`` returns a generator over beads whose items are the
    member outputs joined along the feature axis (axis 2 for features, axis 1 for divergences);
    ``"names"`` is ``None``.  Member iterables are advanced only when an item is requested.
    """

    generator_keys = frozenset([KNAME_FEATS, KNAME_DIVS])
    name_key = "names"
    joiners: ClassVar = {
        KNAME_FEATS: lambda args: _cat(args, 2),
        KNAME_DIVS: lambda args: _cat(args, 1),
    }

    def __init__(self, content: List[GeneralizedFeatures]) -> None:
        self.reset(content)
        self.names = None

    def keys(self) -> frozenset:
        return self.generator_keys.union(frozenset([KNAME_NAMES]))

    def reset(self, content: Iterable[GeneralizedFeatures]) -> None:
        content = list(content)
        self.source = {key: zip(*[member[key] for member in content]) for key in self.generator_keys}
        self._queues = {key: SimpleQueue() for key in self.generator_keys}

    def _populate(self, key: Optional[str] = None, exception: bool = True) -> None:
        for k in (self.generator_keys if key is None else frozenset([key])):
            try:
                self._queues[k].put(self.joiners[k](next(self.source[k])))
            except StopIteration:
                if exception:
                    raise

    def _makegenerator(self, key: str) -> Generator[Any, None, None]:
        while True:
            try:
                item = self._queues[key].get(block=False)
            except Empty:
                self._populate(key=key, exception=False)
                try:
                    item = self._queues[key].get(block=False)
                except Empty:
                    return
            yield item

    def __getitem__(self, key: str):
        if key in self.generator_keys:
            return self._makegenerator(key)
        if key == KNAME_NAMES:
            return self.names
        raise KeyError("Invalid key; valid keys are {}".format(self.keys()))


# --------------------------------------------------------------------------------------
# id features
# --------------------------------------------------------------------------------------
def _label_groups(n_fg_sites: int, constraints: Constraints) -> List[frozenset]:
    """Constraint groups plus singletons, in the reference's label order.

    The reference enumerates ``sorted(reduce_constraint_sets(groups))`` (featlinearmap.py:600-602);
    ``sorted`` never reorders disjoint frozensets, so the order is the iteration order of the set
    returned by ``reduce_constraint_sets`` for a set built the way the reference builds it (deep
    copy, then ``union`` with the singletons).  ``tests/test_host_logic.py`` pins the resulting
    label vectors against the reference on random inputs.
    """
    key = (n_fg_sites, frozenset(frozenset(g) for g in constraints))
    if key not in _LABEL_CACHE:
        if len(_LABEL_CACHE) > 32:
            _LABEL_CACHE.clear()
        groups = deepcopy(constraints)
        groups = groups.union(frozenset([x]) for x in range(n_fg_sites))
        _LABEL_CACHE[key] = sorted(reduce_constraint_sets(groups))
    return _LABEL_CACHE[key]


_LABEL_CACHE: Dict[Any, List[frozenset]] = {}


def id_feat(points, cmap: LinearMap, constraints: Constraints, return_ids: bool = False):
    """One-hot constraint-group label of every fine-grained site.

    ``return_ids=True`` returns the ``int32[n_fg]`` label vector.  Otherwise the reference's
    feature dict: one ``(n_frames, n_fg, n_labels)`` float32 array shared by all beads and zero
    divergences ``(n_frames, n_labels, 3)``.
    """
    ordered = _label_groups(cmap.n_fg_sites, constraints)
    ids = np.zeros(cmap.n_fg_sites, dtype=np.int32)
    for label, members in enumerate(ordered):
        ids[list(members)] = label
    if return_ids:
        return ids
    n_frames, n_types = points.shape[0], len(ordered)
    feats = np.zeros((n_frames, cmap.n_fg_sites, n_types), dtype=np.float32)
    feats[:, np.arange(cmap.n_fg_sites), ids] = 1
    divs = np.zeros((n_frames, n_types, cmap.n_dim), dtype=np.float32)
    return {"feats": [feats] * cmap.n_cg_sites, "divs": [divs] * cmap.n_cg_sites, "names": None}


def multifeaturize(featurizers: List[GeneralizedFeaturizer]) -> GeneralizedFeaturizer:
    """Closure form of :class:`Multifeaturize`."""

    def composite(copoints, coord_map: LinearMap, constraints: Constraints) -> GeneralizedFeatures:
        return FeatZipper(content=[f(copoints, coord_map, constraints) for f in featurizers])

    composite.featurizers = featurizers  # type: ignore[attr-defined]
    return composite


class Multifeaturize:
    """Combine featurizers into one featurizer (outputs joined lazily by ``FeatZipper``)."""

    def __init__(self, featurizers: Iterable[GeneralizedFeaturizer]) -> None:
        self.featurizers = featurizers

    def __call__(self, *args, **kwargs) -> GeneralizedFeatures:
        return FeatZipper(content=[f(*args, **kwargs) for f in self.featurizers])

    def __str__(self) -> str:
        lines = [f"{self.__class__} instance:"]
        for ind, func in enumerate(self.featurizers):
            lines.append(f"Callable {ind}:")
            lines.extend("    " + ln for ln in str(func).split("\n"))
        return "\n".join(lines)

    def __repr__(self) -> str:
        parts = [f"{self.__class__}():"]
        for ind, func in enumerate(self.featurizers):
            parts += [f"C{ind}:", repr(func)]
        return " ".join(parts)


# --------------------------------------------------------------------------------------
# recognising fusable featurizers
# --------------------------------------------------------------------------------------
class _Plan:
    """Feature layout of a fusable featurizer: blocks in user order, each ("id") or ("gb", spec)."""

    def __init__(self, blocks: List[Tuple[str, Optional[GbSpec]]]) -> None:
        self.blocks = blocks
        gbs = [b[1] for b in blocks if b[0] == "gb"]
        self.spec: Optional[GbSpec] = gbs[0] if gbs else None
        self.has_id = any(b[0] == "id" for b in blocks)


def _as_block(f) -> Optional[Tuple[str, Optional[GbSpec]]]:
    if f is id_feat:
        return ("id", None)
    func, args, kwargs = f, (), {}
    if isinstance(f, Curry):
        func, args, kwargs = f.func, f.args, f.kwargs
    elif isinstance(f, functools.partial):
        func, args, kwargs = f.func, f.args, f.keywords
    if func is gb_feat and not args and "outer" in kwargs:
        allowed = {"outer", "inner", "n_basis", "width", "dist_power", "batch_size", "lazy", "div_method",
                   "drop_last_channel"}
        if set(kwargs) <= allowed:
            keys = ("outer", "inner", "n_basis", "width", "dist_power", "drop_last_channel")
            return ("gb", GbSpec(**{k: kwargs[k] for k in keys if k in kwargs}))
    return None


def _fusable(featurizer) -> Optional[_Plan]:
    members = getattr(featurizer, "featurizers", None)
    blocks = [_as_block(f) for f in (list(members) if members is not None else [featurizer])]
    if not blocks or any(b is None for b in blocks):
        return None
    kinds = [b[0] for b in blocks]  # type: ignore[index]
    if kinds.count("id") > 1 or kinds.count("gb") > 1:
        return None
    return _Plan(blocks)  # type: ignore[arg-type]


class _FusedContext:
    """Device-side description (label groups, bead rows, gb parameters) shared by the fused kernels."""

    def __init__(self, coord_map: LinearMap, constraints: Constraints, plan: _Plan) -> None:
        n_fg = coord_map.n_fg_sites
        self.plan = plan
        self.labels = id_feat(None, coord_map, constraints, return_ids=True)
        self.n_groups = int(self.labels.max()) + 1
        spec = plan.spec
        self.n_channels = spec.n_channels(self.n_groups) if spec is not None else 0
        self.nb = spec.n_basis if spec is not None else 1
        self.width = float(spec.width) if spec is not None else 1.0
        self.clip = float(spec.clip) if spec is not None else 1e-3
        centers = spec.centers() if spec is not None else np.zeros(1)
        ptr_, sites = _engine.csr_from_labels(self.labels, self.n_groups)
        cm = np.asarray(coord_map.standard_matrix, dtype=np.float64)
        rows, cols = np.nonzero(cm)
        bptr = np.zeros(coord_map.n_cg_sites + 1, dtype=np.int32)
        np.cumsum(np.bincount(rows, minlength=coord_map.n_cg_sites), out=bptr[1:])
        self.n_cg, self.n_fg = coord_map.n_cg_sites, n_fg
        self.n_feat_kernel = self.n_groups + self.nb * self.n_channels
        self.d_grp_ptr, self.d_grp_sites = _engine.dev_i32(ptr_), _engine.dev_i32(sites)
        self.d_bead_ptr, self.d_bead_sites = _engine.dev_i32(bptr), _engine.dev_i32(cols)
        self.d_bead_w = _engine.dev_f64(cm[rows, cols])
        self.d_centers = _engine.dev_f64(centers)
        self.d_labels = _engine.dev_i32(self.labels)
        # kernel feature order is [id | gb]; the user's order / subset is a column selection
        sel: List[np.ndarray] = []
        for kind, _ in plan.blocks:
            if kind == "id":
                sel.append(np.arange(self.n_groups))
            else:
                sel.append(self.n_groups + np.arange(self.nb * self.n_channels))
        self.columns = np.concatenate(sel)

    def _common(self):
        p = _engine.ptr
        return (p(self.d_grp_ptr), p(self.d_grp_sites), self.n_groups, self.n_channels, p(self.d_bead_ptr),
                p(self.d_bead_sites), p(self.d_bead_w), self.n_cg, p(self.d_centers), self.nb, self.width, self.clip)

    def grams(self, coords: _engine.Frames, forces: _engine.Frames, kbt: float, on_device: bool = False,
              weights: Optional[torch.Tensor] = None):
        """All-reduced per-bead Grams in the user's feature order, ``(n_cg, n_feat, n_feat)`` float64
        (numpy, or a CUDA tensor with ``on_device``).  ``weights``: per-frame weights
        (``_engine.frame_weights_dev``); weighted Grams run on the FP64 DMMA kernels only."""
        nf = self.n_feat_kernel
        gram = torch.zeros((self.n_cg, nf, nf), dtype=torch.float64, device=_engine.device())
        for t0, c, f in _engine.paired_pieces(coords, forces):
            if c.dtype != f.dtype:
                c, f = c.to(torch.float64), f.to(torch.float64)
            if weights is not None:
                need = int(_lib.lib().agf_gram_feat_workspace_bytes(self.n_groups, self.n_channels, self.nb,
                                                                    self.n_cg, c.shape[0]))
                ws = _engine.workspace(need)
                _lib.call("agf_gram_feat_ws_weighted", _engine.ptr(c), _engine.ptr(f), _engine.dtype_code(c),
                          c.shape[0], self.n_fg, *self._common(), float(kbt), _engine.ptr(gram), _engine.ptr(ws),
                          C.c_size_t(ws.numel()), _engine.ptr(weights[t0 : t0 + c.shape[0]]), _engine.stream_ptr())
                continue
            need_i8 = 0
            if _engine._GRAM_I8[0] and nf > 97 and c.shape[0] >= _engine._GRAM_I8T_MIN_FRAMES:
                need_i8 = int(_lib.lib().agf_gram_feat_i8_workspace_bytes(self.n_groups, self.n_channels, self.nb,
                                                                          self.n_cg, c.shape[0]))
            if need_i8 > 0:  # regression rows -> int8 digit planes -> batched tcgen05 SYRK (csrc/featgram.cu)
                ws = _engine.workspace(need_i8)
                _lib.call("agf_gram_feat_i8", _engine.ptr(c), _engine.ptr(f), _engine.dtype_code(c), c.shape[0],
                          self.n_fg, *self._common(), float(kbt), _engine.ptr(gram), _engine.ptr(ws),
                          C.c_size_t(ws.numel()), _engine.stream_ptr())
                continue
            need = int(_lib.lib().agf_gram_feat_workspace_bytes(self.n_groups, self.n_channels, self.nb, self.n_cg,
                                                                c.shape[0]))
            ws = _engine.workspace(need)
            _lib.call("agf_gram_feat_ws", _engine.ptr(c), _engine.ptr(f), _engine.dtype_code(c), c.shape[0], self.n_fg,
                      *self._common(), float(kbt), _engine.ptr(gram), _engine.ptr(ws), C.c_size_t(ws.numel()),
                      _engine.stream_ptr())
        _engine.allreduce_sum_(gram)
        _lib.call("agf_symmetrize_batch", _engine.ptr(gram), nf, self.n_cg, _engine.stream_ptr())
        if on_device:
            if np.array_equal(self.columns, np.arange(nf)):
                return gram
            sel = torch.as_tensor(self.columns, device=gram.device)
            return gram[:, sel][:, :, sel].contiguous()
        host = _engine.to_host(gram)
        return host[:, self.columns][:, :, self.columns]

    def constraint_rows(self, coords: _engine.Frames, bead: int, frame_indices: np.ndarray, on_device: bool = False):
        """``(n_sel * n_cg, n_feat)`` equality rows of one bead (user feature order); numpy, or a CUDA tensor
        with ``on_device`` (nothing synchronises then)."""
        idx = np.asarray(frame_indices, dtype=np.int64)
        n_sel = int(idx.size)
        picked = coords.gather(idx)
        sel = torch.arange(n_sel, dtype=torch.int64, device=_engine.device())
        rows = torch.empty((n_sel, self.n_cg, self.n_feat_kernel), dtype=torch.float64, device=_engine.device())
        _lib.call("agf_feat_rows", _engine.ptr(picked), _engine.dtype_code(picked), self.n_fg, _engine.ptr(sel), n_sel,
                  int(bead), _engine.ptr(self.d_labels), *self._common(), _engine.ptr(rows), _engine.stream_ptr())
        if on_device:
            rows = rows.reshape(n_sel * self.n_cg, self.n_feat_kernel)
            if np.array_equal(self.columns, np.arange(self.n_feat_kernel)):
                return rows
            return rows[:, _engine._dev_cached(np.ascontiguousarray(self.columns, dtype=np.int64))]
        return _engine.to_host(rows).reshape(n_sel * self.n_cg, self.n_feat_kernel)[:, self.columns]

    def apply(self, coords: _engine.Frames, forces: _engine.Frames, coefs: np.ndarray, want_sumsq: bool = False):
        """Mapped forces of the fitted map; ``coefs`` is ``(n_cg, n_feat)`` in the user's order."""
        full = np.zeros((self.n_cg, self.n_feat_kernel))
        full[:, self.columns] = coefs
        d_coef = _engine.dev_f64(full)
        out = torch.empty((coords.n_frames, self.n_cg, 3), dtype=torch.float64, device=_engine.device())
        sumsq = torch.zeros(1, dtype=torch.float64, device=_engine.device()) if want_sumsq else None
        for t0, c, f in _engine.paired_pieces(coords, forces):
            if c.dtype != f.dtype:
                c, f = c.to(torch.float64), f.to(torch.float64)
            o = out[t0 : t0 + c.shape[0]]
            _lib.call("agf_feat_apply", _engine.ptr(c), _engine.ptr(f), _engine.dtype_code(c), c.shape[0], self.n_fg,
                      *self._common(), _engine.ptr(d_coef), _engine.ptr(o), _engine.dtype_code(o), _engine.ptr(sumsq),
                      _engine.stream_ptr())
        return out, sumsq


class FeatCLAMap(CLAMap):
    """``CLAMap`` of a fused featurised fit: ``__call__`` runs ``agf_feat_apply``; ``scale`` /
    ``trans`` (materialising per-frame weights, as the reference does) stay available."""

    def __init__(self, ctx: _FusedContext, coefs: np.ndarray, scale: Callable, trans: Callable, **kwargs) -> None:
        super().__init__(scale=scale, trans=trans, n_fg_sites=ctx.n_fg, n_cg_sites=ctx.n_cg, zeroes_check=False,
                         **kwargs)
        self._ctx = ctx
        self._coefs = np.asarray(coefs, dtype=np.float64)

    def __call__(self, points, copoints):
        f, c = _engine.Frames(points), _engine.Frames(copoints)
        out, _ = self._ctx.apply(c, f, self._coefs)
        return _engine.to_host(out) if f.on_host else out


# --------------------------------------------------------------------------------------
# the fit
# --------------------------------------------------------------------------------------
def _pick_frames(n_total: int, n_frames: int, constraint_frames) -> np.ndarray:
    """Frames used for the equality rows of one bead (reference: unseeded draw, :445)."""
    if constraint_frames is None:
        return default_rng().choice(n_total, size=n_frames, replace=False)
    if callable(constraint_frames):
        return np.asarray(constraint_frames(n_total, n_frames))
    return np.asarray(constraint_frames)


class _ConstraintFrames:
    """Per-bead choice of the frames that carry the equality rows, made ONCE for all ranks.

    Under ``frame_sharding`` every rank holds a slice of the frames; the frame indices are GLOBAL
    (rank r's frames follow those of ranks < r).  Rank 0 draws (or takes the caller's indices), the
    choice is broadcast, every rank evaluates the rows of the frames it owns and the rows are summed
    across ranks -- so all ranks solve the same QP.  Without sharding this is ``_pick_frames``."""

    def __init__(self, n_local: int, n_beads: int, n_frames: int, constraint_frames) -> None:
        self.n_local = int(n_local)
        counts = np.asarray([c[0] for c in _engine.allgather_host(np.asarray([float(n_local)]))], dtype=np.int64)
        rank = _engine.shard_rank()
        self.offset = int(counts[:rank].sum())
        n_total = int(counts.sum())
        picks = np.stack([np.asarray(_pick_frames(n_total, n_frames, constraint_frames), dtype=np.int64)
                          for _ in range(n_beads)])
        self.picks = _engine.broadcast_host(picks.astype(np.float64)).astype(np.int64)

    def rows(self, bead: int, evaluate: Callable[[np.ndarray], np.ndarray], n_cg: int) -> np.ndarray:
        """``evaluate(local frame indices) -> (n_sel_local * n_cg, n_feat)``; returns the rows of all
        chosen frames in the order of the choice."""
        glob = self.picks[bead]
        if not _engine.sharded():
            return evaluate(glob)
        mine = np.nonzero((glob >= self.offset) & (glob < self.offset + self.n_local))[0]
        local = evaluate(glob[mine] - self.offset) if mine.size else None
        n_feat = np.asarray([float(local.shape[1]) if local is not None else 0.0])
        n_feat = int(max(v[0] for v in _engine.allgather_host(n_feat)))
        full = np.zeros((glob.size, n_cg, n_feat))
        if local is not None:
            full[mine] = local.reshape(mine.size, n_cg, n_feat)
        return _engine.allreduce_host_sum(full).reshape(glob.size * n_cg, n_feat)


def qp_feat_linear_map(
    traj: Trajectory,
    coord_map: LinearMap,
    featurizer: Featurizer,
    kbt: float,
    n_constraint_frames: int = 20,
    constraints: Union[None, Constraints] = None,
    sparse: bool = True,
    solver_args: SolverOptions = DEFAULT_SOLVER_OPTIONS,
    l2_regularization: float = 1e1,
    constraint_frames=None,
    frame_weights=None,
) -> CLAFTMap:
    """Force map linear in user features, minimising the mean squared mapped force.

    Arguments as the reference (``featlinearmap.py:249-259``).  ``l2_regularization`` penalises the
    coefficient vector (``+ l2 * I``, not the linear map's ``l2 * C'C``); the objective is the raw
    frame sum.  Extra keyword ``constraint_frames`` (array of frame indices, or callable
    ``(n_total, n) -> indices``) replaces the reference's unseeded random choice of the frames on
    which the bead-orthogonality constraints are imposed.

    ``frame_weights`` (extension): one non-negative weight per frame (numpy or CUDA tensor; under
    ``frame_sharding`` this rank's slice).  Every regression row of frame t (the ``kbt`` divergence term
    included) is multiplied by ``sqrt(w_t)``, so ``P_c = sum_t w_t v_t v_t^T (+ l2 I)``.  The frames that
    carry the equality rows are chosen as without weights: a constraint holds on a configuration whatever
    its weight.
    """
    if constraints is None:
        constraints = set()
    warn_if_solver_ignored(solver_args)
    weights = _engine.frame_weights_dev(frame_weights, traj.forces.shape[0])
    plan = _fusable(featurizer)
    if plan is not None:
        return _fit_fused(traj, coord_map, featurizer, plan, kbt, n_constraint_frames, constraints, solver_args,
                          l2_regularization, constraint_frames, weights)
    return _fit_generic(traj, coord_map, featurizer, kbt, n_constraint_frames, constraints, sparse, solver_args,
                        l2_regularization, constraint_frames, weights)


def _fit_fused(traj, coord_map, featurizer, plan, kbt, n_constraint_frames, constraints, solver_args,
               l2_regularization, constraint_frames, weights=None) -> CLAFTMap:
    ctx = _FusedContext(coord_map, constraints, plan)
    coords, forces = _engine.Frames(traj.coords), _engine.Frames(traj.forces)
    backend = dict(solver_args or {}).get("backend", "exact")
    on_device = backend == "exact" and ctx.columns.size >= _DEVICE_SOLVE_MIN
    grams = ctx.grams(coords, forces, kbt, on_device=on_device, weights=weights)  # large problems never leave the device
    n_feat = grams.shape[1]
    coefs = []
    chosen = _ConstraintFrames(coords.n_frames, coord_map.n_cg_sites, n_constraint_frames, constraint_frames)
    n_cg = coord_map.n_cg_sites
    if on_device:
        # all beads at once: equality rows stay on the device (single GPU), one batched Cholesky / Schur solve,
        # one read for the checks -- the per-bead loop below is the fallback when any bead's solve declines
        if _engine.sharded():
            # every rank evaluates the rows of the chosen frames it owns, for all beads, into one zero-filled
            # device array: ONE sum over the ranks instead of two host collectives per bead
            n_sel_all = int(chosen.picks.shape[1])
            a_dev = torch.zeros((n_cg, n_sel_all, n_cg, n_feat), dtype=torch.float64, device=grams.device)
            for b in range(n_cg):
                glob = chosen.picks[b]
                mine = np.nonzero((glob >= chosen.offset) & (glob < chosen.offset + chosen.n_local))[0]
                if mine.size:
                    local = ctx.constraint_rows(coords, b, glob[mine] - chosen.offset, on_device=True)
                    a_dev[b, torch.as_tensor(mine, device=grams.device)] = local.reshape(mine.size, n_cg, n_feat)
            a_dev = _engine.allreduce_sum_(a_dev).reshape(n_cg, n_sel_all * n_cg, n_feat)
            a_all = list(a_dev)
        else:
            a_all = [chosen.rows(b, lambda idx, b=b: ctx.constraint_rows(coords, b, idx, on_device=True), n_cg)
                     for b in range(n_cg)]
        if len({tuple(a.shape) for a in a_all}) == 1:
            a_dev = torch.stack(list(a_all))
            n_sel = a_dev.shape[1] // n_cg
            rhs = torch.zeros((n_cg, n_sel, n_cg), dtype=torch.float64, device=grams.device)
            rhs[torch.arange(n_cg), :, torch.arange(n_cg)] = 1.0
            qp_all = grams.clone()
            if l2_regularization > 0:
                qp_all.diagonal(dim1=1, dim2=2).add_(l2_regularization)
            sol = solve_equality_qp_device_batched(qp_all, a_dev, rhs.reshape(n_cg, n_sel * n_cg))
            if sol is not None:
                coefs = [sol[b] for b in range(n_cg)]
    for bead in range(n_cg if not coefs else 0):
        frames = chosen.picks[bead]
        a_mat = chosen.rows(bead, lambda idx, b=bead: ctx.constraint_rows(coords, b, idx), coord_map.n_cg_sites)
        target = np.zeros((len(frames), coord_map.n_cg_sites))
        target[:, bead] = 1
        params = None
        if on_device:
            qp_dev = grams[bead].clone()
            if l2_regularization > 0:
                qp_dev.diagonal().add_(l2_regularization)
            params = solve_equality_qp_device(qp_dev, a_mat, target.reshape(-1))
            qp_mat = None if params is not None else _engine.to_host(qp_dev)
        else:
            qp_mat = grams[bead]
            if l2_regularization > 0:
                qp_mat = qp_mat + l2_regularization * np.eye(n_feat)
        if params is None:
            params = solve(qp_mat, a_mat, target.reshape(-1), solver_args)
        if params is None:
            raise ValueError("Map optimization failed.")
        coefs.append(params)
    scale_f, trans_f = _weight_functions(featurizer, coefs, coord_map, constraints)
    force_map = FeatCLAMap(ctx, np.stack(coefs), scale_f, trans_f,
                           tags={"feat_names": None, "coef_list": coefs})
    return CLAFTMap(coord_map=coord_map, force_map=force_map)


def _fit_generic(traj, coord_map, featurizer, kbt, n_constraint_frames, constraints, sparse, solver_args,
                 l2_regularization, constraint_frames, weights=None) -> CLAFTMap:
    dev = _engine.device()
    feat_results = featurizer(traj.coords, coord_map, constraints)
    feats, divs, names = (feat_results[k] for k in (KNAME_FEATS, KNAME_DIVS, KNAME_NAMES))
    forces = _engine.Frames(traj.forces).resident().to(torch.float64)
    cm = torch.as_tensor(np.asarray(coord_map.standard_matrix, dtype=np.float64), device=dev)
    coefs = []
    chosen = _ConstraintFrames(forces.shape[0], coord_map.n_cg_sites, n_constraint_frames, constraint_frames)
    for bead, (feat, div) in enumerate(zip(feats, divs)):
        phi = torch.as_tensor(feat).to(device=dev, dtype=torch.float64)
        dv = torch.as_tensor(div).to(device=dev, dtype=torch.float64)
        frames = chosen.picks[bead]

        def rows_of(idx, phi=phi):
            mult = torch.einsum("ca,saf->scf", cm, phi[torch.as_tensor(np.asarray(idx), device=dev)])
            return _engine.to_host(mult.reshape(-1, mult.shape[-1]))

        a_mat = chosen.rows(bead, rows_of, coord_map.n_cg_sites)
        target = np.zeros((len(frames), coord_map.n_cg_sites))
        target[:, bead] = 1
        rows = torch.einsum("tad,taf->tdf", forces, phi) + kbt * dv.transpose(1, 2)
        if weights is not None:
            rows = rows * weights.sqrt()[:, None, None]
        reg = rows.reshape(-1, rows.shape[2])
        gram = reg.T @ reg
        _engine.allreduce_sum_(gram)
        qp_mat = _engine.to_host(gram)
        if l2_regularization > 0:
            qp_mat = qp_mat + l2_regularization * np.eye(qp_mat.shape[0])
        a_use = ss.csc_matrix(a_mat) if sparse else a_mat
        params = solve(qp_mat, a_use, target.reshape(-1), solver_args)
        if params is None:
            raise ValueError("Map optimization failed.")
        coefs.append(params)
    force_map = _feat_linear_mapping(featurizer=featurizer, coefs=coefs, mapping=coord_map, constraints=constraints,
                                     tags={"feat_names": names, "coef_list": coefs})
    return CLAFTMap(coord_map=coord_map, force_map=force_map)


def _weight_functions(featurizer, coefs, mapping, constraints):
    def scale_f(copoints):
        feats = featurizer(copoints, mapping, constraints)["feats"]
        return np.stack([np.einsum("...ij,j->...i", np.asarray(f), c) for f, c in zip(feats, coefs)], axis=1)

    def trans_f(copoints):
        divs = featurizer(copoints, mapping, constraints)["divs"]
        return np.stack([np.einsum("tij,i->tj", np.asarray(d), c) for d, c in zip(divs, coefs)], axis=1)

    return scale_f, trans_f


def _constr_arrays(features, cg_ind: int, coord_map: LinearMap, n_frames: int, sparse: bool = True):
    """Equality rows ``A`` and targets ``b`` for one bead from materialised features
    (``(n_cg*n_frames, n_feat)``, ``(n_cg*n_frames,)``); frames drawn at random."""
    idx = default_rng().choice(len(features), size=n_frames, replace=False)
    mult = np.einsum("ca,...af->...cf", coord_map.standard_matrix, np.asarray(features)[idx])
    target = np.zeros((n_frames, coord_map.n_cg_sites))
    target[:, cg_ind] = 1
    mult = mult.reshape((-1, mult.shape[-1]))
    return (ss.csc_matrix(mult) if sparse else mult, target.reshape(-1))


def _feat_linear_mapping(featurizer, coefs, mapping: LinearMap, constraints: Constraints, **kwargs) -> CLAMap:
    """``CLAMap`` whose per-frame weights are ``features . coefs`` (generic featurizers)."""
    scale_f, trans_f = _weight_functions(featurizer, coefs, mapping, constraints)
    return CLAMap(scale=scale_f, trans=trans_f, n_fg_sites=mapping.n_fg_sites, zeroes_check=True, **kwargs)
