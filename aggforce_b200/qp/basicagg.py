"""Uniform (0/1) force map that respects constraints; pure index logic on the host.

Drop-in for the reference's ``src/aggforce/qp/basicagg.py:11-62``.
"""
from __future__ import annotations

import hashlib
from typing import Union

import numpy as np

from ..constraints import Constraints, merged_groups
from ..map import LinearMap, SeperableTMap
from ..trajectory import ForcesTrajectory


def constraint_aware_uni_map(
    traj: ForcesTrajectory,  # noqa: ARG001
    coord_map: LinearMap,
    constraints: Union[None, Constraints] = None,
    frame_weights=None,  # noqa: ARG001
) -> SeperableTMap:
    """Each bead sums, unweighted, the forces of its own sites and of every site constrained
    (transitively) to one of them.  ``traj`` is ignored, and so is ``frame_weights``: the map reads no
    frames (it is accepted so that ``project_forces(..., frame_weights=w)`` reports the weighted residual
    of this map too)."""
    matrix = np.asarray(coord_map.standard_matrix)
    try:  # pure index bookkeeping: memoised on the content of its two inputs (a fresh matrix per call)
        key = (matrix.shape, str(matrix.dtype), hashlib.blake2b(np.ascontiguousarray(matrix).tobytes(), digest_size=16).digest(),
               frozenset(() if constraints is None else constraints))
    except TypeError:
        key = None
    if key is not None and key in _UNI_CACHE:
        return SeperableTMap(coord_map=coord_map, force_map=LinearMap(_UNI_CACHE[key].copy()))
    groups = merged_groups(set() if constraints is None else constraints)
    group_of = {site: gi for gi, g in enumerate(groups) for site in g}  # merged groups are disjoint
    out = np.zeros_like(matrix)
    for bead, row in enumerate(matrix):
        members = set(np.nonzero(row)[0].tolist())
        for gi in {group_of[m] for m in members if m in group_of}:
            members.update(groups[gi])
        out[bead, sorted(members)] = 1.0
    if key is not None:
        if len(_UNI_CACHE) > 32:
            _UNI_CACHE.clear()
        _UNI_CACHE[key] = out.copy()
    return SeperableTMap(coord_map=coord_map, force_map=LinearMap(out))


_UNI_CACHE: dict = {}
