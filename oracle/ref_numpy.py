"""Float64 numpy restatement of the aggforce hot path (TEST INFRASTRUCTURE, not product).

Every function cites the reference lines (relative to /root/reference) it restates.
All arithmetic is float64 regardless of input dtype: this is the arbiter the CUDA
kernels are compared against (SURVEY.md section 8c; Q4, Q10).

Nothing here is imported by ``aggforce_b200``.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence, Set, Tuple

import numpy as np

__all__ = [
    "pair_distance_sd",
    "pair_distance_moments",
    "guess_pairwise_constraints",
    "guess_pairwise_constraints_literal",
    "merge_constraint_groups",
    "group_columns",
    "bond_constraint_matrix",
    "gram_linear",
    "l2_linear_term",
    "solve_equality_qp",
    "qp_linear_weights",
    "uni_map_matrix",
    "apply_map",
    "apply_map_nan_protocol",
    "force_smoothness",
    "canonical_labels",
    "gb_centers",
    "gb_features",
    "gb_divergence_fd",
    "feat_regressor_rows",
    "feat_gram",
    "feat_constraint_rows",
    "feat_map_apply",
    "gauss_augment",
    "gauss_log_gradient",
    "sq_gaussian_forces",
    "mscg_ip",
    "random_force_proj",
    "random_residual_shift",
]


# --------------------------------------------------------------------------------------
# (c) constraint detection
# --------------------------------------------------------------------------------------
def pair_distance_sd(xyz: np.ndarray, cross_xyz: Optional[np.ndarray] = None) -> np.ndarray:
    """Population standard deviation over frames of every pair distance.

    Restates src/aggforce/util.py:64-70 (displacement ``xyz[:,None,:,:]-other[:,:,None,:]``
    then an l2 norm) followed by src/aggforce/constraints/constfinder.py:47
    (``sqrt(var(axis=0))``, ddof=0), evaluated in float64 (SURVEY Q10).

    Returns shape (n_other, n) with ``out[i, j]`` = sd of |xyz[:, j] - other[:, i]|.
    Frames are processed in blocks so the (T, n, n, 3) temporary is never formed; the
    two-pass mean/variance is numerically equivalent to numpy's ``var``.
    """
    x = np.asarray(xyz, dtype=np.float64)
    o = x if cross_xyz is None else np.asarray(cross_xyz, dtype=np.float64)
    n_frames = x.shape[0]
    n, m = x.shape[1], o.shape[1]
    block = max(1, int(4e6 // max(1, n * m)))
    total = np.zeros((m, n))
    for s in range(0, n_frames, block):
        d = x[s : s + block, None, :, :] - o[s : s + block, :, None, :]
        total += np.sqrt((d * d).sum(-1)).sum(0)
    mean = total / n_frames
    m2 = np.zeros((m, n))
    for s in range(0, n_frames, block):
        d = x[s : s + block, None, :, :] - o[s : s + block, :, None, :]
        dev = np.sqrt((d * d).sum(-1)) - mean
        m2 += (dev * dev).sum(0)
    return np.sqrt(m2 / n_frames)


def pair_distance_moments(xyz: np.ndarray, other: Optional[np.ndarray], pairs: np.ndarray,
                          shift: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Per-pair shifted moments ``(sum_t e_t, sum_t e_t**2)`` with ``e_t = d_t - shift[p]`` and
    ``d_t = |xyz[t, j] - other[t, i]|`` for ``pairs[p] = (i over other, j over xyz)``, in float64.

    ``other=None`` is the self case.  This is what kernel (c) accumulates for a pair list; with it
    ``pair_distance_sd`` of a listed pair is ``sqrt((s2 - s1**2 / T) / T)``."""
    x = np.asarray(xyz, dtype=np.float64)
    o = x if other is None else np.asarray(other, dtype=np.float64)
    p = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    c = np.asarray(shift, dtype=np.float64).reshape(-1)
    s1, s2 = np.zeros(len(p)), np.zeros(len(p))
    block = max(1, int(4e6 // max(1, 3 * len(p))))
    for s in range(0, x.shape[0], block):
        d = x[s : s + block, p[:, 1]] - o[s : s + block, p[:, 0]]
        e = np.sqrt((d * d).sum(-1)) - c
        s1 += e.sum(0)
        s2 += (e * e).sum(0)
    return s1, s2


def guess_pairwise_constraints(
    xyz: np.ndarray, cross_xyz: Optional[np.ndarray] = None, threshold: float = 1e-3
) -> set:
    """Restates src/aggforce/constraints/constfinder.py:46-57.

    Self mode: diagonal forced to ``2*threshold`` (:51), strict ``<`` (:52), unordered
    frozenset pairs (:53).  Cross mode: ordered ``(i over cross_xyz, j over xyz)`` tuples
    (:56-57).  NaN distances never compare ``<`` so NaN coordinates yield no pair (Q13).
    """
    sds = pair_distance_sd(xyz, cross_xyz)
    if cross_xyz is None:
        np.fill_diagonal(sds, 2 * threshold)
        ii, jj = np.nonzero(sds < threshold)
        return {frozenset((int(i), int(j))) for i, j in zip(ii, jj)}
    ii, jj = np.nonzero(sds < threshold)
    return {(int(i), int(j)) for i, j in zip(ii, jj)}


def guess_pairwise_constraints_literal(xyz: np.ndarray, threshold: float = 1e-3) -> set:
    """The reference's formula AT THE REFERENCE'S COST: one materialised (T, n, n, 3)
    displacement array in the INPUT dtype, its norm, ``np.var`` over frames
    (util.py:65,70; constfinder.py:46-53).  Used only as the timed CPU baseline; small T."""
    x = np.asarray(xyz)
    dists = np.linalg.norm(x[:, None, :, :] - x[:, :, None, :], axis=-1)
    sds = np.sqrt(np.var(dists, axis=0))
    np.fill_diagonal(sds, threshold * 2)
    ii, jj = np.nonzero(sds < threshold)
    return {frozenset((int(i), int(j))) for i, j in zip(ii, jj)}


# --------------------------------------------------------------------------------------
# constraint-group algebra
# --------------------------------------------------------------------------------------
def merge_constraint_groups(constraints: Iterable[Iterable[int]]) -> List[Tuple[int, ...]]:
    """Disjoint groups obtained by transitively merging overlapping constraint sets.

    Same partition as src/aggforce/constraints/tools.py:7-77 (probe, SURVEY Q15), computed
    with a union-find instead of the reference's repeated flood; returned as sorted tuples
    ordered by smallest member, which is an ordering the reference never relies on for the
    linear path (column order comes from ``group_columns`` below).
    """
    parent: Dict[int, int] = {}

    def find(a: int) -> int:
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a

    for grp in constraints:
        members = [int(v) for v in grp]
        for v in members:
            parent.setdefault(v, v)
        for v in members[1:]:
            ra, rb = find(members[0]), find(v)
            if ra != rb:
                parent[max(ra, rb)] = min(ra, rb)
    comps: Dict[int, List[int]] = {}
    for v in parent:
        comps.setdefault(find(v), []).append(v)
    return sorted((tuple(sorted(v)) for v in comps.values()), key=lambda g: g[0])


def group_columns(n_sites: int, constraints: Iterable[Iterable[int]]) -> np.ndarray:
    """Reduced-column index of every fine-grained site (``int64[n_sites]``).

    Restates the column layout of src/aggforce/qp/qplinear.py:147-163: a site that is
    not a *dependent* member of a constraint group (i.e. it is unconstrained, or it is
    the smallest index -- the anchor -- of its merged group, constraints/tools.py:111-115)
    receives the next free column in increasing site order; dependent sites copy their
    anchor's column.
    """
    anchor = np.arange(n_sites)
    for grp in merge_constraint_groups(constraints):
        anchor[list(grp)] = grp[0]
    cols = np.full(n_sites, -1, dtype=np.int64)
    nxt = 0
    for s in range(n_sites):
        if anchor[s] == s:
            cols[s] = nxt
            nxt += 1
    return cols[anchor]


def bond_constraint_matrix(n_sites: int, constraints: Iterable[Iterable[int]]) -> np.ndarray:
    """One-hot (n_sites, n_red) expansion matrix C (qplinear.py:106-164)."""
    cols = group_columns(n_sites, constraints)
    mat = np.zeros((n_sites, int(cols.max()) + 1 if n_sites else 0))
    mat[np.arange(n_sites), cols] = 1.0
    return mat


# --------------------------------------------------------------------------------------
# (a) linear Gram + host QP
# --------------------------------------------------------------------------------------
def gram_linear(forces: np.ndarray, constraints: Iterable[Iterable[int]] = ()) -> np.ndarray:
    """Unnormalised second-moment matrix of the group-summed forces.

    Restates qplinear.py:66-71: rows of ``qp_form(F)`` are (frame, dim) pairs (:101-102),
    ``reg = R @ C`` sums the forces of each reduced group, ``P = reg.T @ reg``.  Never
    divided by the number of frames (Q1).
    """
    f = np.asarray(forces, dtype=np.float64)
    n_frames, n_sites, n_dim = f.shape
    cmat = bond_constraint_matrix(n_sites, constraints)
    reg = f.transpose(0, 2, 1).reshape(n_frames * n_dim, n_sites) @ cmat
    return reg.T @ reg


def l2_linear_term(n_sites: int, constraints: Iterable[Iterable[int]] = ()) -> np.ndarray:
    """``C.T @ C`` = diag(group sizes) (qplinear.py:76-77, Q3)."""
    cmat = bond_constraint_matrix(n_sites, constraints)
    return cmat.T @ cmat


def solve_equality_qp(p_mat: np.ndarray, a_mat: np.ndarray, b_vec: np.ndarray) -> np.ndarray:
    """Exact minimiser of ``0.5 x'Px`` subject to ``Ax=b``.

    Stands in for ``qpsolvers.solve_qp(P, q=0, A, b, solver="osqp")`` at
    qplinear.py:83-85 / featlinearmap.py:375-381 (qpsolvers+osqp are third-party,
    unpinned, and absent here; SURVEY 8c).  Closed form ``x = P^-1 A'(A P^-1 A')^+ b``;
    a singular ``P`` (fewer than n_red independent rows, no l2) falls back to the
    null-space method so a minimiser of the same problem is still returned.
    ``b_vec`` may be a matrix of right-hand sides (one column per problem).
    """
    p = np.asarray(p_mat, dtype=np.float64)
    a = np.asarray(a_mat, dtype=np.float64)
    b = np.asarray(b_vec, dtype=np.float64)
    try:
        chol = np.linalg.cholesky(p)
        y = np.linalg.solve(chol, a.T)
        pia = np.linalg.solve(chol.T, y)  # P^-1 A'
        s = a @ pia
        lam = np.linalg.lstsq(s, b, rcond=None)[0]
        return pia @ lam
    except np.linalg.LinAlgError:
        u, sv, vt = np.linalg.svd(a, full_matrices=True)
        rank = int((sv > sv.max() * 1e-12).sum()) if sv.size else 0
        x0 = np.linalg.lstsq(a, b, rcond=None)[0]
        z = vt[rank:].T
        if z.shape[1] == 0:
            return x0
        h = z.T @ p @ z
        w = np.linalg.lstsq(h, -(z.T @ (p @ x0)), rcond=None)[0]
        return x0 + z @ w


def qp_linear_weights(
    forces: np.ndarray,
    cmap_matrix: np.ndarray,
    constraints: Iterable[Iterable[int]] = (),
    l2_regularization: float = 0.0,
) -> np.ndarray:
    """Optimal linear force map (n_cg, n_fg), qplinear.py:64-88 with the exact solve."""
    constraints = list(constraints)
    cm = np.asarray(cmap_matrix, dtype=np.float64)
    n_cg, n_fg = cm.shape
    cmat = bond_constraint_matrix(n_fg, constraints)
    p = gram_linear(forces, constraints)
    if l2_regularization > 0.0:
        p = p + l2_regularization * (cmat.T @ cmat)
    a = cm @ cmat
    x = solve_equality_qp(p, a, np.eye(n_cg))  # columns = beads (Q2: same P, same A)
    return (cmat @ x).T


def uni_map_matrix(cmap_matrix: np.ndarray, constraints: Iterable[Iterable[int]] = ()) -> np.ndarray:
    """0/1 force map pulling in constraint partners (src/aggforce/qp/basicagg.py:46-60)."""
    cm = np.asarray(cmap_matrix)
    groups = merge_constraint_groups(constraints)
    out = np.zeros_like(cm, dtype=np.float64)
    for c, row in enumerate(cm):
        members = set(np.nonzero(row)[0].tolist())
        # basicagg.py:51-53 tests every group once against the *growing* member set; since
        # merged groups are disjoint one sweep is already the fixed point.
        for g in groups:
            if members.intersection(g):
                members.update(g)
        out[c, sorted(members)] = 1.0
    return out


# --------------------------------------------------------------------------------------
# (d) map application
# --------------------------------------------------------------------------------------
def apply_map(points: np.ndarray, matrix: np.ndarray) -> np.ndarray:
    """``out[t,c,d] = sum_f M[c,f] X[t,f,d]`` (src/aggforce/util.py:119-124), float64.

    ``matrix`` may be (n_cg, n_fg) or per-frame (T, n_cg, n_fg).
    """
    x = np.asarray(points, dtype=np.float64)
    m = np.asarray(matrix, dtype=np.float64)
    path = ["einsum_path", (0, 1)]  # the contraction order the reference requests (util.py:121)
    if m.ndim == 2:
        return np.einsum("tfd,cf->tcd", x, m, optimize=path)
    return np.einsum("tfd,tcf->tcd", x, m, optimize=path)


def apply_map_nan_protocol(points: np.ndarray, matrix: np.ndarray, atol: float = 1e-6) -> np.ndarray:
    """NaN-tolerant application, src/aggforce/map/core.py:219-240 (Q12).

    NaNs are masked to 0 and to -1; if the two results differ beyond ``atol`` (numpy
    ``allclose``, rtol 1e-5) a ValueError is raised, otherwise the 0-masked result is
    returned.  The input is not modified (the reference's ``"safe"`` flavour).
    """
    x = np.asarray(points, dtype=np.float64)
    mask = np.isnan(x)
    if not mask.any():
        return apply_map(x, matrix)
    a = apply_map(np.where(mask, 0.0, x), matrix)
    b = apply_map(np.where(mask, -1.0, x), matrix)
    if not np.allclose(a, b, atol=atol):
        raise ValueError("result depends on NaN positions")
    return a


def force_smoothness(mapped: np.ndarray) -> float:
    """``mean(x**2)`` (src/aggforce/agg.py:291-297)."""
    x = np.asarray(mapped, dtype=np.float64)
    return float((x * x).mean())


# --------------------------------------------------------------------------------------
# (b) featurised path: id features + Gaussian-binned distances
# --------------------------------------------------------------------------------------
def canonical_labels(n_sites: int, constraints: Iterable[Iterable[int]] = ()) -> np.ndarray:
    """A label per site shared inside merged constraint groups, ordered by anchor.

    The reference's label *order* is the iteration order of a Python set
    (featlinearmap.py:600-602, Q9); the math below takes the label vector as an input
    so either ordering can be fed in.  This helper gives the anchor-ordered one.
    """
    return group_columns(n_sites, constraints).astype(np.int32)


def gb_centers(inner: float, outer: float, n_basis: int, dist_power: float = 0.5) -> np.ndarray:
    """Gaussian centres: linspace in ``d**p`` mapped back (jaxfeat.py:235-236)."""
    grid = np.linspace(float(inner) ** dist_power, float(outer) ** dist_power, n_basis)
    return grid ** (1.0 / dist_power)


def _smear_matrix(n_sites: int, constraints: Iterable[Iterable[int]]) -> np.ndarray:
    """Group-mean matrix (src/aggforce/map/tools.py:96-100), built from merged groups
    exactly as jaxfeat.py:106-114 feeds it (``reduce_constraint_sets(constraints)``)."""
    mat = np.eye(n_sites)
    for g in merge_constraint_groups(constraints):
        idx = np.asarray(g)
        mat[np.ix_(idx, idx)] = 1.0 / len(g)
    return mat


def gb_features(
    points: np.ndarray,
    cmap_matrix: np.ndarray,
    constraints: Iterable[Iterable[int]],
    labels: Sequence[int],
    bead: int,
    outer: float,
    inner: float = 0.0,
    n_basis: int = 10,
    width: float = 1.0,
    dist_power: float = 0.5,
    clip: float = 1e-3,
    drop_last_channel: bool = True,
    div_method: str = "basic",
) -> Tuple[np.ndarray, np.ndarray]:
    """Literal float64 restatement of ``gb_feat`` for ONE bead.

    Returns ``(feats (T, n_fg, n_ch*n_basis), divs (T, n_ch*n_basis, 3))``.

    Steps, following src/aggforce/qp/jaxfeat.py:
      * bead position from the *unsmeared* coordinates (:104) ;
      * ``points <- smear @ points`` (:443-444) ;
      * distance of every smeared site to the bead (:445; jaxutil.py:168-179) ;
      * clipped Gaussians ``max(exp(-((d-mu)/w)^2), clip) - clip`` (:272-276) ;
      * channelise: site a's n_basis values go to columns
        ``labels[a]*n_basis + k`` of an array ``n_basis*max(labels)`` wide (:115,
        :343-349).  With ``drop_last_channel`` the block of the largest label falls off
        the end and is silently lost (Q5, [inferred] from JAX's empty-slice scatter) ;
      * divergence, ``div_method="reorder"`` (:544-565): Jacobian of
        ``sum_a g_k(d_a)`` w.r.t. every site with the bead held fixed (Q6), placed in the
        differentiated site's channel and summed over sites.  Because the smear rows sum
        to one this is ``m_ch * g_k'(d_ch) * (p_ch - R)/d_ch`` (SURVEY 8a, A11).

    A smeared site that coincides with the bead (``d = 0``: a bead atom in no constraint group
    under a slice map) has an undefined direction.  Pinned against the reference run behind the
    jax shim (``tests/golden/ref_gbfeat.npz``): with ``div_method="basic"`` (forward mode, :525-543)
    the NaN stays in the coincident site's own channel -- and vanishes when that channel is the
    dropped one; with ``div_method="reorder"`` (reverse mode, :544-565, the reference default) the
    NaN cotangent of the coincident site is multiplied by the zeros of the smear matrix in the
    transposed contraction, ``0 * NaN = NaN``, and the whole frame's divergence is NaN.
    """
    x = np.asarray(points, dtype=np.float64)
    cm = np.asarray(cmap_matrix, dtype=np.float64)
    lab = np.asarray(labels, dtype=np.int64)
    n_frames, n_sites, _ = x.shape
    n_ch_full = int(lab.max()) + 1
    n_ch = n_ch_full - 1 if drop_last_channel else n_ch_full
    mu = gb_centers(inner, outer, n_basis, dist_power)

    bead_pos = np.einsum("f,tfd->td", cm[bead], x)
    sm = _smear_matrix(n_sites, constraints)
    xs = np.einsum("af,tfd->tad", sm, x)
    disp = xs - bead_pos[:, None, :]
    dist = np.sqrt((disp * disp).sum(-1))  # (T, n_sites)
    z = (dist[..., None] - mu) / width  # (T, n_sites, n_basis)
    e = np.exp(-(z * z))
    g = np.maximum(e, clip) - clip
    gprime = np.where(e > clip, -2.0 * z / width * e, 0.0)

    feats = np.zeros((n_frames, n_sites, n_ch * n_basis))
    divs = np.zeros((n_frames, n_ch * n_basis, 3))
    with np.errstate(invalid="ignore", divide="ignore"):
        unit = disp / dist[..., None]  # NaN where a site sits on the bead (Q6)
    # d/dx_b of sum_a g_k(|sum_f sm[a,f] x_f - R|) = sum_a sm[a,b] g_k'(d_a) unit_a
    site_grad = np.zeros((n_frames, n_sites, n_basis, 3))
    for a_idx, b_idx in zip(*np.nonzero(sm)):  # explicit sum: a NaN unit vector must not leak via 0*NaN
        site_grad[:, b_idx] += sm[a_idx, b_idx] * gprime[:, a_idx, :, None] * unit[:, a_idx, None, :]
    for a in range(n_sites):
        ch = int(lab[a])
        if ch >= n_ch:
            continue
        feats[:, a, ch * n_basis : (ch + 1) * n_basis] = g[:, a, :]
        divs[:, ch * n_basis : (ch + 1) * n_basis, :] += site_grad[:, a, :, :]
    if div_method == "reorder":
        divs[(dist == 0.0).any(axis=1)] = np.nan
    elif div_method != "basic":
        raise ValueError("Unknown method for jacobian calculation.")
    return feats, divs


def gb_divergence_fd(
    points: np.ndarray,
    cmap_matrix: np.ndarray,
    constraints: Iterable[Iterable[int]],
    labels: Sequence[int],
    bead: int,
    h: float = 1e-6,
    **kw,
) -> np.ndarray:
    """Central finite-difference check of the divergence (bead position held fixed).

    Differentiates the un-channelised collapsed features w.r.t. each site, then places the
    result in that site's channel -- the "reorder" recipe of jaxfeat.py:544-565 with
    ``jacrev`` swapped for finite differences.  Small inputs only.
    """
    x = np.asarray(points, dtype=np.float64)
    cm = np.asarray(cmap_matrix, dtype=np.float64)
    lab = np.asarray(labels, dtype=np.int64)
    n_frames, n_sites, _ = x.shape
    n_basis = kw.get("n_basis", 10)
    drop = kw.get("drop_last_channel", True)
    n_ch = int(lab.max()) + (0 if drop else 1)
    mu = gb_centers(kw.get("inner", 0.0), kw["outer"], n_basis, kw.get("dist_power", 0.5))
    width, clip = kw.get("width", 1.0), kw.get("clip", 1e-3)
    sm = _smear_matrix(n_sites, constraints)
    bead_pos = np.einsum("f,tfd->td", cm[bead], x)  # constant under differentiation

    def collapsed(xx: np.ndarray) -> np.ndarray:
        xs = np.einsum("af,tfd->tad", sm, xx)
        d = np.sqrt(((xs - bead_pos[:, None, :]) ** 2).sum(-1))
        zz = (d[..., None] - mu) / width
        return (np.maximum(np.exp(-(zz * zz)), clip) - clip).sum(1)  # (T, n_basis)

    divs = np.zeros((n_frames, n_ch * n_basis, 3))
    for b in range(n_sites):
        ch = int(lab[b])
        if ch >= n_ch:
            continue
        for dim in range(3):
            xp, xm = x.copy(), x.copy()
            xp[:, b, dim] += h
            xm[:, b, dim] -= h
            divs[:, ch * n_basis : (ch + 1) * n_basis, dim] += (collapsed(xp) - collapsed(xm)) / (2 * h)
    return divs


def id_features(n_frames: int, labels: Sequence[int]) -> Tuple[np.ndarray, np.ndarray]:
    """One-hot label features and zero divergences (featlinearmap.py:621-627)."""
    lab = np.asarray(labels, dtype=np.int64)
    n_types = int(lab.max()) + 1
    feats = np.zeros((n_frames, lab.size, n_types))
    feats[:, np.arange(lab.size), lab] = 1.0
    return feats, np.zeros((n_frames, n_types, 3))


__all__.append("id_features")


def feat_regressor_rows(forces: np.ndarray, feats: np.ndarray, divs: np.ndarray, kbt: float) -> np.ndarray:
    """Rows of the featurised regression matrix, shape (3T, n_feat).

    featlinearmap.py:361-369: ``ff[t,d,f] = sum_a F[t,a,d] phi[t,a,f]``, plus
    ``kbt * div[t,f,d]`` with the axes swapped, rows ordered (frame, dim).
    """
    f = np.asarray(forces, dtype=np.float64)
    ff = np.einsum("tad,taf->tdf", f, np.asarray(feats, dtype=np.float64))
    rows = ff + kbt * np.swapaxes(np.asarray(divs, dtype=np.float64), 1, 2)
    return rows.reshape(-1, rows.shape[2])


def feat_gram(
    forces: np.ndarray, feats: np.ndarray, divs: np.ndarray, kbt: float, l2_regularization: float = 0.0
) -> np.ndarray:
    """``reg.T @ reg (+ l2*I)`` for one bead (featlinearmap.py:370-372, Q3)."""
    reg = feat_regressor_rows(forces, feats, divs, kbt)
    p = reg.T @ reg
    if l2_regularization > 0:
        p = p + l2_regularization * np.eye(p.shape[0])
    return p


def feat_constraint_rows(
    feats: np.ndarray, cmap_matrix: np.ndarray, bead: int, frame_indices: Sequence[int]
) -> Tuple[np.ndarray, np.ndarray]:
    """Equality rows for one bead's feature QP (featlinearmap.py:446-458).

    ``A[(s, c'), f] = sum_a cmap[c', a] phi[t_s, a, f]`` and ``b = 1[c' == bead]``; the
    frame choice (unseeded in the reference, :445, Q8) is an argument here.
    """
    sub = np.asarray(feats, dtype=np.float64)[np.asarray(frame_indices)]
    cm = np.asarray(cmap_matrix, dtype=np.float64)
    mult = np.einsum("ca,saf->scf", cm, sub)
    target = np.zeros(mult.shape[:2])
    target[:, bead] = 1.0
    return mult.reshape(-1, mult.shape[-1]), target.reshape(-1)


def feat_map_apply(
    forces: np.ndarray, feats_per_bead: Sequence[np.ndarray], divs_per_bead: Sequence[np.ndarray],
    coefs: Sequence[np.ndarray],
) -> np.ndarray:
    """Mapped forces of the fitted featurised map.

    featlinearmap.py:512-520 with core.py:428-430: per-frame weights
    ``w[t,c,a] = phi_c[t,a,:] . coef_c``, translation ``sum_f div_c[t,f,:] coef_c[f]``
    (no kbt factor: Q7), result ``sum_a w[t,c,a] F[t,a,:] + trans[t,c,:]``.
    """
    f = np.asarray(forces, dtype=np.float64)
    out = np.zeros((f.shape[0], len(coefs), 3))
    for c, (ph, dv, co) in enumerate(zip(feats_per_bead, divs_per_bead, coefs)):
        w = np.einsum("taf,f->ta", np.asarray(ph, dtype=np.float64), co)
        out[:, c, :] = np.einsum("ta,tad->td", w, f) + np.einsum("tfd,f->td", np.asarray(dv, dtype=np.float64), co)
    return out


# --------------------------------------------------------------------------------------
# config 5: Gaussian augmentation with injected noise
# --------------------------------------------------------------------------------------
def gauss_augment(
    coords: np.ndarray, forces: np.ndarray, cmap_matrix: np.ndarray, var: float, kbt: float, noise: np.ndarray
) -> Tuple[np.ndarray, np.ndarray]:
    """Augmented coordinates/forces for ``joptgauss_map`` given the noise draw.

    ``y = A x + sqrt(var) * noise`` (jaxgausstraj.py:232-234, 311-319 with a diagonal
    covariance); closed-form log-gradients (simplegausstraj.py:108-110 generalised to a
    premap A): ``grad_y = -(y - A x)/var``, ``grad_x = A'(y - A x)/var``; then
    trajectory/core.py:382-389: ``F_aug = kbt*grad_y``, ``F_real += kbt*grad_x``,
    concatenate along sites.  ``noise`` has shape (T, n_cg, 3), standard normal.
    """
    x = np.asarray(coords, dtype=np.float64)
    f = np.asarray(forces, dtype=np.float64)
    a = np.asarray(cmap_matrix, dtype=np.float64)
    eps = np.sqrt(var) * np.asarray(noise, dtype=np.float64)
    y = np.einsum("cf,tfd->tcd", a, x) + eps
    grad_y = -eps / var
    grad_x = np.einsum("cf,tcd->tfd", a, eps) / var
    full_coords = np.concatenate([x, y], axis=1)
    full_forces = np.concatenate([f + kbt * grad_x, kbt * grad_y], axis=1)
    return full_coords, full_forces


def gauss_log_gradient(
    source: np.ndarray, generated: np.ndarray, premap_matrix: Optional[np.ndarray], var: float
) -> Tuple[np.ndarray, np.ndarray]:
    """Log-gradients of ``g(y|x) = N(y; A x, var I)`` w.r.t. ``x`` and ``y``.

    Closed form of what ``JCondNormal.log_gradient`` obtains by autodiff
    (src/aggforce/trajectory/jaxgausstraj.py:77-96, 263-284): ``grad_y = -(y - A x)/var``,
    ``grad_x = A'(y - A x)/var``; ``premap_matrix=None`` is the identity premap
    (src/aggforce/trajectory/simplegausstraj.py:108-110).  Returns ``(grad_x, grad_y)`` in the
    reference's order (source first).
    """
    x = np.asarray(source, dtype=np.float64)
    y = np.asarray(generated, dtype=np.float64)
    if premap_matrix is None:
        resid = y - x
        return resid / var, -resid / var
    a = np.asarray(premap_matrix, dtype=np.float64)
    resid = y - np.einsum("cf,tfd->tcd", a, x)
    return np.einsum("cf,tcd->tfd", a, resid) / var, -resid / var


# --------------------------------------------------------------------------------------
# validation projections (SURVEY 8f-4; src/aggforce/jaxmapval.py)
# --------------------------------------------------------------------------------------
def sq_gaussian_forces(positions: np.ndarray, offset: float, width: float) -> np.ndarray:
    """Forces of the potential ``E = sum_{i,j} exp(-((|x_j - x_i|^2 - offset)/width)^2)``.

    jaxmapval.py:365-401: one unclipped Gaussian of every entry of the full SQUARED distance matrix
    (both orders of each pair and the zero diagonal, jaxutil.py:168-176), summed per frame, and
    ``-dE/dx`` by autodiff.  Closed form: each unordered pair appears twice, so
    ``F_i = -4 sum_j G'(s_ij) (x_i - x_j)`` with ``G'(s) = -2 (s - offset)/width^2 * G(s)``.
    """
    x = np.asarray(positions, dtype=np.float64)
    disp = x[:, :, None, :] - x[:, None, :, :]  # [t, i, j] = x_i - x_j
    s = (disp * disp).sum(-1)
    z = (s - offset) / width
    gprime = -2.0 * z / width * np.exp(-(z * z))
    return -4.0 * np.einsum("tij,tijd->tid", gprime, disp)


def rsqpg_offset(inner: float, outer: float, width: float, randg, sq_args: bool = True) -> Tuple[float, float]:
    """``(offset, width)`` as ``rsqpg_forces`` draws / squares them (jaxmapval.py:131-139)."""
    if sq_args:
        outer, inner, width = outer**2, inner**2, width**2
    return randg.random() * (outer - inner) + inner, width


__all__.append("rsqpg_offset")


def mscg_ip(forces: np.ndarray, funcs: np.ndarray) -> float:
    """``sum(funcs * forces) / n_steps`` (jaxmapval.py:359-360)."""
    f = np.asarray(forces, dtype=np.float64)
    return float((np.asarray(funcs, dtype=np.float64) * f).sum() / f.shape[0])


def random_force_proj(coords, forces, n_samples, randg, inner, outer, width, sq_args=True) -> List[float]:
    """Projections of ``forces`` on ``n_samples`` random Gaussian force fields (jaxmapval.py:309-319)."""
    vals = []
    for _ in range(n_samples):
        off, w = rsqpg_offset(inner, outer, width, randg, sq_args)
        vals.append(mscg_ip(forces, sq_gaussian_forces(coords, off, w)))
    return vals


def random_residual_shift(coords, forces, n_samples, randg, inner, outer, width, sq_args=True) -> List[float]:
    """``mean((F - G_s)^2) - mean(F^2)`` per random force field ``G_s`` (jaxmapval.py:227-237)."""
    f = np.asarray(forces, dtype=np.float64)
    base = float(np.mean(f**2))
    vals = []
    for _ in range(n_samples):
        off, w = rsqpg_offset(inner, outer, width, randg, sq_args)
        vals.append(float(np.mean((f - sq_gaussian_forces(coords, off, w)) ** 2)) - base)
    return vals
