"""GPU parity of the featurised-map kernels (kernel b, ``csrc/featgram.cu``) against float64 references, on
multi-site weighted bead maps: the Gram entry points (agf_gram_feat, agf_gram_feat_ws, their ``_weighted``
forms, agf_gram_feat_i8), agf_feat_rows and agf_feat_apply called directly through the C ABI, and the three
Gram routes of ``qp_feat_linear_map``.

The other featurised tests run the cln025 slice map only (one site per bead, weight 1) and compare whole Grams
in Frobenius norm, where the id block dominates.  Here every bead row has 1 to 6 weighted sites (one site in two
beads, one row over several groups), Grams are compared element by element on the scale of their diagonal,
``|P - R|_ij <= tol sqrt(R_ii R_jj)``, so a wrong small Gaussian column fails, and the shapes straddle the
8-frame chunks, the 128-column blocks, the int8 threshold n_feat 97/98 and both group-count limits of the Gram
routes (int8 up to 332 groups, packed panels up to 400).  Outputs start from sentinels: Grams from a known
non-zero matrix (they accumulate), rows and mapped forces from NaN.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import oracle
from conftest import rel_fro

pytestmark = pytest.mark.gpu

KBT = 0.6955215
WIDTH, CLIP, OUTER = 1.0, 1e-3, 8.0
BLOCK = 128                 # feature columns per Gram block
PANEL_BYTES = 24 * 132 * 8  # one packed 8-frame panel of one block
TOL_FP64, TOL_I8 = 1e-11, 1e-9
MEASURED = {}               # entry point -> largest |P - R| / sqrt(R_ii R_jj) seen (printed at teardown with -s)
I8_EVIDENCE = {}            # the int8 Gram's worst diagonal element, its column exponent and largest value


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for name, worst in sorted(MEASURED.items()):
        print(f"\n{name}: max |P-R|/sqrt(Rii Rjj) = {worst:.3e}", end="")
    if I8_EVIDENCE:
        print(f"\nagf_gram_feat_i8 worst diagonal: {I8_EVIDENCE}", end="")


def _lib():
    from aggforce_b200 import _lib

    return _lib


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), device="cuda")


class System:
    """Seeded featurised system: constraint groups of 1 to 5 sites plus one of 12 over shuffled sites (group 1 has
    one site), a coordinate map whose rows hold 1 to 6 sites with positive weights summing to one (bead 0 spans
    six groups, one of its sites is also in bead 1, bead 2 holds a site of the last group), and frames whose
    group positions spread over a 10-wide box, so that group-to-bead distances cover the centres 0..8."""

    def __init__(self, seed, n_groups, nb, n_channels, n_frames, dtype, n_cg=4):
        rng = np.random.default_rng(seed)
        sizes = rng.integers(1, 6, size=n_groups)
        if n_groups > 2:
            sizes[1] = 1
            sizes[int(rng.integers(2, n_groups))] = 12
        n = int(sizes.sum())
        members = np.split(rng.permutation(n), np.cumsum(sizes)[:-1])
        labels = np.empty(n, dtype=np.int32)
        for g, mem in enumerate(members):
            labels[mem] = g
        self.members = [np.sort(m) for m in members]
        self.cons = {frozenset((int(a), int(b))) for m in self.members for a, b in zip(m[:-1], m[1:])}
        cm = np.zeros((n_cg, n))
        for c in range(n_cg):
            k = int(rng.integers(1, 7))
            cm[c, rng.choice(n, size=k, replace=False)] = rng.uniform(0.2, 1.0, size=k)
        spread = [int(self.members[g][0]) for g in rng.choice(n_groups, size=min(6, n_groups), replace=False)]
        cm[0] = 0.0
        cm[0, spread] = rng.uniform(0.2, 1.0, size=len(spread))
        if n_cg > 1:
            cm[1, spread[0]] = 0.5
        if n_cg > 2:
            cm[2, self.members[-1][-1]] = 0.6
        cm /= cm.sum(1, keepdims=True)
        centres = rng.uniform(-5.0, 5.0, size=(n_frames, n_groups, 3))
        x = np.empty((n_frames, n, 3))
        for g, mem in enumerate(self.members):
            x[:, mem] = centres[:, g, None, :] + rng.normal(0.0, 0.4, size=(n_frames, mem.size, 3))
        self.rng = rng
        self.dtype = dtype
        self.coords = x.astype(dtype)
        self.forces = rng.normal(0.0, 5.0, size=(n_frames, n, 3)).astype(dtype)
        self.labels, self.cm = labels, cm
        self.G, self.nb, self.n_ch, self.n_cg, self.n_sites, self.T = n_groups, nb, n_channels, n_cg, n, n_frames
        self.n_feat = n_groups + nb * n_channels
        self.centers = oracle.gb_centers(0.0, OUTER, nb)
        self.upload()

    def upload(self):
        """(Re)build the device copies (after a test edits coords or cm)."""
        ptr = np.zeros(self.G + 1, dtype=np.int32)
        ptr[1:] = np.cumsum([m.size for m in self.members])
        rows, cols = np.nonzero(self.cm)
        bptr = np.zeros(self.n_cg + 1, dtype=np.int32)
        bptr[1:] = np.cumsum(np.bincount(rows, minlength=self.n_cg))
        self.d = dict(coords=_dev(self.coords), forces=_dev(self.forces), grp_ptr=_dev(ptr),
                      grp_sites=_dev(np.concatenate(self.members).astype(np.int32)), bead_ptr=_dev(bptr),
                      bead_sites=_dev(cols.astype(np.int32)), bead_w=_dev(self.cm[rows, cols]),
                      centers=_dev(self.centers), labels=_dev(self.labels))

    @property
    def code(self):
        return _lib().F32 if self.dtype == np.float32 else _lib().F64

    def maps(self):
        d = self
        return (_p(d.d["grp_ptr"]), _p(d.d["grp_sites"]), d.G, d.n_ch, _p(d.d["bead_ptr"]), _p(d.d["bead_sites"]),
                _p(d.d["bead_w"]), d.n_cg, _p(d.d["centers"]), d.nb, WIDTH, CLIP)

    def gram_args(self, t0=0, t1=None):
        t1 = self.T if t1 is None else t1
        c, f = self.d["coords"][t0:t1], self.d["forces"][t0:t1]
        return (_p(c), _p(f), self.code, t1 - t0, self.n_sites) + self.maps() + (KBT,)

    # ---------------------------------------------------------------- float64 references
    def rows(self, bead, t0=0, t1=None):
        x, f = self.coords[t0:t1].astype(np.float64), self.forces[t0:t1].astype(np.float64)
        return oracle.feat_group_rows(x, f, self.cm, self.labels, bead, self.centers, WIDTH, CLIP, self.n_ch, KBT)

    def ref_grams(self, weights=None, t0=0, t1=None):
        """(n_cg, n_feat, n_feat) float64: R = V^T V of the oracle rows (row-scaled by sqrt(w)), NaN in the rows and
        columns of every feature column that holds a NaN."""
        out = np.empty((self.n_cg, self.n_feat, self.n_feat))
        for b in range(self.n_cg):
            v = self.rows(b, t0, t1)
            if weights is not None:
                v = v * np.repeat(np.sqrt(weights), 3)[:, None]
            bad = np.isnan(v).any(0)
            r = _dev(np.where(np.isnan(v), 0.0, v))
            out[b] = (r.T @ r).cpu().numpy()
            out[b][bad, :] = np.nan
            out[b][:, bad] = np.nan
        return out

    def weights(self):
        w = self.rng.uniform(0.5, 2.0, size=self.T)
        if self.T > 1:
            w[0] = 0.0
        w[self.T // 2] = 1e3
        return w


# ---------------------------------------------------------------------------------------------- Gram entry points
def _block_lower(n):
    i = np.arange(n)
    return (i[:, None] // BLOCK) > (i[None, :] // BLOCK)


def _gram(s, entry, ref, weights=None, ws_bytes=None, t0=0, t1=None, keep=None):
    """Run one Gram entry point into a sentinel-filled buffer.  Checks that the strict lower block triangle is
    untouched and that agf_symmetrize_batch mirrors the upper triangle; returns the accumulated Gram minus the
    sentinel (valid on and above the diagonal).  ``keep`` (a dict) receives the workspace."""
    lib = _lib()
    d = np.sqrt(np.nan_to_num(np.diagonal(ref, axis1=1, axis2=2), nan=0.0))
    scale = d[:, :, None] * d[:, None, :]
    sentinel = np.where(scale > 0, 0.5 * scale, 0.25)  # known, non-zero, on the Gram's scale (exact for zeros)
    out = _dev(sentinel)
    args = s.gram_args(t0, t1)
    ws = None if ws_bytes is None else torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    w = None if weights is None else _dev(np.asarray(weights, dtype=np.float64))
    tail = {"agf_gram_feat": (), "agf_gram_feat_weighted": (_p(w),),
            "agf_gram_feat_ws": (_p(ws), C.c_size_t(ws_bytes or 0)),
            "agf_gram_feat_ws_weighted": (_p(ws), C.c_size_t(ws_bytes or 0), _p(w)),
            "agf_gram_feat_i8": (_p(ws), C.c_size_t(ws_bytes or 0))}[entry]
    lib.call(entry, *args, _p(out), *tail, _stream())
    if keep is not None:
        keep["ws"] = ws
    got = out.cpu().numpy()
    low = _block_lower(s.n_feat)
    assert np.array_equal(got[:, low], sentinel[:, low]), f"{entry} wrote below the diagonal blocks"
    lib.call("agf_symmetrize_batch", _p(out), s.n_feat, s.n_cg, _stream())
    sym = out.cpu().numpy()
    up = np.triu(np.ones((s.n_feat, s.n_feat), dtype=bool))
    assert np.array_equal(sym[:, up], got[:, up], equal_nan=True)
    assert np.array_equal(sym, sym.transpose(0, 2, 1), equal_nan=True)
    return got - sentinel


def _assert_gram(got, ref, tol, what, allowance=None):
    """|P - R|_ij <= tol sqrt(R_ii R_jj) (+ allowance_ij) on and above the diagonal, per bead; the same NaN entries;
    a reference column that is exactly zero is exactly zero."""
    n = ref.shape[-1]
    up = np.triu(np.ones((n, n), dtype=bool))
    worst = 0.0
    for b in range(ref.shape[0]):
        r, p = ref[b], got[b]
        nan = np.isnan(r)
        assert np.array_equal(np.isnan(p)[up], nan[up]), f"{what}: bead {b}: NaN pattern differs"
        dg = np.sqrt(np.nan_to_num(np.diag(r), nan=0.0))
        scale = dg[:, None] * dg[None, :]
        ok = up & ~nan
        err = np.abs(np.where(ok, p - r, 0.0))
        bound = tol * scale + (0.0 if allowance is None else allowance[b])
        bad = ok & (~(err <= bound) | ((scale == 0) & (err != 0)))
        if bad.any():
            i, j = np.argwhere(bad)[np.argmax(err[bad] / np.maximum(bound[bad], 1e-300))]
            raise AssertionError(f"{what}: bead {b}: {int(bad.sum())} entries off; worst ({i}, {j}): got "
                                 f"{p[i, j]:.17g}, ref {r[i, j]:.17g}, sqrt(RiiRjj) {scale[i, j]:.3e}, "
                                 f"bound {bound[i, j]:.3e}")
        live = ok & (scale > 0)
        if live.any():
            worst = max(worst, float((err[live] / scale[live]).max()))
    key = what.split(" ")[0]
    MEASURED[key] = max(MEASURED.get(key, 0.0), worst)


def _i8_bytes(s):
    return int(_lib().lib().agf_gram_feat_i8_workspace_bytes(s.G, s.n_ch, s.nb, s.n_cg, s.T))


def _i8_exponents(s, ws, n_frames):
    """The column exponents E of agf_gram_feat_i8 (``exps`` of its workspace, feat_i8_layout), ``(n_cg, n_feat)``:
    column x is held in 39-bit fixed point with step 2^(E_x - 39)."""
    up = lambda v: -(-v // 1024) * 1024  # noqa: E731
    n_pad = max(-(-s.n_feat // 128) * 128, -(-s.n_feat // 96) * 96)
    cols = s.n_cg * n_pad
    off = up(cols * 8 * 64) + up(cols * 8)
    e = ws[off : off + cols * 4].view(torch.int32).cpu().numpy().reshape(s.n_cg, n_pad)[:, : s.n_feat]
    assert n_frames > 0 and np.all((e >= -900) & (e <= 900))
    return e.astype(np.int64)


def _i8_allowance(exps, n_frames):
    """What the int8 digit scheme may lose per Gram element on top of float64 rounding.  A value v of column x is
    q = v 2^(39 - E_x) rounded to an integer (|q| <= 0x8080808080 < 2^39.01, or the frame goes to the float64 pass)
    and split into five signed 8-bit digits; the 15 digit products of levels s + t <= 4 are kept.  Per row, rounding
    costs at most |v_i| 2^(E_j - 40) + |v_j| 2^(E_i - 40) + 2^(E_i + E_j - 80) < 2^(E_i + E_j - 38.98), the dropped
    levels at most 2^14 (4 * 2^24 + 3 * 2^16 + 2 * 2^8 + 1) 2^(E_i + E_j - 78) < 1.001 * 2^(E_i + E_j - 38); with
    3 rows per frame, |err_ij| < 5 T 2^(E_i + E_j - 38).  The bound is relative to the column scales, not to the
    columns themselves."""
    return 5.0 * n_frames * np.ldexp(1.0, exps[:, :, None] + exps[:, None, :] - 38)


def _check_i8(s, ref, what, t0=0, t1=None):
    """agf_gram_feat_i8 element by element: 1e-9 of sqrt(R_ii R_jj) plus the digit scheme's allowance computed from
    the exponents the kernel chose.  Also records, for the element furthest beyond 1e-9 sqrt(R_ii R_jj), how far
    its column's exponent sits above the column's largest value (the evidence behind the allowance)."""
    t1 = s.T if t1 is None else t1
    need = int(_lib().lib().agf_gram_feat_i8_workspace_bytes(s.G, s.n_ch, s.nb, s.n_cg, t1 - t0))
    assert need > 0
    keep = {}
    got = _gram(s, "agf_gram_feat_i8", ref, ws_bytes=need, t0=t0, t1=t1, keep=keep)
    exps = _i8_exponents(s, keep["ws"], t1 - t0)
    allow = _i8_allowance(exps, t1 - t0)
    _assert_gram(got, ref, TOL_I8, what, allowance=allow)
    for b in range(s.n_cg):
        dg = np.sqrt(np.nan_to_num(np.diag(ref[b]), nan=0.0))
        rel = np.where(dg > 0, np.abs(np.nan_to_num(np.diag(got[b]) - np.diag(ref[b]))) / np.maximum(dg * dg, 1e-300), 0)
        k = int(np.argmax(rel))
        if rel[k] > I8_EVIDENCE.get("rel", 0.0):
            vmax = np.nanmax(np.abs(s.rows(b, t0, t1)[:, k]))
            I8_EVIDENCE.update(rel=float(rel[k]), where=f"{what} bead {b} column {k}", exp=int(exps[b, k]),
                               ilogb_max=int(np.floor(np.log2(vmax))) if vmax > 0 else None,
                               frac_of_allowance=float(abs(got[b][k, k] - ref[b][k, k]) / allow[b][k, k]))


def _check_all_grams(s, i8_expected=None):
    lib = _lib().lib()
    ref = s.ref_grams()
    full = int(lib.agf_gram_feat_workspace_bytes(s.G, s.n_ch, s.nb, s.n_cg, s.T))
    one = s.n_cg * math.ceil(s.n_feat / BLOCK) * PANEL_BYTES  # one 8-frame chunk per slab
    assert full >= one
    tag = f"G={s.G} n_feat={s.n_feat} T={s.T} {np.dtype(s.dtype).name}"
    _assert_gram(_gram(s, "agf_gram_feat", ref), ref, TOL_FP64, f"agf_gram_feat {tag}")
    _assert_gram(_gram(s, "agf_gram_feat_ws", ref, ws_bytes=full), ref, TOL_FP64, f"agf_gram_feat_ws {tag}")
    _assert_gram(_gram(s, "agf_gram_feat_ws", ref, ws_bytes=one), ref, TOL_FP64, f"agf_gram_feat_ws {tag} (slabs)")
    need = _i8_bytes(s)
    if i8_expected is not None:
        assert (need > 0) == i8_expected
    if need:
        _check_i8(s, ref, f"agf_gram_feat_i8 {tag}")
    w = s.weights()
    ref_w = s.ref_grams(w)
    _assert_gram(_gram(s, "agf_gram_feat_weighted", ref_w, weights=w), ref_w, TOL_FP64,
                 f"agf_gram_feat_weighted {tag}")
    _assert_gram(_gram(s, "agf_gram_feat_ws_weighted", ref_w, weights=w, ws_bytes=full), ref_w, TOL_FP64,
                 f"agf_gram_feat_ws_weighted {tag}")
    _assert_gram(_gram(s, "agf_gram_feat_ws_weighted", ref_w, weights=w, ws_bytes=one), ref_w, TOL_FP64,
                 f"agf_gram_feat_ws_weighted {tag} (slabs)")


DTYPES = [np.float32, np.float64]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n_frames", [1, 7, 8, 9, 33])
@pytest.mark.parametrize("n_channels", [24, 25, 0])
def test_gram_small(n_channels, n_frames, dtype):
    """25 groups, 4 centres: one 128-column block (drop and keep the last channel), and id features only; frame
    counts around the 8-frame chunk of the fused and packed kernels."""
    s = System(100 + n_channels * 40 + n_frames, 25, 4, n_channels, n_frames, dtype)
    _check_all_grams(s)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n_frames", [21, 64])
@pytest.mark.parametrize("G,nb,n_channels", [(25, 3, 24), (14, 6, 14), (32, 3, 32), (33, 3, 32)])
def test_gram_block_edges(G, nb, n_channels, n_frames, dtype):
    """n_feat 97 / 98 (the int8 route's lower bound in qp_feat_linear_map) and 128 / 129 (one block / a one-column
    second block)."""
    s = System(200 + G * 7 + n_frames, G, nb, n_channels, n_frames, dtype)
    assert s.n_feat in (97, 98, 128, 129)
    _check_all_grams(s)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("G", [332, 333, 400, 401])
def test_gram_route_edges(G, dtype):
    """Group counts at the limits of the Gram routes: agf_gram_feat_i8 takes up to 332 groups (per-frame group
    records of 8 frames plus two staging tiles in 200 KiB of shared memory), the packed kernel up to 400 (records
    alone); above that agf_gram_feat_ws runs the fused kernel."""
    s = System(300 + G, G, 2, G - 1, 50, dtype, n_cg=3)
    assert s.n_feat == 3 * G - 2
    _check_all_grams(s, i8_expected=G <= 332)


def test_gram_i8_many_frames_at_the_group_limit():
    """2 100 frames (a ragged last 32-frame chunk) at 332 groups through agf_gram_feat_i8, element by element."""
    s = System(332, 332, 2, 331, 2100, np.float32, n_cg=3)
    need = _i8_bytes(s)
    assert need > 0
    _check_i8(s, s.ref_grams(), "agf_gram_feat_i8 G=332 T=2100")


def _kernel_names(fn):
    """Names of the CUDA kernels ``fn`` launched (torch.profiler), or None if the profiler saw no kernel."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return names or None


@pytest.mark.parametrize("G", [400, 401])
def test_packed_kernel_limit_is_400_groups(G):
    """agf_gram_feat_ws packs panels up to 400 groups and runs the fused kernel above."""
    s = System(400 + G, G, 2, G - 1, 16, np.float32, n_cg=2)
    ref = s.ref_grams()
    full = int(_lib().lib().agf_gram_feat_workspace_bytes(s.G, s.n_ch, s.nb, s.n_cg, s.T))
    names = _kernel_names(lambda: _gram(s, "agf_gram_feat_ws", ref, ws_bytes=full))
    if names is None:
        pytest.skip("torch.profiler recorded no CUDA kernels on this machine")
    assert any("feat_pack_kernel" in n for n in names) == (G <= 400), sorted(names)
    assert any("feat_gram_kernel" in n for n in names) == (G > 400), sorted(names)


# ---------------------------------------------------------------------------------------------- agf_feat_rows
def _literal_rows(s, bead, frames):
    """Equality rows from the materialised features of the literal oracle (id_features + gb_features)."""
    x = s.coords[frames].astype(np.float64)
    idf, _ = oracle.id_features(len(frames), s.labels)
    parts = [idf]
    if s.n_ch:
        gf, _ = oracle.gb_features(x, s.cm, s.cons, s.labels, bead, outer=OUTER, inner=0.0, n_basis=s.nb,
                                   width=WIDTH, clip=CLIP, drop_last_channel=s.n_ch < s.G, div_method="basic")
        parts.append(gf)
    a, _ = oracle.feat_constraint_rows(np.concatenate(parts, axis=2), s.cm, bead, np.arange(len(frames)))
    return a


def _feat_rows(s, bead, frames):
    rows = torch.full((len(frames), s.n_cg, s.n_feat), float("nan"), dtype=torch.float64, device="cuda")
    sel = _dev(np.asarray(frames, dtype=np.int64))
    _lib().call("agf_feat_rows", _p(s.d["coords"]), s.code, s.n_sites, _p(sel), len(frames), bead,
                _p(s.d["labels"]), *s.maps(), _p(rows), _stream())
    return rows.cpu().numpy().reshape(len(frames) * s.n_cg, s.n_feat)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n_channels", [8, 9])
def test_feat_rows_every_bead(n_channels, dtype):
    """Frames out of order and repeated, every bead, sites of the last group (whose channel is dropped at
    n_channels = G - 1) in a bead row."""
    s = System(500 + n_channels, 9, 5, n_channels, 12, dtype, n_cg=5)
    frames = np.array([7, 0, 7, 11, 3, 3])
    assert s.cm[2, s.members[-1]].any()
    for bead in range(s.n_cg):
        got = _feat_rows(s, bead, frames)
        want = _literal_rows(s, bead, frames)
        assert np.all(np.abs(got - want) <= 1e-13 * np.maximum(1.0, np.abs(want))), f"bead {bead}"
        grp = oracle.feat_group_constraint_rows(s.coords.astype(np.float64), s.cm, s.labels, bead, frames, s.centers,
                                                WIDTH, CLIP, s.n_ch)
        assert np.all(np.abs(grp - want) <= 1e-13 * np.maximum(1.0, np.abs(want)))


# ---------------------------------------------------------------------------------------------- agf_feat_apply
def _feat_apply(s, coefs, out_dtype, t0=0, t1=None):
    t1 = s.T if t1 is None else t1
    d_coef = _dev(coefs)
    out = torch.full((t1 - t0, s.n_cg, 3), float("nan"), dtype=out_dtype, device="cuda")
    sumsq = torch.zeros(1, dtype=torch.float64, device="cuda")
    code = _lib().F32 if out_dtype == torch.float32 else _lib().F64
    _lib().call("agf_feat_apply", _p(s.d["coords"][t0:t1]), _p(s.d["forces"][t0:t1]), s.code, t1 - t0, s.n_sites,
                *s.maps(), _p(d_coef), _p(out), code, _p(sumsq), _stream())
    return out.cpu().numpy(), float(sumsq.item())


def _assert_apply(s, coefs, got, sumsq, t0=0, t1=None):
    x, f = s.coords[t0:t1].astype(np.float64), s.forces[t0:t1].astype(np.float64)
    ref = oracle.feat_group_apply(x, f, s.cm, s.labels, coefs, s.centers, WIDTH, CLIP, s.n_ch)
    mag = oracle.feat_group_apply(x, f, s.cm, s.labels, coefs, s.centers, WIDTH, CLIP, s.n_ch, magnitude=True)
    bar = 1e-12 * mag
    if got.dtype == np.float32:
        bar = bar + 2.0 ** -24 * np.abs(ref)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan)
    err = np.abs(got.astype(np.float64) - ref)
    bad = ~nan & ~(err <= bar)
    if bad.any():
        k = np.unravel_index(np.argmax(np.where(bad, err / np.maximum(bar, 1e-300), 0)), err.shape)
        raise AssertionError(f"{int(bad.sum())} mapped forces off; worst {k}: got {got[k]:.17g}, ref {ref[k]:.17g}")
    stored = got.astype(np.float64)
    if not nan.any():
        total = float((stored * stored).sum())
        assert abs(sumsq - total) <= 1e-12 * total
    return ref


@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("which", ["G", "G-1", "0"])
def test_feat_apply(which, dtype, out_dtype):
    G = 11
    n_ch = {"G": G, "G-1": G - 1, "0": 0}[which]
    s = System(600 + n_ch, G, 4, n_ch, 37, dtype, n_cg=5)
    coefs = s.rng.normal(size=(s.n_cg, s.n_feat))
    got, sumsq = _feat_apply(s, coefs, out_dtype)
    _assert_apply(s, coefs, got, sumsq)


def test_feat_apply_grid_stride_second_pass():
    """More (frame, bead) items than the kernel's capped grid (8 blocks of 256 threads per SM) holds: the
    grid-stride loop makes a second pass."""
    n_cg = 8
    items = int(1.1 * 8 * int(_lib().lib().agf_device_sm_count()) * 256) + 1
    s = System(700, 6, 3, 5, -(-items // n_cg), np.float32, n_cg=n_cg)
    coefs = s.rng.normal(size=(s.n_cg, s.n_feat))
    got, sumsq = _feat_apply(s, coefs, torch.float64)
    _assert_apply(s, coefs, got, sumsq)


# ---------------------------------------------------------------------------------------------- edges
def _every_gram_entry(s, ref, t0=0, t1=None):
    """Every Gram entry point on frames [t0, t1) against ``ref`` (unit weights for the weighted forms)."""
    lib = _lib().lib()
    nf = (s.T if t1 is None else t1) - t0
    full = int(lib.agf_gram_feat_workspace_bytes(s.G, s.n_ch, s.nb, s.n_cg, nf))
    one = s.n_cg * math.ceil(s.n_feat / BLOCK) * PANEL_BYTES
    w = np.ones(nf)
    runs = [("agf_gram_feat", {}), ("agf_gram_feat_ws", dict(ws_bytes=full)), ("agf_gram_feat_ws", dict(ws_bytes=one)),
            ("agf_gram_feat_weighted", dict(weights=w)), ("agf_gram_feat_ws_weighted", dict(weights=w, ws_bytes=full))]
    for entry, kw in runs:
        _assert_gram(_gram(s, entry, ref, t0=t0, t1=t1, **kw), ref, TOL_FP64, f"{entry} frames [{t0}, {t1})")
    _check_i8(s, ref, f"agf_gram_feat_i8 frames [{t0}, {t1})", t0, t1)


def test_clip_boundary():
    """A one-site group placed, in float64, at distances where exp(-z^2) = clip (1 +- 1e-9) for one centre, on both
    sides of it: just inside the clip g = e - clip > 0 and g' != 0, just outside both are exactly zero.  Grams
    frame by frame, the equality rows and the mapped forces follow the reference on every frame."""
    s = System(800, 8, 7, 8, 4, np.float64, n_cg=3)
    k = 4
    mu = s.centers[k]
    z_in = math.sqrt(math.log(1 / CLIP) - math.log1p(1e-9))
    z_out = math.sqrt(math.log(1 / CLIP) - math.log1p(-1e-9))
    dist = np.array([mu + WIDTH * z_in, mu + WIDTH * z_out, mu - WIDTH * z_in, mu - WIDTH * z_out])
    site = int(s.members[1][0])
    s.cm[0, site] = 0.0  # the placed site is not part of bead 0, but of bead 1's row (equality rows of bead 0)
    s.cm[1, site] = 0.3
    s.cm /= s.cm.sum(1, keepdims=True)
    bead = np.einsum("k,tkd->td", s.cm[0], s.coords)
    direction = np.array([0.6, -0.48, 0.64])
    s.coords[:, site] = bead + dist[:, None] * direction
    s.upload()
    col = s.G + 1 * s.nb + k
    v = s.rows(0)
    gp_term = v[:, col].reshape(4, 3)
    assert np.all(gp_term[[0, 2]] != 0) and np.all(gp_term[[1, 3]] == 0)  # the reference switches here
    for t in range(4):
        ref = s.ref_grams(t0=t, t1=t + 1)
        assert (ref[0, col, col] > 0) == (t in (0, 2))
        _every_gram_entry(s, ref, t, t + 1)
    frames = np.arange(4)
    got = _feat_rows(s, 0, frames)
    want = oracle.feat_group_constraint_rows(s.coords, s.cm, s.labels, 0, frames, s.centers, WIDTH, CLIP, s.n_ch)
    g_col = want.reshape(4, s.n_cg, -1)[:, 1, col]
    assert np.all(g_col[[0, 2]] > 0) and np.all(g_col[[1, 3]] == 0)
    assert np.all(np.abs(got - want) <= 1e-13 * np.maximum(1.0, np.abs(want)))
    assert np.array_equal(got == 0, want == 0)
    coefs = s.rng.normal(size=(s.n_cg, s.n_feat))
    out, sumsq = _feat_apply(s, coefs, torch.float64)
    _assert_apply(s, coefs, out, sumsq)


@pytest.mark.parametrize("dtype", DTYPES)
def test_group_on_a_slice_bead_gives_the_basic_nan_pattern(dtype):
    """SURVEY Q6: a one-site group that is bead 0's only site has d = 0 and no direction.  Every Gram entry point
    (the int8 one through its float64 pass for flagged frames) gives NaN in exactly that group's channel rows and
    columns and the reference's values elsewhere; the mapped force of bead 0 is NaN, the others are not."""
    s = System(900, 10, 3, 10, 9, dtype, n_cg=3)
    site = int(s.members[1][0])
    s.cm[0] = 0.0
    s.cm[0, site] = 1.0
    s.upload()
    ref = s.ref_grams()
    nan_cols = np.nonzero(np.isnan(np.diagonal(ref[0])))[0]
    assert np.array_equal(nan_cols, s.G + 1 * s.nb + np.arange(s.nb))
    assert not np.isnan(ref[1:]).any()
    _every_gram_entry(s, ref)
    coefs = s.rng.normal(size=(s.n_cg, s.n_feat))
    out, sumsq = _feat_apply(s, coefs, torch.float64)
    ref_out = _assert_apply(s, coefs, out, sumsq)
    assert np.isnan(ref_out[:, 0]).all() and np.isfinite(ref_out[:, 1:]).all()


# ---------------------------------------------------------------------------------------------- public API routes
ROUTES = {"ws": (60, 500, "agf_gram_feat_ws"), "i8": (60, 2048, "agf_gram_feat_i8"), "fused": (401, 40, "agf_gram_feat_ws")}


@pytest.mark.parametrize("route", list(ROUTES))
def test_qp_feat_linear_map_routes(route, monkeypatch):
    """qp_feat_linear_map on a centre-of-mass map in each Gram regime: packed panels (60 groups, < 2 048 frames),
    int8 tensor cores (60 groups, 2 048 frames, n_feat > 97) and the fused kernel behind agf_gram_feat_ws (401
    groups).  Coefficients against the exact QP solve of the float64 Gram, mapped forces against the oracle."""
    from aggforce_b200 import LinearMap, Trajectory, _engine
    from aggforce_b200 import _lib as lib
    from aggforce_b200.qp import Multifeaturize, gb_feat, id_feat, qp_feat_linear_map
    from aggforce_b200.util import Curry

    G, T, gram_entry = ROUTES[route]
    s = System(1000 + G + T, G, 2, G - 1, T, np.float32, n_cg=4)
    cmap = LinearMap(s.cm)
    feat = Multifeaturize([id_feat, Curry(gb_feat, outer=OUTER, inner=0.0, n_basis=2, width=WIDTH)])
    labels = id_feat(None, cmap, s.cons, return_ids=True)
    assert int(labels.max()) + 1 == G
    frames = s.rng.choice(T, size=20, replace=False)
    l2 = 1e3
    monkeypatch.setattr(_engine, "_GRAM_I8", [True])
    monkeypatch.setattr(_engine, "_GRAM_I8T_MIN_FRAMES", 2048)
    seen = []
    real = lib.call

    def spy(name, *args):
        seen.append(name)
        return real(name, *args)

    monkeypatch.setattr(lib, "call", spy)
    traj = Trajectory(coords=s.coords, forces=s.forces)
    fit = {}

    def run():
        fit["tmap"] = qp_feat_linear_map(traj, cmap, feat, KBT, constraints=s.cons, l2_regularization=l2,
                                         constraint_frames=frames)

    names = _kernel_names(run) if route == "fused" else run()
    mapped = fit["tmap"](traj).forces
    monkeypatch.setattr(lib, "call", real)
    grams_called = {n for n in seen if n.startswith("agf_gram_feat")}
    assert grams_called == {gram_entry}, seen
    assert "agf_feat_rows" in seen and "agf_feat_apply" in seen
    coefs = np.stack([np.asarray(c.cpu() if isinstance(c, torch.Tensor) else c) for c in
                      fit["tmap"].force_map.tags["coef_list"]])
    x, f = s.coords.astype(np.float64), s.forces.astype(np.float64)
    ref_coefs = []
    for b in range(s.n_cg):
        v = oracle.feat_group_rows(x, f, s.cm, labels, b, s.centers, WIDTH, CLIP, G - 1, KBT)
        r = _dev(v)
        p = (r.T @ r).cpu().numpy() + l2 * np.eye(v.shape[1])
        a = oracle.feat_group_constraint_rows(x, s.cm, labels, b, frames, s.centers, WIDTH, CLIP, G - 1)
        target = np.zeros((len(frames), s.n_cg))
        target[:, b] = 1.0
        ref_coefs.append(oracle.solve_equality_qp(p, a, target.reshape(-1)))
    ref_coefs = np.stack(ref_coefs)
    assert rel_fro(coefs, ref_coefs) < 1e-6
    ref_mapped = oracle.feat_group_apply(x, f, s.cm, labels, ref_coefs, s.centers, WIDTH, CLIP, G - 1)
    assert rel_fro(mapped, ref_mapped) < 1e-6
    if route == "fused":
        if names is None:
            pytest.skip("torch.profiler recorded no CUDA kernels on this machine: kernel check not made")
        assert any("feat_gram_kernel" in n for n in names), sorted(names)
        assert not any("feat_pack_kernel" in n for n in names), sorted(names)
