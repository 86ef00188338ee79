"""GPU parity of kernel (c), the pair-distance kernels behind constraint detection, against plain float64
references: the four entry points (agf_pair_screen, agf_pair_select, agf_pair_first, agf_pair_moments)
called directly through the C ABI, and every path of ``_engine.pair_constraints``.

The constraint sets alone are a weak check: on molecular trajectories the X-H bonds have sd near 1e-5
and every other pair 1e-1 or more, so a kernel that drops frames or leaves part of a matrix unwritten
can still return the right set.  These tests compare the numbers.  References are numpy float64 for
small shapes and float64 torch element-wise ops on the device for large ones (plain torch arithmetic,
none of this project's kernels).  Output buffers are filled with sentinels before each call, so a
buffer that should be overwritten cannot pass by holding stale values, and one that should be left
alone is checked to be.
"""
import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

F64 = torch.float64
THR = 1e-3
SENTINEL_INT = -7


def _lib():
    from aggforce_b200 import _lib

    return _lib


def _engine():
    from aggforce_b200 import _engine

    return _engine


def _ptr(t):
    return _engine().ptr(t)


def _stream():
    return _engine().stream_ptr()


def _code(t):
    return _engine().dtype_code(t)


def _traj(rng, T, n, dtype, noise=0.3, box=15.0):
    """Random sites in a box, each jittered per frame: every pair has sd of order `noise`."""
    base = rng.uniform(0.0, box, size=(1, n, 3))
    return (base + rng.normal(0.0, noise, size=(T, n, 3))).astype(dtype)


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), device="cuda")


# ------------------------------------------------------------------ float64 references on the device
def _dists(x, o):
    """``[tb, m, n]`` distances ``|x[t, j] - o[t, i]|`` in float64."""
    d = x[:, None, :, :] - o[:, :, None, :]
    return torch.sqrt((d * d).sum(-1))


def _ref_m2(x, o=None):
    """All pairs ``[m, n]``: M2 = sum_t (d_t - mean)^2 (two passes), and the tolerance of a kernel that
    shifts by d_0 and reduces in one pass:  1e-11 * sum_t (d_t - d_0)^2  for the one-pass formula, plus
    1e-14 * max_t d_t * sqrt(T * sum_t (d_t - d_0)^2)  for distances that differ in their last bits
    (fused multiply-adds): that term only matters for pairs that barely move, e.g. two frames with
    d_1 ~ d_0."""
    x = torch.as_tensor(x, device="cuda").to(F64)
    o = x if o is None else torch.as_tensor(o, device="cuda").to(F64)
    T, n, m = x.shape[0], x.shape[1], o.shape[1]
    tb = max(1, (1 << 24) // (3 * n * m))
    d0 = _dists(x[:1], o[:1])[0]
    s = torch.zeros((m, n), dtype=F64, device="cuda")
    q = torch.zeros_like(s)
    dmax = torch.zeros_like(s)
    for a in range(0, T, tb):
        d = _dists(x[a : a + tb], o[a : a + tb])
        s += d.sum(0)
        q += ((d - d0) ** 2).sum(0)
        dmax = torch.maximum(dmax, d.amax(0))
    mean = s / T
    m2 = torch.zeros_like(s)
    for a in range(0, T, tb):
        m2 += ((_dists(x[a : a + tb], o[a : a + tb]) - mean) ** 2).sum(0)
    return m2, 1e-11 * q + 1e-14 * dmax * torch.sqrt(T * q) + 1e-300


def _ref_sd(x, o=None):
    m2, _ = _ref_m2(x, o)
    return torch.sqrt(m2 / x.shape[0]).cpu().numpy()


def _ref_moments_dev(x, o, pairs, shift):
    """Per-pair (sum e, sum e^2, sum |e|), e = d - shift, for a pair list, float64 on the device."""
    x = torch.as_tensor(x, device="cuda")
    o = x if o is None else torch.as_tensor(o, device="cuda")
    p = torch.as_tensor(np.asarray(pairs), device="cuda").long()
    c = torch.as_tensor(np.asarray(shift), device="cuda").to(F64)
    s1, s2, sa = (torch.zeros(p.shape[0], dtype=F64, device="cuda") for _ in range(3))
    tb = max(1, (1 << 24) // (3 * max(1, p.shape[0])))
    for a in range(0, x.shape[0], tb):
        d = x[a : a + tb][:, p[:, 1]].to(F64) - o[a : a + tb][:, p[:, 0]].to(F64)
        e = torch.sqrt((d * d).sum(-1)) - c
        s1 += e.sum(0)
        s2 += (e * e).sum(0)
        sa += e.abs().sum(0)
    return s1.cpu().numpy(), s2.cpu().numpy(), sa.cpu().numpy()


def _ref_pair_m2(x, o, pairs):
    """Two-pass M2 of listed pairs over all frames (device float64)."""
    T = x.shape[0]
    s1, _, _ = _ref_moments_dev(x, o, pairs, np.zeros(len(pairs)))
    s1b, s2b, _ = _ref_moments_dev(x, o, pairs, s1 / T)
    return s2b - s1b * s1b / T


def _ref_set(sd, self_mode, thr=THR):
    """The reference's rule on an sd matrix (as oracle.guess_pairwise_constraints applies it)."""
    sd = np.array(sd, dtype=np.float64)
    if self_mode:
        np.fill_diagonal(sd, 2 * thr)
    with np.errstate(invalid="ignore"):
        ii, jj = np.nonzero(sd < thr)
    if self_mode:
        return {frozenset((int(i), int(j))) for i, j in zip(ii, jj)}
    return {(int(i), int(j)) for i, j in zip(ii, jj)}


# ------------------------------------------------------------------ (a) agf_pair_screen
def _screen(x, o, n_other=None, pad=64):
    """Run the screen into a NaN-filled buffer; returns (matrix [m, n], the untouched tail)."""
    n = x.shape[1]
    m = n if n_other is None else n_other
    buf = torch.full((m * n + pad,), float("nan"), dtype=F64, device="cuda")
    _lib().call("agf_pair_screen", _ptr(x), _ptr(o), _code(x), x.shape[0], n, m, _ptr(buf), _stream())
    out = buf.cpu().numpy()
    return out[: m * n].reshape(m, n), out[m * n :]


def _assert_m2_close(got, ref, tol, mask=None):
    ref, tol = ref.cpu().numpy(), tol.cpu().numpy()
    if mask is not None:
        got, ref, tol = got[mask], ref[mask], tol[mask]
    err = np.abs(got - ref)
    bad = err > tol
    if bad.any():
        k = np.argmax(err / tol)
        raise AssertionError(f"{int(bad.sum())} pairs off; worst: got {got[k]:.17g}, ref {ref[k]:.17g}, "
                             f"tol {tol[k]:.3e}")


SELF_SCREEN = [(1, 1), (2, 2), (31, 8), (32, 9), (33, 32), (33, 512), (255, 100), (256, 512), (257, 1), (300, 2),
               (300, 9), (520, 100), (520, 512)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,T", SELF_SCREEN)
def test_screen_self_matches_float64_m2(n, T, dtype):
    """Self mode (other = NULL) straddles one 32-column block and the eight blocks of a row; above 256
    sites the blocks of a row loop over column blocks.  Below and on the diagonal: exactly +inf."""
    rng = np.random.default_rng(n * 1000 + T)
    x = _dev(_traj(rng, T, n, dtype))
    got, tail = _screen(x, None)
    assert np.isnan(tail).all()
    upper = np.triu(np.ones((n, n), dtype=bool), k=1)
    assert np.all(got[~upper] == np.inf)
    assert np.isfinite(got[upper]).all()
    ref, tol = _ref_m2(x)
    _assert_m2_close(got, ref, tol, upper)


CROSS_SCREEN = [(7, 33, 8), (7, 33, 512), (45, 300, 1), (45, 300, 100), (300, 7, 9), (257, 257, 32)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("m,n,T", CROSS_SCREEN)
def test_screen_cross_matches_float64_m2(m, n, T, dtype):
    """Cross mode: row-major [i over other, j over xyz], every entry visited, the diagonal not masked."""
    rng = np.random.default_rng(m * n + T)
    x, o = _dev(_traj(rng, T, n, dtype)), _dev(_traj(rng, T, m, dtype))
    got, tail = _screen(x, o, m)
    assert np.isnan(tail).all()
    assert np.isfinite(got).all()
    ref, tol = _ref_m2(x, o)
    _assert_m2_close(got, ref, tol)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,T", [(33, 9), (300, 100)])
def test_screen_aliased_cross_is_cross_mode(n, T, dtype):
    """The same device array passed as xyz and as other is cross mode: only NULL means self.  The
    diagonal is a real pair (d = 0, M2 = 0) and both orders of every pair are computed."""
    rng = np.random.default_rng(n + T)
    x = _dev(_traj(rng, T, n, dtype))
    got, tail = _screen(x, x, n)
    assert np.isnan(tail).all()
    assert np.isfinite(got).all()
    assert np.all(np.diag(got) == 0.0)
    ref, tol = _ref_m2(x, x)
    _assert_m2_close(got, ref, tol)


# ------------------------------------------------------------------ (b) agf_pair_select
def _select(m2, bound, x0, o0, cap, counts=None, pad=16):
    """Run the compaction into sentinel-filled buffers one `pad` longer than `cap`."""
    m, n = m2.shape
    d_m2 = _dev(m2.astype(np.float64))
    pairs = torch.full(((cap + pad) * 2,), SENTINEL_INT, dtype=torch.int32, device="cuda")
    shift = torch.full((cap + pad,), float("nan"), dtype=F64, device="cuda")
    acc = torch.full(((cap + pad) * 2,), float("nan"), dtype=F64, device="cuda")
    count = torch.full((1,), SENTINEL_INT, dtype=torch.int32, device="cuda")
    d_counts = None if counts is None else _dev(np.asarray(counts, dtype=np.float64))
    _lib().call("agf_pair_select", _ptr(d_m2), float(bound), _ptr(d_counts), 0 if counts is None else len(counts),
                _ptr(x0), _ptr(o0), _code(x0), n, m, cap, _ptr(pairs), _ptr(shift), _ptr(acc), _ptr(count), _stream())
    return (int(count.item()), pairs.cpu().numpy().reshape(-1, 2), shift.cpu().numpy(),
            acc.cpu().numpy().reshape(-1, 2))


def _select_matrix(rng, m, n, bound):
    """About 5 % of the entries below the bound, plus the edges: exactly at the bound, one ulp either
    side, slightly negative (cancellation in M2), +inf and NaN."""
    m2 = bound * rng.uniform(0.0, 20.0, size=(m, n))
    flat = m2.reshape(-1)
    specials = [bound, np.nextafter(bound, np.inf), np.nextafter(bound, 0.0), -1e-18, 0.0, np.inf, np.nan,
                np.inf, np.nan]
    if flat.size == 1:
        flat[0] = bound
        return m2
    at = rng.choice(flat.size, size=min(flat.size, len(specials)), replace=False)
    flat[at] = specials[: len(at)]
    return m2


def _frame0(rng, m, n, dtype, self_mode):
    x0 = _dev(rng.uniform(0.0, 15.0, size=(n, 3)).astype(dtype))
    o0 = None if self_mode else _dev(rng.uniform(0.0, 15.0, size=(m, 3)).astype(dtype))
    return x0, o0


def _shift_ref(x0, o0, pairs):
    x = x0.cpu().numpy().astype(np.float64)
    o = x if o0 is None else o0.cpu().numpy().astype(np.float64)
    return np.linalg.norm(x[pairs[:, 1]] - o[pairs[:, 0]], axis=-1)


# (n_other, n_sites, self): totals 1, 1023, 1024, 1025, 90 000 and 2^18 (self and cross)
SELECT_SHAPES = [(1, 1, True), (31, 33, False), (32, 32, True), (5, 205, False), (300, 300, True),
                 (512, 512, True), (256, 1024, False)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("m,n,self_mode", SELECT_SHAPES)
def test_select_is_row_major_nonzero(m, n, self_mode, dtype):
    """cap equal to the survivor count: the list is nonzero(m2 <= bound) in row-major order (never
    +inf or NaN), shift is the frame-0 distance, acc is zero; nothing past the survivors is written."""
    rng = np.random.default_rng(m * n)
    bound = 0.37
    m2 = _select_matrix(rng, m, n, bound)
    with np.errstate(invalid="ignore"):
        ii, jj = np.nonzero(m2 <= bound)
    want = np.stack([ii, jj], axis=1)
    k = len(want)
    assert k > 0
    x0, o0 = _frame0(rng, m, n, dtype, self_mode)
    count, pairs, shift, acc = _select(m2, bound, x0, o0, cap=k)
    assert count == k
    assert np.array_equal(pairs[:k], want)
    assert np.all(pairs[k:] == SENTINEL_INT)
    ref = _shift_ref(x0, o0, want)
    assert np.all(np.abs(shift[:k] - ref) <= 1e-14 * ref + 1e-300)
    assert np.isnan(shift[k:]).all()
    assert np.all(acc[:k] == 0.0)
    assert np.isnan(acc[k:]).all()


@pytest.mark.parametrize("m,n,self_mode", SELECT_SHAPES[1:])
def test_select_over_capacity_writes_nothing(m, n, self_mode):
    """cap one below the survivor count: count = -survivors and the list, shift and acc are untouched."""
    rng = np.random.default_rng(m + n)
    bound = 0.37
    m2 = _select_matrix(rng, m, n, bound)
    with np.errstate(invalid="ignore"):
        k = int((m2 <= bound).sum())
    assert k > 1
    x0, o0 = _frame0(rng, m, n, np.float32, self_mode)
    count, pairs, shift, acc = _select(m2, bound, x0, o0, cap=k - 1)
    assert count == -k
    assert np.all(pairs == SENTINEL_INT)
    assert np.isnan(shift).all() and np.isnan(acc).all()


def test_select_rejects_more_than_2_18_candidates():
    from aggforce_b200._lib import AgfError

    rng = np.random.default_rng(0)
    for m, n, self_mode in [(1, (1 << 18) + 1, False), (513, 513, True)]:
        x0, o0 = _frame0(rng, m, n, np.float32, self_mode)
        with pytest.raises(AgfError):
            _select(np.zeros((m, n)), 1.0, x0, o0, cap=8)


def test_select_sharded_bound_from_counts():
    """counts != NULL: `bound` is threshold^2 and the kernel compares with
    threshold^2 * sum(counts) * (1 + 1e-6) + 1e-300."""
    rng = np.random.default_rng(5)
    counts = [100.0, 250.0, 37.0]
    thr2 = THR * THR
    b = thr2 * sum(counts) * (1.0 + 1e-6) + 1e-300
    n = 40
    m2 = b * rng.uniform(0.5, 20.0, size=(n, n))
    planted = {
        (0, 1): (b, True),
        (0, 2): (np.nextafter(b, np.inf), False),
        (3, 4): (thr2 * sum(counts), True),  # inside only through the sum of the counts
        (5, 6): (thr2 * sum(counts) * (1.0 + 0.5e-6), True),  # inside only through the widening
        (7, 8): (thr2 * sum(counts) * (1.0 + 2e-6), False),
        (9, 9): (np.inf, False),
        (10, 11): (np.nan, False),
    }
    for (i, j), (v, _) in planted.items():
        m2[i, j] = v
    with np.errstate(invalid="ignore"):
        ii, jj = np.nonzero(m2 <= b)
    want = np.stack([ii, jj], axis=1)
    got_set = {(int(i), int(j)) for i, j in want}
    for ij, (_, inside) in planted.items():
        assert (ij in got_set) == inside
    x0, _ = _frame0(rng, n, n, np.float64, True)
    count, pairs, shift, acc = _select(m2, thr2, x0, None, cap=len(want), counts=counts)
    assert count == len(want)
    assert np.array_equal(pairs[: len(want)], want)
    ref = _shift_ref(x0, None, want)
    assert np.all(np.abs(shift[: len(want)] - ref) <= 1e-14 * ref + 1e-300)
    assert np.all(acc[: len(want)] == 0.0)


# ------------------------------------------------------------------ (c) agf_pair_first
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("mode", ["self", "aliased", "cross"])
def test_pair_first_is_frame0_distance(mode, dtype):
    rng = np.random.default_rng(11)
    n, m, P = 97, 41, 3000
    x = _dev(_traj(rng, 4, n, dtype))
    o = {"self": None, "aliased": x, "cross": _dev(_traj(rng, 4, m, dtype))}[mode]
    n_o = m if mode == "cross" else n
    pairs = np.stack([rng.integers(0, n_o, P), rng.integers(0, n, P)], axis=1).astype(np.int32)
    shift = torch.full((P + 16,), float("nan"), dtype=F64, device="cuda")
    d_pairs = _dev(pairs)
    _lib().call("agf_pair_first", _ptr(x), _ptr(o), _code(x), n, n_o, _ptr(d_pairs), P, _ptr(shift), _stream())
    got = shift.cpu().numpy()
    ref = _shift_ref(x[0], None if o is None else o[0], pairs)
    assert np.all(np.abs(got[:P] - ref) <= 1e-14 * ref + 1e-300)
    assert np.isnan(got[P:]).all()


# ------------------------------------------------------------------ (d) agf_pair_moments
def _moments(x, o, n_other, pairs, shift, acc=None, n_frames=None, pad=8):
    P = len(pairs)
    if acc is None:
        acc = torch.zeros(((P + pad) * 2,), dtype=F64, device="cuda")
        acc[2 * P :] = float("nan")
    T = x.shape[0] if n_frames is None else n_frames
    d_pairs, d_shift = _dev(pairs), _dev(np.asarray(shift, dtype=np.float64))  # alive until the call returns
    _lib().call("agf_pair_moments", _ptr(x), _ptr(o), _code(x), T, x.shape[1], n_other, _ptr(d_pairs), P,
                _ptr(d_shift), _ptr(acc), _stream())
    return acc


def _random_pairs(rng, P, n_o, n):
    return np.stack([rng.integers(0, n_o, P), rng.integers(0, n, P)], axis=1).astype(np.int32)


def _shift_near_frame0(rng, xh, oh, pairs):
    """Frame-0 distance moved by a random offset, so that no e_t is identically zero."""
    o = xh if oh is None else oh
    d0 = np.linalg.norm(xh[0, pairs[:, 1]].astype(np.float64) - o[0, pairs[:, 0]], axis=-1)
    return d0 + rng.normal(0.0, 0.05, size=len(pairs))


def _moments_ref(xh, oh, pairs, shift):
    """(s1, s2, sum|e|): numpy (the oracle helper) for small shapes, the device for large ones."""
    if xh.shape[0] * len(pairs) <= 2_000_000:
        s1, s2 = oracle.pair_distance_moments(xh, oh, pairs, shift)
        o = xh if oh is None else oh
        d = np.linalg.norm(xh[:, pairs[:, 1]].astype(np.float64) - o[:, pairs[:, 0]], axis=-1)
        return s1, s2, np.abs(d - shift).sum(0)
    return _ref_moments_dev(xh, oh, pairs, shift)


def _assert_moments(acc, P, ref, times=1.0):
    got = acc.cpu().numpy()
    s1, s2, sa = ref
    assert np.isnan(got[2 * P :]).all()
    got = got[: 2 * P].reshape(P, 2)
    e1, e2 = np.abs(got[:, 0] - times * s1), np.abs(got[:, 1] - times * s2)
    assert np.all(e1 <= 1e-12 * times * sa), f"sum e: worst {e1.max():.3e}"
    assert np.all(e2 <= 1e-12 * times * s2), f"sum e^2: worst {e2.max():.3e}"


MOMENT_CASES = [(1, 1), (7, 3), (255, 15), (256, 16), (257, 17), (1000, 100), (7, 5000), (1000, 17),
                (70000, 5000)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", [355, 356])
@pytest.mark.parametrize("P,T", MOMENT_CASES)
def test_moments_self(P, T, n, dtype):
    """Self mode: the staged ring up to 355 sites (three stages of 16 float32 / 8 float64 frames within
    200 KiB), the gather kernel from 356.  Below 256 pairs several threads share a pair."""
    rng = np.random.default_rng(P + T + n)
    xh = _traj(rng, T, n, dtype)
    pairs = _random_pairs(rng, P, n, n)
    shift = _shift_near_frame0(rng, xh, None, pairs)
    acc = _moments(_dev(xh), None, n, pairs, shift)
    _assert_moments(acc, P, _moments_ref(xh, None, pairs, shift))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("P,T", [(7, 5000), (257, 100), (1000, 17)])
def test_moments_cross(P, T, dtype):
    rng = np.random.default_rng(P * T)
    n, m = 300, 45
    xh, oh = _traj(rng, T, n, dtype), _traj(rng, T, m, dtype)
    pairs = _random_pairs(rng, P, m, n)
    shift = _shift_near_frame0(rng, xh, oh, pairs)
    acc = _moments(_dev(xh), _dev(oh), m, pairs, shift)
    _assert_moments(acc, P, _moments_ref(xh, oh, pairs, shift))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", [33, 34])
@pytest.mark.parametrize("start", [1, 2, 3])
def test_moments_views_into_a_trajectory(start, n, dtype):
    """A device view that starts a few frames in: the head chunk of the schedule is loaded
    cooperatively until a frame start is 16-byte aligned (odd and even n give different heads)."""
    rng = np.random.default_rng(start * 100 + n)
    T = 100
    big = _traj(rng, T + start, n, dtype)
    x = _dev(big)[start:]
    xh = big[start:]
    pairs = _random_pairs(rng, 500, n, n)
    shift = _shift_near_frame0(rng, xh, None, pairs)
    acc = _moments(x, None, n, pairs, shift)
    _assert_moments(acc, len(pairs), _moments_ref(xh, None, pairs, shift))


def test_moments_base_never_16_byte_aligned():
    """A float32 buffer viewed from element 1 with n a multiple of 4: no frame start is ever 16-byte
    aligned, so every chunk takes the cooperative-load branch."""
    rng = np.random.default_rng(21)
    T, n = 200, 32
    xh = _traj(rng, T, n, np.float32)
    flat = torch.empty(1 + T * n * 3, dtype=torch.float32, device="cuda")
    flat[1:] = _dev(xh.reshape(-1))
    x = flat[1:].view(T, n, 3)
    assert x.data_ptr() % 16 != 0 and (n * 3 * 4) % 16 == 0
    pairs = _random_pairs(rng, 700, n, n)
    shift = _shift_near_frame0(rng, xh, None, pairs)
    acc = _moments(x, None, n, pairs, shift)
    _assert_moments(acc, len(pairs), _moments_ref(xh, None, pairs, shift))


@pytest.mark.parametrize("n", [100, 400])
def test_moments_accumulate_and_zero_frames(n):
    """acc is +=: two calls give twice the sums; n_frames = 0 leaves acc bitwise unchanged.  Passing
    the same array as other (n_other = n) is the self fast path and gives the same sums."""
    rng = np.random.default_rng(n)
    T, P = 60, 900
    xh = _traj(rng, T, n, np.float32)
    x = _dev(xh)
    pairs = _random_pairs(rng, P, n, n)
    shift = _shift_near_frame0(rng, xh, None, pairs)
    ref = _moments_ref(xh, None, pairs, shift)
    acc = _moments(x, None, n, pairs, shift)
    _moments(x, None, n, pairs, shift, acc=acc)
    _assert_moments(acc, P, ref, times=2.0)
    before = acc.clone()
    _moments(x, None, n, pairs, shift, acc=acc, n_frames=0)
    assert torch.equal(acc.view(torch.int64), before.view(torch.int64))
    aliased = _moments(x, x, n, pairs, shift)
    _assert_moments(aliased, P, ref)


# ------------------------------------------------------------------ (e) _engine.pair_constraints paths
@pytest.fixture
def spy(monkeypatch):
    """Names of the entry points called (in order) while the test runs."""
    from aggforce_b200 import _lib

    names = []
    real = _lib.call

    def call(name, *args):
        names.append(name)
        return real(name, *args)

    monkeypatch.setattr(_lib, "call", call)
    return names


def _constraints(x, o=None, thr=THR):
    eng = _engine()
    return eng.pair_constraints(eng.Frames(x), None if o is None else eng.Frames(o), thr)


def _check_paths_result(pairs, sd, sd_ref, self_mode, thr=THR):
    """No false negatives against the full reference matrix, and the sd of every returned pair."""
    got = {(int(i), int(j)) for i, j in pairs}
    ii, jj = np.nonzero(np.nan_to_num(sd_ref, nan=np.inf) < thr)
    missing = [(int(i), int(j)) for i, j in zip(ii, jj) if (not self_mode or i < j) and (int(i), int(j)) not in got]
    assert not missing, f"pairs below the threshold that were pruned: {missing[:10]}"
    ref = sd_ref[pairs[:, 0], pairs[:, 1]]
    assert np.array_equal(np.isnan(sd), np.isnan(ref))
    ok = ~np.isnan(ref)
    err = np.abs(sd[ok] - ref[ok])
    assert np.all(err <= 1e-9 * ref[ok] + 1e-13), f"worst sd error {err.max():.3e}"
    return got


def _chignolin(T, seed=3):
    from aggforce_b200.synth import chignolin_topology, synth_trajectory_host

    coords, _ = synth_trajectory_host(chignolin_topology(), T, seed=seed)
    return coords


def test_path_one_kernel_select(spy):
    """Small system (n * n_other <= 2^18, <= 8192 survivors): screen, one-kernel select, moments."""
    from aggforce_b200 import guess_pairwise_constraints

    coords = _chignolin(1000)
    pairs, sd = _constraints(coords)
    assert spy == ["agf_pair_screen", "agf_pair_select", "agf_pair_moments"]
    _check_paths_result(pairs, sd, _ref_sd(coords), True)
    assert guess_pairwise_constraints(coords) == oracle.guess_pairwise_constraints(coords)
    x, o = np.ascontiguousarray(coords[:, :120]), np.ascontiguousarray(coords[:, 60:])
    spy.clear()
    pairs, sd = _constraints(x, o)
    assert spy == ["agf_pair_screen", "agf_pair_select", "agf_pair_moments"]
    _check_paths_result(pairs, sd, _ref_sd(x, o), False)
    assert guess_pairwise_constraints(x, cross_xyz=o) == oracle.guess_pairwise_constraints(x, cross_xyz=o)


def _rigid_partner(x, parent, offset):
    return x[:, parent] + np.asarray(offset)


def test_path_select_overflow_goes_general(spy):
    """More than 8192 pairs survive the 32-frame screen: the select reports the overflow and the general
    path (nonzero, agf_pair_first) takes over."""
    from aggforce_b200 import guess_pairwise_constraints

    rng = np.random.default_rng(7)
    T, n = 2000, 300
    x = _traj(rng, T, n, np.float64, noise=0.002)
    for k in range(8):
        x[:, 2 * k + 1] = _rigid_partner(x, 2 * k, rng.normal(size=3))
    pairs, sd = _constraints(x)
    assert spy[:2] == ["agf_pair_screen", "agf_pair_select"] and "agf_pair_first" in spy
    assert len(pairs) > 8192
    sd_ref = _ref_sd(x)
    _check_paths_result(pairs, sd, sd_ref, True)
    got = guess_pairwise_constraints(x)
    assert got == _ref_set(sd_ref, True) and {frozenset((2 * k, 2 * k + 1)) for k in range(8)} <= got


@pytest.mark.parametrize("cross", [False, True])
def test_path_general_many_candidates_gather(spy, cross):
    """Above 2^18 candidates (self n = 600, cross 500 x 600) there is no select; self mode at 600 sites
    streams with the gather moments kernel (the ring holds at most 355 sites)."""
    from aggforce_b200 import guess_pairwise_constraints
    from aggforce_b200.synth import protein_like_topology, synth_trajectory_host

    topo = protein_like_topology(60)
    coords, _ = synth_trajectory_host(topo, 400, seed=9)
    o = np.ascontiguousarray(coords[:, 100:]) if cross else None
    pairs, sd = _constraints(coords, o)
    assert "agf_pair_select" not in spy
    assert spy[0] == "agf_pair_screen" and spy[1] == "agf_pair_first" and spy.count("agf_pair_moments") >= 1
    sd_ref = _ref_sd(coords, o)
    _check_paths_result(pairs, sd, sd_ref, not cross)
    got = guess_pairwise_constraints(coords, cross_xyz=o)
    assert got == _ref_set(sd_ref, not cross)
    if not cross:
        assert got == topo.xh_constraints


def test_path_second_pruning_point_with_planted_pairs(spy):
    """17 000 float32 frames with small noise: more than 4n pairs survive the screen and the rescreen
    after 4096 frames prunes them.  Planted pairs:
      (40, 41) sd 0.99 thr, all of it inside the 32-frame prefix: prefix variance far above thr^2, prefix
               M2 below thr^2 T -- it must survive both pruning points and be a constraint;
      (50, 51) rigid for 4096 frames, then flexible: survives both, and its sd proves the later frames
               were streamed;
      (60, 61) rigid only in the prefix: pruned at the rescreen;
      site 70 NaN at frame 0, site 80 NaN at frame 5000 (both rigidly bonded): every pair touching
               them is excluded and nothing else changes."""
    from aggforce_b200 import guess_pairwise_constraints

    rng = np.random.default_rng(17)
    T, n = 17_000, 300
    x = _traj(rng, T, n, np.float64, noise=0.005)
    for k in range(10):
        x[:, 2 * k + 1] = _rigid_partner(x, 2 * k, rng.normal(size=3))
    t = np.arange(T)
    alt = np.where(t % 2 == 0, 1.0, -1.0)
    ex = np.array([1.0, 0.0, 0.0])
    a = 0.99 * THR * np.sqrt(T / 32.0)  # sd over T of a +-a square wave on 32 frames
    x[:, 41] = x[:, 40] + ex * (1.2 + a * alt * (t < 32))[:, None]
    x[:, 51] = x[:, 50] + ex * (1.3 + 0.01 * alt * (t >= 4096))[:, None]
    x[:, 61] = x[:, 60] + ex * (1.4 + 0.01 * alt * (t >= 32))[:, None]
    x[:, 71] = _rigid_partner(x, 70, [0.0, 1.1, 0.0])
    x[:, 81] = _rigid_partner(x, 80, [0.0, 0.0, 1.05])
    x = x.astype(np.float32)
    x[0, 70] = np.nan
    x[5000, 80, 1] = np.nan
    pairs, sd = _constraints(x)
    assert spy[0] == "agf_pair_screen" and "agf_pair_first" in spy
    assert spy.count("agf_pair_moments") >= 2
    sd_ref = _ref_sd(x)
    got = _check_paths_result(pairs, sd, sd_ref, True)
    assert (40, 41) in got and (50, 51) in got and (60, 61) not in got
    assert len(got) < 4 * n  # the rescreen pruned the flexible pairs
    by_pair = dict(zip(map(tuple, pairs.tolist()), sd))
    assert by_pair[(40, 41)] < THR and by_pair[(50, 51)] > 5 * THR
    # NaN at frame 0: pruned by the screen; NaN after the rescreen: the rigid pair survives with sd NaN
    assert not any(70 in p for p in got)
    assert all(np.isnan(s) for p, s in by_pair.items() if 80 in p) and (80, 81) in got
    cons = guess_pairwise_constraints(x)
    assert cons == _ref_set(sd_ref, True)
    assert frozenset((40, 41)) in cons and frozenset((50, 51)) not in cons
    assert frozenset((70, 71)) not in cons and frozenset((80, 81)) not in cons
    assert {frozenset((2 * k, 2 * k + 1)) for k in range(10)} <= cons


@pytest.mark.parametrize("cross", [False, True])
def test_path_streamed_host_pieces(spy, monkeypatch, cross):
    """A host array that is not kept resident streams in pieces of a few dozen frames, in self mode and
    for a host cross_xyz (which used to demand a resident copy and raise)."""
    from aggforce_b200 import guess_pairwise_constraints

    eng = _engine()
    coords = _chignolin(1500, seed=5)
    x = np.ascontiguousarray(coords[:, :120]) if cross else coords
    o = np.ascontiguousarray(coords[:, 60:]) if cross else None
    monkeypatch.setattr(eng, "_PIECE_BYTES", 48 * x.shape[1] * 12)  # 48 float32 frames per piece
    monkeypatch.setattr(eng, "_RESIDENT_FRACTION", 0.0)
    pairs, sd = _constraints(x, o)
    assert spy.count("agf_pair_moments") >= 1500 // 48
    _check_paths_result(pairs, sd, _ref_sd(x, o), not cross)
    assert guess_pairwise_constraints(x, cross_xyz=o) == oracle.guess_pairwise_constraints(x, cross_xyz=o)


def test_path_aliased_cross(spy):
    """cross_xyz is the same CUDA tensor as xyz: cross semantics, so (i, i) for every site and both
    orders of every rigid pair."""
    from aggforce_b200 import guess_pairwise_constraints

    coords = _chignolin(500, seed=6)
    x = _dev(coords)
    pairs, sd = _constraints(x, x)
    assert spy[:2] == ["agf_pair_screen", "agf_pair_select"]
    _check_paths_result(pairs, sd, _ref_sd(coords, coords), False)
    got = guess_pairwise_constraints(x, cross_xyz=x)
    want = oracle.guess_pairwise_constraints(coords, cross_xyz=coords)
    assert got == want
    assert all((i, i) in got for i in range(coords.shape[1]))


def test_path_config4_scale(spy):
    """protein_like_topology(500): 5 000 sites, 20 000 device frames.  The reference sd of every survivor,
    and the reference M2 of a random sample of 20 000 pruned pairs, which must exceed the bound."""
    from aggforce_b200 import guess_pairwise_constraints
    from aggforce_b200.synth import protein_like_topology, synth_trajectory_device

    topo = protein_like_topology(500)
    T = 20_000
    coords, _ = synth_trajectory_device(topo, T, seed=12, want_forces=False)
    spy.clear()
    pairs, sd = _constraints(coords)
    assert "agf_pair_select" not in spy and spy[:2] == ["agf_pair_screen", "agf_pair_first"]
    assert "agf_pair_moments" in spy
    m2 = _ref_pair_m2(coords, None, pairs)
    sd_ref = np.sqrt(m2 / T)
    assert np.all(np.abs(sd - sd_ref) <= 1e-9 * sd_ref + 1e-13)
    n = topo.n_sites
    alive = {(int(i), int(j)) for i, j in pairs}
    rng = np.random.default_rng(0)
    cand = np.stack([rng.integers(0, n, 60_000), rng.integers(0, n, 60_000)], axis=1)
    cand = np.array([p for p in map(tuple, cand.tolist()) if p[0] < p[1] and p not in alive][:20_000])
    assert len(cand) == 20_000
    bound = THR * THR * T * (1.0 + 1e-6) + 1e-300
    assert np.all(_ref_pair_m2(coords, None, cand) > bound)
    assert guess_pairwise_constraints(coords) == topo.xh_constraints
