"""GPU parity of the linear Gram (kernel a: ``csrc/gram.cu``, ``csrc/gram_i8.cu``, ``csrc/gram_i8t.cu``) against a
float64 reference, element by element, through the C ABI and through ``_engine.gram_linear``.

The other linear-Gram tests compare whole matrices in relative Frobenius norm, where the large diagonal entries
dominate, and reach few of the compile-time instantiations.  Here every entry point runs on seeded column tables
with per-site force magnitudes spread over six decades (so small columns matter), groups of 1 to 4 sites plus one
of 6 where the route takes it, sites in no column and an empty column, at the shapes where each kernel changes
plan: all 16 static tile plans of ``gram_tri_kernel`` with both frames-per-chunk values and a one-column last
tile, frame counts around the chunk, unaligned and hopelessly aligned frame arrays, the gather kernel for
n_red > 128 and for frames too wide to stage, packed panels with narrow and full last blocks and slabs of one or
three chunks, the four ``gram_i8_kernel`` instantiations from n_red 1 to 97, and ``agf_gram_linear_i8t`` up to
its maximum n_red of 8 192.

Every Gram starts from a known non-zero sentinel (they accumulate): the entries strictly below the blocks a kernel
writes must stay the sentinel, ``agf_symmetrize`` must mirror the upper triangle, and on and above the diagonal
``|P - R| <= tol sqrt(R_ii R_jj)`` with tol = 1e-11 for the FP64 DMMA kernels.  The int8 kernels add the digit
scheme's own bound, ``5 T 2^(E_i + E_j - 38)``, with the column exponents E read back from their workspace, and
their count of frames handed to the float64 pass must equal the number of frames the test planted out of range.
``torch.profiler`` kernel names (template arguments included) show which instantiation ran.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

TOL_FP64, TOL_I8 = 1e-11, 1e-9
BLOCK = 128                  # reduced columns per block of the gather and packed-panel kernels
TILE = 8                     # tile width of gram_tri_kernel's static plans
SMEM_BUDGET = 226 * 1024     # shared memory the Gram launchers allow a CTA
PANEL_BYTES = 24 * 132 * 8   # one packed 8-frame panel of one 128-column block
I8_PANEL_BYTES = 61440       # one digit panel of gram_i8_kernel (kI8PanelBytes)
I8_COUNT_AT = 1008           # byte offset of agf_gram_linear_i8's leftover count in its workspace
I8_SAMPLE = 4096             # frames agf_gram_linear_i8 takes its column scales from
I8T_SLAB = 16384             # frames agf_gram_linear_i8t holds as digits at a time
DTYPES = [torch.float32, torch.float64]
MEASURED = {}                # route -> largest |P - R| / sqrt(R_ii R_jj) seen (printed at teardown with -s)
I8_USE = {}                  # int8 route -> largest |P - R| / (its allowance 5 T 2^(E_i + E_j - 38)) seen


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for name, worst in sorted(MEASURED.items()):
        print(f"\n{name}: max |P-R|/sqrt(Rii Rjj) = {worst:.3e}", end="")
    for name, frac in sorted(I8_USE.items()):
        print(f"\n{name}: largest fraction of the int8 allowance used = {frac:.3e}", end="")


def _lib():
    from aggforce_b200 import _lib

    return _lib


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _code(dtype):
    return _lib().F32 if dtype == torch.float32 else _lib().F64


def _tname(dtype):
    return "float" if dtype == torch.float32 else "double"


def _sm_count():
    return int(_lib().lib().agf_device_sm_count())


# ---------------------------------------------------------------------------------------------- route mirrors
def _up(v, a):
    return -(-v // a) * a


def _kf_pair(dtype):
    """Frames per chunk of the staged kernel: the larger one when it fits in shared memory, else the smaller."""
    return (16, 8) if dtype == torch.float32 else (8, 4)


def _tri_smem(dtype, kf, n_red, n_sites):
    """tri_smem_bytes of csrc/gram.cu: two f64 panels, barriers, the CSR copy and three raw frame stages."""
    item = 4 if dtype == torch.float32 else 8
    off = _up(2 * 3 * kf * 132 * 8 + 64 + (n_red + 1 + n_sites) * 4, 128)
    return off + 3 * _up(kf * n_sites * 3 * item, 16)


def _tri_kf(dtype, n_red, n_sites):
    """KF of the gram_tri_kernel that agf_gram_linear runs, or None for the gather kernel."""
    if n_red > BLOCK:
        return None
    for kf in _kf_pair(dtype):
        if _tri_smem(dtype, kf, n_red, n_sites) <= SMEM_BUDGET:
            return kf
    return None


@functools.lru_cache(maxsize=None)
def _sites_range(dtype, n_red, kf):
    """(lo, hi): the n_sites for which agf_gram_linear runs gram_tri_kernel with ``kf`` (None: the gather kernel)."""
    ok = [n for n in range(1, 4000) if _tri_kf(dtype, n_red, n) == kf]
    return ok[0], ok[-1]


def _i8_smem(n_sites, n_red):
    """gram_i8_smem of csrc/gram_i8.cu: two digit panels, barriers, exponents, the CSR copy, three raw stages."""
    off = _up(2 * I8_PANEL_BYTES + 128 + 16 + 112 * 4 + (n_red + 1 + n_sites) * 4, 128)
    return off + 3 * _up(16 * n_sites * 12, 16)


def _i8_max_sites(n_red):
    return max(n for n in range(1, 400) if _i8_smem(n, n_red) <= SMEM_BUDGET)


# ---------------------------------------------------------------------------------------------- seeded systems
def _sizes(rng, n_red, top=4, big=0, empty=True):
    """Group sizes of n_red columns: mostly small (P(k) ~ 1/k^2 for 1..top), one of ``top`` sites, one of ``big``
    sites (0: none) and one empty column where n_red allows."""
    k = np.arange(1, top + 1)
    p = 1.0 / k ** 2
    sizes = rng.choice(k, size=n_red, p=p / p.sum())
    special = rng.permutation(n_red)
    sizes[special[0]] = top
    if big and n_red >= 2:
        sizes[special[1]] = big
    if empty and n_red >= 3:
        sizes[special[2]] = 0
    return sizes, set(special[:3].tolist())


def _shrink(rng, sizes, limit, keep=()):
    """Take members off random columns (not those in ``keep``) until the sizes sum to at most ``limit``."""
    sizes = sizes.copy()
    while sizes.sum() > limit:
        can = [i for i in np.nonzero(sizes > 1)[0] if i not in keep] or list(np.nonzero(sizes > 1)[0])
        sizes[rng.choice(can)] -= 1
    return sizes


class System:
    """A column table of the C ABI (col_ptr, col_sites over shuffled sites; the sites left over are in no column)."""

    def __init__(self, rng, sizes, n_sites):
        sizes = np.asarray(sizes, dtype=np.int64)
        assert n_sites >= sizes.sum()
        self.sizes, self.n_red, self.n_sites = sizes, sizes.size, int(n_sites)
        self.ptr = np.zeros(self.n_red + 1, dtype=np.int32)
        self.ptr[1:] = np.cumsum(sizes)
        self.sites = rng.permutation(n_sites)[: sizes.sum()].astype(np.int32)
        self.d_ptr = torch.as_tensor(self.ptr, device="cuda")
        self.d_sites = torch.as_tensor(self.sites, device="cuda")
        self.max_group = int(max(1, min(4, sizes.max())))

    def members(self, x):
        return self.sites[self.ptr[x] : self.ptr[x + 1]]

    def args(self, f):
        return (_p(f), _code(f.dtype), f.shape[0], self.n_sites, _p(self.d_ptr), _p(self.d_sites), self.n_red)


def _forces(seed, n_frames, n_sites, dtype, pad=0):
    """(pad + n_frames, n_sites, 3) device forces: normal values times a per-site magnitude in 1e-3 .. 1e3."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    mag = 10.0 ** (6.0 * torch.rand(n_sites, generator=g, device="cuda", dtype=torch.float64) - 3.0)
    f = torch.randn((pad + n_frames, n_sites, 3), generator=g, device="cuda", dtype=torch.float64)
    return (f * mag[None, :, None]).to(dtype)


def _weights(rng, n_frames):
    w = rng.uniform(0.5, 2.0, size=n_frames)
    if n_frames > 1:
        w[0] = 0.0
    w[n_frames // 2] = 1e3
    return torch.as_tensor(w, device="cuda")


# ---------------------------------------------------------------------------------------------- reference and checks
def _reference(s, f, weights=None):
    """float64 R = sum_t w_t v_t v_t^T on the device: group sums in float64 by index_add_, then V^T V, per slab."""
    n_frames = f.shape[0]
    col = torch.as_tensor(np.repeat(np.arange(s.n_red), s.sizes), device="cuda")
    sites = s.d_sites.long()
    ref = torch.zeros((s.n_red, s.n_red), dtype=torch.float64, device="cuda")
    slab = max(1, (1 << 25) // max(1, 3 * sites.numel()))
    for t0 in range(0, n_frames, slab):
        x = f[t0 : t0 + slab].to(torch.float64)
        v = torch.zeros((x.shape[0], s.n_red, 3), dtype=torch.float64, device="cuda")
        v.index_add_(1, col, x[:, sites, :])
        if weights is not None:
            v = v * weights[t0 : t0 + slab].sqrt()[:, None, None]
        v = v.transpose(1, 2).reshape(-1, s.n_red)
        ref += v.T @ v
    return ref


def _same(a, b):
    """Equal, NaN where the other is NaN."""
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(torch.where(na, 0.0, a), torch.where(nb, 0.0, b))


def _scale(ref):
    d = torch.diagonal(ref)
    d = torch.sqrt(torch.where(torch.isfinite(d) & (d > 0), d, torch.zeros_like(d)))
    return d[:, None] * d[None, :]


def _gram(entry, s, f, ref, block, tail=(), head=None):
    """Run one Gram entry point into a sentinel-filled buffer.  The entries strictly below the ``block``-wide
    diagonal blocks must stay the sentinel and agf_symmetrize must mirror the upper triangle; returns the
    accumulated Gram minus the sentinel (valid on and above the diagonal)."""
    n = s.n_red
    scale = _scale(ref)
    sentinel = torch.where(scale > 0, 0.5 * scale, torch.full_like(scale, 0.25))  # exact for zero columns
    out = sentinel.clone()
    _lib().call(entry, *(s.args(f) if head is None else head), _p(out), *tail, _stream())
    got = out.clone()
    i = torch.arange(n, device="cuda") // block
    low = i[:, None] > i[None, :]
    assert torch.equal(got[low], sentinel[low]), f"{entry} wrote below the diagonal blocks"
    _lib().call("agf_symmetrize", _p(out), n, _stream())
    up = ~(torch.arange(n, device="cuda")[:, None] > torch.arange(n, device="cuda")[None, :])
    assert _same(out[up], got[up]) and _same(out, out.T), "agf_symmetrize did not mirror the upper triangle"
    return got - sentinel


def _assert_gram(got, ref, tol, route, allowance=None, what=""):
    """|P - R|_ij <= tol sqrt(R_ii R_jj) (+ allowance_ij) on and above the diagonal; the same NaN entries and the
    same infinite ones; a reference column that is exactly zero is exactly zero."""
    n = ref.shape[0]
    idx = torch.arange(n, device="cuda")
    up = idx[:, None] <= idx[None, :]
    assert torch.equal(torch.isnan(got)[up], torch.isnan(ref)[up]), f"{route} {what}: NaN pattern differs"
    inf = up & torch.isinf(ref)
    assert torch.equal(got[inf], ref[inf]), f"{route} {what}: infinite entries differ"
    scale = _scale(ref)
    ok = up & torch.isfinite(ref)
    err = torch.where(ok, (got - ref).abs(), torch.zeros_like(ref))
    bound = tol * scale + (0.0 if allowance is None else allowance)
    bad = ok & (~(err <= bound) | ((scale == 0) & (err != 0)))
    if bool(bad.any()):
        ratio = torch.where(bad, err / bound.clamp_min(1e-300), torch.zeros_like(err))
        k = int(torch.argmax(ratio))
        i, j = divmod(k, n)
        raise AssertionError(f"{route} {what}: {int(bad.sum())} entries off; worst ({i}, {j}): got "
                             f"{float(got[i, j]):.17g}, ref {float(ref[i, j]):.17g}, sqrt(RiiRjj) "
                             f"{float(scale[i, j]):.3e}, bound {float(bound[i, j]):.3e}")
    live = ok & (scale > 0)
    if bool(live.any()):
        MEASURED[route] = max(MEASURED.get(route, 0.0), float((err[live] / scale[live]).max()))
    if allowance is not None:  # where the allowance is a real part of the bar (not under a column of exponent -900)
        a = ok & (allowance > 1e-3 * tol * scale)
        if bool(a.any()):
            I8_USE[route] = max(I8_USE.get(route, 0.0), float((err[a] / allowance[a]).max()))


def _allowance(exps, n_frames):
    """What the int8 digit scheme may lose per element on top of float64 rounding.  A value v of column x is
    q = v 2^(39 - E_x) rounded to an integer (|q| <= 0x8080808080 < 2^39.01, or the frame goes to the float64 pass)
    and split into five signed 8-bit digits, of whose products the 15 with levels s + t <= 4 are kept.  Per row,
    rounding costs less than 2^(E_i + E_j - 38.98) and the dropped levels less than 1.001 * 2^(E_i + E_j - 38);
    with 3 rows per frame, |err_ij| < 5 T 2^(E_i + E_j - 38)."""
    e = torch.as_tensor(exps, dtype=torch.float64, device="cuda")
    return 5.0 * n_frames * torch.exp2(e[:, None] + e[None, :] - 38.0)


def _i8_exponents(ws, n_red):
    """Column exponents of agf_gram_linear_i8: E = ilogb(colmax) + 3 from the float64 column maxima at byte 0 of
    its workspace (column_exponent in csrc/i8.cuh; a maximum of 0 gives -900)."""
    m = ws[: 8 * n_red].view(torch.float64).cpu().numpy()
    e = np.frexp(m)[1].astype(np.int64) - 1 + 3
    e = np.where((m > 0) & (m < 1e300), np.clip(e, -900, 900), -900)
    return e


def _i8_count(ws):
    return int(ws[I8_COUNT_AT : I8_COUNT_AT + 4].view(torch.int32).item())


def _i8t_layout(n_red):
    """Byte offsets of ``exps`` and ``count`` in agf_gram_linear_i8t's workspace (i8t_layout in csrc/gram_i8t.cu)."""
    n_pad = max(_up(n_red, 128), _up(n_red, 96))
    exps = _up(n_pad * 8 * 64, 1024)
    count = exps + _up(n_pad * 4, 1024) + 2 * _up(n_pad * 8, 1024)
    return exps, count


def _i8t_exponents(ws, n_red):
    at = _i8t_layout(n_red)[0]
    e = ws[at : at + 4 * n_red].view(torch.int32).cpu().numpy().astype(np.int64)
    assert np.all((e >= -900) & (e <= 900))
    return e


def _i8t_count(ws, n_red):
    at = _i8t_layout(n_red)[1]
    return int(ws[at : at + 4].view(torch.int32).item())


def _kernel_names(fn):
    """Names of the CUDA kernels ``fn`` launched (torch.profiler), without blanks."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    assert names, "torch.profiler recorded no CUDA kernels"
    return names


def _ran(names, kernel, *targs):
    """Whether the instantiation kernel<targs...> is among the profiled names (demangled or mangled)."""
    demangled = f"{kernel}<{','.join(str(a).lower() for a in targs)}>"

    def mangle(a):
        if a in ("float", "double"):
            return a[0]
        if isinstance(a, bool):
            return f"Lb{int(a)}E"
        return f"Li{a}E"

    mangled = f"{kernel}I{''.join(mangle(a) for a in targs)}E"
    return any(demangled in n or mangled in n for n in names)


# ---------------------------------------------------------------------------------------------- gram_tri_kernel
def _tri_system(rng, dtype, n_red, kf, big):
    """Groups of 1-4 sites (and one of 6 with ``big``: the generic fill) with n_sites inside the range where
    agf_gram_linear stages ``kf`` frames per chunk."""
    sizes, keep = _sizes(rng, n_red, big=6 if big else 0)
    lo, hi = _sites_range(dtype, n_red, kf)
    sizes = _shrink(rng, sizes, hi - 3, keep)
    n_sites = max(int(sizes.sum()) + 3, lo + (hi - lo) // 3)
    assert lo <= n_sites <= hi and _tri_kf(dtype, n_red, n_sites) == kf
    return System(rng, sizes, n_sites)


def _run_fp64(s, f, w, route, what, block):
    ref = _reference(s, f, w)
    if w is None:
        got = _gram("agf_gram_linear", s, f, ref, block)
    else:
        got = _gram("agf_gram_linear_weighted", s, f, ref, block, tail=(_p(w),))
    _assert_gram(got, ref, TOL_FP64, route, what=what)


@pytest.mark.parametrize("nt", range(1, 17))
@pytest.mark.parametrize("which", ["big", "small"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_tri_kernel_every_tile_plan(dtype, which, nt):
    """gram_tri_kernel<T, KF, NT, W> for NT = ceil(n_red / 8) at n_red = 8 NT (full last tile) and 8 NT - 7 (one
    column in the last tile), with both frames-per-chunk values KF, unweighted and weighted (a zero and a 1e3
    weight), the fast fill (groups of at most 4) and the generic one (a group of 6), T = 1, 2, 3, KF - 1, KF,
    KF + 1, 2 KF + 3 frames starting 0 to 3 frames into the array (the head chunk of the schedule)."""
    kf = _kf_pair(dtype)[0 if which == "big" else 1]
    route = f"gram_tri_kernel {_tname(dtype)} KF={kf}"
    rng = np.random.default_rng(1000 * nt + 10 * kf + (dtype == torch.float64))

    def run():
        for n_red in sorted({8 * nt - 7, 8 * nt}):
            for big in (False, True):
                s = _tri_system(rng, dtype, n_red, kf, big)
                frames = [1, 2, 3, kf - 1, kf, kf + 1, 2 * kf + 3]
                for i, n_frames in enumerate(frames if not big else frames[::3]):
                    off = i % 4
                    f = _forces(int(rng.integers(1 << 31)), n_frames, s.n_sites, dtype, pad=off)[off:]
                    for w in (None, _weights(rng, n_frames)):
                        _run_fp64(s, f, w, route, f"n_red={n_red} T={n_frames} offset={off} big={big}", TILE)

    names = _kernel_names(run)
    for weighted in (False, True):
        assert _ran(names, "gram_tri_kernel", _tname(dtype), kf, nt, weighted), sorted(names)
    assert not any("gram_block_kernel" in n for n in names), sorted(names)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("which", ["big", "small"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_tri_kernel_many_chunks_per_cta(dtype, which, weighted):
    """3 SM-count x KF + 5 frames at n_red = 100: every CTA streams several chunks through its ring of raw stages
    and double-buffered panels, and the last chunk is short."""
    kf = _kf_pair(dtype)[0 if which == "big" else 1]
    rng = np.random.default_rng(77 + kf + 2 * weighted)
    s = _tri_system(rng, dtype, 100, kf, False)
    n_frames = 3 * _sm_count() * kf + 5
    f = _forces(5 + kf, n_frames, s.n_sites, dtype)
    w = _weights(rng, n_frames) if weighted else None
    names = _kernel_names(lambda: _run_fp64(s, f, w, f"gram_tri_kernel {_tname(dtype)} KF={kf}", f"T={n_frames}",
                                            TILE))
    assert _ran(names, "gram_tri_kernel", _tname(dtype), kf, 13, weighted), sorted(names)


def _unaligned(f):
    """A copy of ``f`` that starts one element past a 16-byte boundary."""
    buf = torch.empty(f.numel() + 1, dtype=f.dtype, device="cuda")
    buf[1:] = f.reshape(-1)
    return buf[1:].view(f.shape)


@pytest.mark.parametrize("which", ["big", "small", "gather"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_hopeless_alignment(dtype, which):
    """Frames that start one element past a 16-byte boundary with 12 n_sites (float32) or 24 n_sites (float64) a
    multiple of 16 bytes never reach an aligned address: the schedule's head is one chunk and every chunk is copied
    cooperatively instead of by TMA.  With fewer than 16 frames the alignment search ends early; KF + 3 frames
    (more than a chunk) once made the head chunk overflow its shared-memory stage."""
    kf = _kf_pair(dtype)[0 if which == "big" else 1]
    rng = np.random.default_rng(31 + kf + (which == "gather"))
    if which == "gather":
        sizes, _ = _sizes(rng, 200, big=6)
        n_red, n_sites, block = 200, int(sizes.sum()) + 5, BLOCK
    else:
        sizes, n_red, block = _tri_system(rng, dtype, 61, kf, False).sizes, 61, TILE
        lo, hi = _sites_range(dtype, 61, kf)
        n_sites = max(int(sizes.sum()) + 3, lo + (hi - lo) // 3)
    n_sites += (-n_sites) % 4
    s = System(rng, sizes, n_sites)
    assert which == "gather" or _tri_kf(dtype, n_red, n_sites) == kf
    for n_frames in (kf + 3, 3 * kf + 2, 21):
        f = _unaligned(_forces(9 + n_frames, n_frames, n_sites, dtype))
        assert f.data_ptr() % 16 == f.element_size() and (3 * n_sites * f.element_size()) % 16 == 0
        for w in (None, _weights(rng, n_frames)):
            route = f"gram_block_kernel {_tname(dtype)}" if which == "gather" else f"gram_tri_kernel {_tname(dtype)} KF={kf}"
            _run_fp64(s, f, w, route, f"hopeless alignment T={n_frames}", block)


# ---------------------------------------------------------------------------------------------- gram_block_kernel
@pytest.mark.parametrize("n_red", [129, 200, 256, 257, 385])
@pytest.mark.parametrize("dtype", DTYPES)
def test_block_kernel(dtype, n_red):
    """agf_gram_linear without a workspace above 128 columns: the gather kernel over 128-column block pairs."""
    kf = _kf_pair(dtype)[1]
    rng = np.random.default_rng(n_red + 7 * (dtype == torch.float64))
    sizes, _ = _sizes(rng, n_red, big=6)
    s = System(rng, sizes, int(sizes.sum()) + 5)

    def run():
        for n_frames in (1, kf + 1, 300):
            f = _forces(int(rng.integers(1 << 31)), n_frames, s.n_sites, dtype)
            for w in (None, _weights(rng, n_frames)):
                _run_fp64(s, f, w, f"gram_block_kernel {_tname(dtype)}", f"n_red={n_red} T={n_frames}", BLOCK)

    names = _kernel_names(run)
    for weighted in (False, True):
        assert _ran(names, "gram_block_kernel", _tname(dtype), kf, weighted), sorted(names)


@pytest.mark.parametrize("n_red", [1, 37, 100, 128])
@pytest.mark.parametrize("dtype", DTYPES)
def test_block_kernel_frames_too_wide_to_stage(dtype, n_red):
    """n_red <= 128 with more sites than three raw stages of the smaller chunk hold: agf_gram_linear runs the
    gather kernel with a single block (n_blocks == 1)."""
    kf = _kf_pair(dtype)[1]
    rng = np.random.default_rng(500 + n_red + (dtype == torch.float64))
    sizes, _ = _sizes(rng, n_red, big=6)
    n_sites = _sites_range(dtype, n_red, kf)[1] + 40
    assert _tri_kf(dtype, n_red, n_sites) is None
    s = System(rng, sizes, n_sites)

    def run():
        for n_frames in (1, kf + 1, 300):
            f = _forces(int(rng.integers(1 << 31)), n_frames, s.n_sites, dtype)
            for w in (None, _weights(rng, n_frames)):
                _run_fp64(s, f, w, f"gram_block_kernel {_tname(dtype)}", f"wide n_red={n_red} T={n_frames}", BLOCK)

    names = _kernel_names(run)
    for weighted in (False, True):
        assert _ran(names, "gram_block_kernel", _tname(dtype), kf, weighted), sorted(names)
    assert not any("gram_tri_kernel" in n for n in names), sorted(names)


# ---------------------------------------------------------------------------------------------- packed panels
@pytest.mark.parametrize("n_red", [129, 248, 249, 256, 257, 385, 1000])
@pytest.mark.parametrize("dtype", DTYPES)
def test_packed_panels(dtype, n_red):
    """agf_gram_linear_ws[_weighted]: the full recommended workspace (600 frames: k_splits > 1), slabs of one and
    of three 8-frame chunks, and a workspace one chunk short, with which the call must run the gather kernel."""
    rng = np.random.default_rng(3000 + n_red + (dtype == torch.float64))
    sizes, _ = _sizes(rng, n_red, big=6)
    s = System(rng, sizes, int(sizes.sum()) + 5)
    per_chunk = -(-n_red // BLOCK) * PANEL_BYTES
    route = f"pack+panel_syrk {_tname(dtype)}"

    def call(f, w, ws_bytes, what):
        ref = _reference(s, f, w)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        if w is None:
            got = _gram("agf_gram_linear_ws", s, f, ref, BLOCK, tail=(_p(ws), C.c_size_t(ws_bytes)))
        else:
            got = _gram("agf_gram_linear_ws_weighted", s, f, ref, BLOCK, tail=(_p(ws), C.c_size_t(ws_bytes), _p(w)))
        _assert_gram(got, ref, TOL_FP64, route if ws_bytes >= per_chunk else f"gram_block_kernel {_tname(dtype)}",
                     what=f"n_red={n_red} T={f.shape[0]} {what}")

    def packed():
        for n_frames, kinds in ((5, ("full",)), (600, ("full",)), (37, ("one", "three"))):
            f = _forces(int(rng.integers(1 << 31)), n_frames, s.n_sites, dtype)
            full = int(_lib().lib().agf_gram_linear_workspace_bytes(s.n_sites, n_red, n_frames))
            assert full >= per_chunk
            for kind in kinds:
                ws_bytes = {"full": full, "one": per_chunk, "three": 3 * per_chunk}[kind]
                for w in (None, _weights(rng, n_frames)):
                    call(f, w, ws_bytes, kind)

    names = _kernel_names(packed)
    for weighted in (False, True):
        assert _ran(names, "gram_pack_kernel", _tname(dtype), weighted), sorted(names)
    assert any("panel_syrk_kernel" in n for n in names) and not any("gram_block_kernel" in n for n in names)

    def short():
        f = _forces(17, 37, s.n_sites, dtype)
        for w in (None, _weights(rng, 37)):
            call(f, w, per_chunk - 16, "workspace below one chunk")

    names = _kernel_names(short)
    assert not any("gram_pack_kernel" in n or "panel_syrk_kernel" in n for n in names), sorted(names)
    for weighted in (False, True):
        assert _ran(names, "gram_block_kernel", _tname(dtype), _kf_pair(dtype)[1], weighted), sorted(names)


# ---------------------------------------------------------------------------------------------- agf_gram_linear_i8
I8_KERNELS = {"1111": ((1, 1, 1, 1), 0x01010101), "2222": ((2, 2, 2, 2), 0x02020202),
              "4221": ((4, 2, 2, 1), 0x01020204), "4444": ((4, 4, 4, 4), 0)}


def _i8_system(rng, n_red, kernel, empty=True):
    """Columns whose sizes fit the members the instantiation visits per quad slot (slot = column % 4), with an
    empty column, a few sites in no column, and no more sites than the kernel's shared memory holds."""
    visit = I8_KERNELS[kernel][0]
    sizes, keep = _sizes(rng, n_red, empty=empty)
    sizes = np.where(sizes > 0, np.minimum(sizes, [visit[x % 4] for x in range(n_red)]), 0)
    sizes = _shrink(rng, sizes, _i8_max_sites(n_red) - 3, keep)
    return System(rng, sizes, int(sizes.sum()) + 3)


def _run_i8(s, kernel, f, ref=None, what=""):
    """agf_gram_linear_i8 against ``ref`` with the int8 bar; returns the leftover count it left in its workspace."""
    n_frames = f.shape[0]
    ref = _reference(s, f) if ref is None else ref
    need = int(_lib().lib().agf_gram_linear_i8_workspace_bytes(s.n_sites, s.n_red, n_frames))
    assert need > 0
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    head = s.args(f) + (s.max_group if kernel != "4444" else 4, C.c_uint32(I8_KERNELS[kernel][1]))
    got = _gram("agf_gram_linear_i8", s, f, ref, 1, head=head, tail=(_p(ws), C.c_size_t(need)))
    allow = _allowance(_i8_exponents(ws, s.n_red), n_frames)
    _assert_gram(got, ref, TOL_I8, "gram_i8", allowance=allow, what=f"<{kernel}> n_red={s.n_red} T={n_frames} {what}")
    return _i8_count(ws)


@pytest.mark.parametrize("n_red", [1, 4, 5, 31, 32, 33, 63, 64, 95, 96, 97])
@pytest.mark.parametrize("kernel", list(I8_KERNELS))
def test_i8_kernel(kernel, n_red):
    """Every gram_i8_kernel<W0, W1, W2, W3> instantiation (slot_members 0 selects <4, 4, 4, 4>) at n_red 1 to 97:
    96 has no column riding along as row 96 of the operand, 97 has.  T around the 16-frame sub-chunk, the 32-frame
    panel and both edges of the 4 096-frame scale sample.  Clean data: no frame may take the float64 pass, the
    empty column included."""
    rng = np.random.default_rng(7000 + 100 * n_red + int(kernel))
    s = _i8_system(rng, n_red, kernel)

    def run():
        for n_frames in (1, 15, 16, 17, 33, 4095, 4096, 4097, 20011):
            f = _forces(int(rng.integers(1 << 31)), n_frames, s.n_sites, torch.float32)
            assert _run_i8(s, kernel, f, what="clean") == 0, f"T={n_frames}: frames went to the float64 pass"

    names = _kernel_names(run)
    assert _ran(names, "gram_i8_kernel", *I8_KERNELS[kernel][0]), sorted(names)


@pytest.mark.parametrize("n_red,kernel", [(97, "4221"), (40, "1111"), (64, "4444")])
def test_i8_planted_leftovers(n_red, kernel):
    """Frames the fixed-point pass must hand to the float64 pass, and only those: NaN and +-Inf frames, a value
    1e8 times its site's scale after the sample, and a column that is zero in all 4 096 sampled frames (exponent
    -900) and non-zero in ten frames after them.  Reference: the host oracle (exact IEEE NaN / Inf arithmetic)."""
    rng = np.random.default_rng(8100 + n_red)
    s = _i8_system(rng, n_red, kernel)
    n_frames = I8_SAMPLE + 300
    f = _forces(81, n_frames, s.n_sites, torch.float32)
    cols = [x for x in rng.permutation(n_red) if s.sizes[x] > 0][:5]
    site = [int(s.members(x)[0]) for x in cols]
    f[5, site[0], 1] = float("nan")
    f[9, site[1], 0] = float("inf")
    f[4200, site[2], 2] = -float("inf")
    f[4300, site[3], 1] *= 1e8
    zero = torch.as_tensor(s.members(cols[4]).astype(np.int64), device="cuda")
    f[:4100, zero] = 0.0
    f[4110:, zero] = 0.0
    planted = {5, 9, 4200, 4300} | set(range(4100, 4110))
    ref = torch.as_tensor(oracle.gram_csr(f.cpu().numpy(), s.ptr, s.sites), device="cuda")
    assert bool(torch.isnan(ref).any()) and bool(torch.isinf(ref).any())
    assert _run_i8(s, kernel, f, ref, what="planted") == len(planted)


def test_i8_leftover_in_the_second_slab():
    """SM count x 8 192 + 4 099 frames (two launches of the main kernel) at 8 sites: an out-of-range value in
    each slab; the leftover list holds frame indices of the whole array across launches."""
    rng = np.random.default_rng(8200)
    s = System(rng, [2, 1, 0, 2, 1], 8)
    slab = _sm_count() * 8192
    n_frames = slab + 4099
    f = _forces(82, n_frames, s.n_sites, torch.float32)
    for t in (5000, slab + 1000):
        f[t, int(s.members(3)[1]), 0] *= 1e8
    assert _run_i8(s, "2222", f, what="two slabs") == 2


# ---------------------------------------------------------------------------------------------- agf_gram_linear_i8t
def _run_i8t(s, f, ref=None, what=""):
    n_frames = f.shape[0]
    ref = _reference(s, f) if ref is None else ref
    need = int(_lib().lib().agf_gram_linear_i8t_workspace_bytes(s.n_sites, s.n_red, n_frames))
    assert need > 0
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    got = _gram("agf_gram_linear_i8t", s, f, ref, 1, tail=(_p(ws), C.c_size_t(need)))
    allow = _allowance(_i8t_exponents(ws, s.n_red), n_frames)
    _assert_gram(got, ref, TOL_I8, "gram_i8t", allowance=allow, what=f"n_red={s.n_red} T={n_frames} {what}")
    return _i8t_count(ws, s.n_red)


@pytest.mark.parametrize("n_red", [98, 127, 128, 129, 191, 192, 193, 385, 2600])
def test_i8t(n_red):
    """agf_gram_linear_i8t around its 128 x 96 tiles, with groups of up to 12 sites and an empty column; T around
    the 32-frame chunk, the 1 024-frame sample and the 16 384-frame slab.  From 1 023 frames on, one value 1e8
    times its site's scale sits three frames before the end (in the last slab): exactly that frame is left over."""
    rng = np.random.default_rng(9000 + n_red)
    sizes, _ = _sizes(rng, n_red, top=12)
    s = System(rng, sizes, int(sizes.sum()) + 5)
    big = int(np.argmax(s.sizes))
    for n_frames in (1, 31, 32, 33, 1023, 1025, 16383, 16384, 16385, 2 * I8T_SLAB + 77):
        f = _forces(int(rng.integers(1 << 31)), n_frames, s.n_sites, torch.float32)
        planted = n_frames >= 1023
        if planted:
            f[n_frames - 3, int(s.members(big)[-1]), 2] *= 1e8
        assert _run_i8t(s, f, what="outlier" if planted else "clean") == int(planted)


def test_i8t_largest_n_red():
    """n_red = 8 192, the largest agf_gram_linear_i8t takes, on 40 frames (the check runs on the device)."""
    rng = np.random.default_rng(9100)
    sizes, _ = _sizes(rng, 8192, top=12)
    s = System(rng, sizes, int(sizes.sum()) + 5)
    f = _forces(91, 40, s.n_sites, torch.float32)
    assert _run_i8t(s, f) == 0


# ---------------------------------------------------------------------------------------------- accumulation
@pytest.mark.parametrize("entry", ["agf_gram_linear", "agf_gram_linear_ws", "agf_gram_linear_i8",
                                   "agf_gram_linear_i8t"])
def test_two_calls_accumulate(entry):
    """Frames split over two calls into the same Gram give the Gram of all frames (the += contract the engine
    relies on for streamed pieces)."""
    rng = np.random.default_rng(len(entry))
    n_red, n_frames, cut = {"agf_gram_linear": (100, 900, 401), "agf_gram_linear_ws": (200, 900, 401),
                            "agf_gram_linear_i8": (97, 9000, 5000), "agf_gram_linear_i8t": (150, 3000, 1700)}[entry]
    if entry == "agf_gram_linear_i8":
        s = _i8_system(rng, n_red, "4221")
    else:
        sizes, _ = _sizes(rng, n_red)
        s = System(rng, sizes, int(sizes.sum()) + 5)
    f = _forces(3, n_frames, s.n_sites, torch.float32)
    ref = _reference(s, f)
    gram = torch.zeros((n_red, n_red), dtype=torch.float64, device="cuda")
    allow = torch.zeros_like(gram)
    for part in (f[:cut], f[cut:]):
        tail, ws = (), None
        if entry == "agf_gram_linear_ws":
            need = int(_lib().lib().agf_gram_linear_workspace_bytes(s.n_sites, n_red, part.shape[0]))
        elif entry == "agf_gram_linear_i8":
            need = int(_lib().lib().agf_gram_linear_i8_workspace_bytes(s.n_sites, n_red, part.shape[0]))
        elif entry == "agf_gram_linear_i8t":
            need = int(_lib().lib().agf_gram_linear_i8t_workspace_bytes(s.n_sites, n_red, part.shape[0]))
        if entry != "agf_gram_linear":
            assert need > 0
            ws = torch.empty(need, dtype=torch.uint8, device="cuda")
            tail = (_p(ws), C.c_size_t(need))
        head = s.args(part)
        if entry == "agf_gram_linear_i8":
            head = head + (s.max_group, C.c_uint32(I8_KERNELS["4221"][1]))
        _lib().call(entry, *head, _p(gram), *tail, _stream())
        if entry == "agf_gram_linear_i8":
            allow += _allowance(_i8_exponents(ws, n_red), part.shape[0])
        elif entry == "agf_gram_linear_i8t":
            allow += _allowance(_i8t_exponents(ws, n_red), part.shape[0])
    int8 = entry in ("agf_gram_linear_i8", "agf_gram_linear_i8t")
    _assert_gram(gram, ref, TOL_I8 if int8 else TOL_FP64, f"{entry} (two calls)", allowance=allow if int8 else None)


# ---------------------------------------------------------------------------------------------- engine routing
def _route_cases():
    """(name, dtype, n_red, n_frames, largest group, wide frames, weighted, int8 on, entry point expected)."""
    f32, f64 = torch.float32, torch.float64
    return [
        ("i8 at T=8192", f32, 97, 8192, 4, False, False, True, "agf_gram_linear_i8"),
        ("T=8191", f32, 97, 8191, 4, False, False, True, "agf_gram_linear"),
        ("float64", f64, 97, 8192, 4, False, False, True, "agf_gram_linear"),
        ("int8 off", f32, 97, 8192, 4, False, False, False, "agf_gram_linear"),
        ("n_red=96", f32, 96, 8192, 4, False, False, True, "agf_gram_linear_i8"),
        ("n_red=95", f32, 95, 8192, 2, False, False, True, "agf_gram_linear_i8"),
        ("group of 5", f32, 97, 8192, 5, False, False, True, "agf_gram_linear"),
        ("frames too wide for i8", f32, 97, 8192, 4, True, False, True, "agf_gram_linear"),
        ("weighted n_red=97", f32, 97, 8192, 4, False, True, True, "agf_gram_linear_ws_weighted"),
        ("n_red=98 T=2048", f32, 98, 2048, 4, False, False, True, "agf_gram_linear_i8t"),
        ("n_red=98 T=2047", f32, 98, 2047, 4, False, False, True, "agf_gram_linear"),
        ("n_red=128 T=2048", f32, 128, 2048, 5, False, False, True, "agf_gram_linear_i8t"),
        ("n_red=128 T=2047", f32, 128, 2047, 4, False, False, True, "agf_gram_linear"),
        ("n_red=129 T=2047", f32, 129, 2047, 4, False, False, True, "agf_gram_linear_ws"),
        ("n_red=129 T=2048", f32, 129, 2048, 4, False, False, True, "agf_gram_linear_i8t"),
        ("n_red=129 float64", f64, 129, 2048, 4, False, False, True, "agf_gram_linear_ws"),
        ("n_red=129 int8 off", f32, 129, 2048, 4, False, False, False, "agf_gram_linear_ws"),
        ("weighted n_red=200", f32, 200, 2048, 4, False, True, True, "agf_gram_linear_ws_weighted"),
    ]


@pytest.mark.parametrize("case", _route_cases(), ids=lambda c: c[0])
def test_engine_routes(case, monkeypatch):
    """_engine.gram_linear picks the entry point by dtype, the int8 switch, frame count (8 192 for the int8 Gram,
    2 048 for the tiled one), n_red (96 / 97 / 98, 128 / 129), largest group (4 / 5), the int8 kernel's shared
    memory (its workspace size is 0 for wider frames) and weights; the symmetric result comes back in the caller's
    column order (GramPlan deals the columns slot-major at n_red 96 / 97) and is checked element by element."""
    from aggforce_b200 import _engine
    from aggforce_b200 import _lib as lib

    name, dtype, n_red, n_frames, top, wide, weighted, i8_on, expected = case
    rng = np.random.default_rng(sum(map(ord, name)))
    sizes, keep = _sizes(rng, n_red, top=min(top, 4), big=top if top > 4 else 0)
    limit = _i8_max_sites(n_red)
    if n_red <= 97:
        sizes = _shrink(rng, sizes, limit - 3, keep)
    n_sites = limit + 1 if wide else int(sizes.sum()) + 3
    if n_red <= 97:
        assert (int(_lib().lib().agf_gram_linear_i8_workspace_bytes(n_sites, n_red, n_frames)) > 0) == (not wide)
    s = System(rng, sizes, n_sites)
    col_of_site = np.full(n_sites, -1, dtype=np.int64)
    for x in range(n_red):
        col_of_site[s.members(x)] = x
    f = _forces(int(rng.integers(1 << 31)), n_frames, n_sites, dtype)
    w = _weights(rng, n_frames) if weighted else None
    ref = _reference(s, f, w)
    monkeypatch.setattr(_engine, "_GRAM_I8", [i8_on])
    monkeypatch.setattr(_engine, "_GRAM_I8T_MIN_FRAMES", 2048)
    seen = []
    real = lib.call

    def spy(entry, *args):
        seen.append(entry)
        return real(entry, *args)

    monkeypatch.setattr(lib, "call", spy)
    wd = None if w is None else _engine.frame_weights_dev(w, n_frames)
    got = _engine.gram_linear(_engine.Frames(f), col_of_site, n_red, weights=wd)
    monkeypatch.setattr(lib, "call", real)
    grams = [e for e in seen if e.startswith("agf_gram_linear")]
    assert grams == [expected], seen
    assert _same(got, got.T)
    allow = None
    if expected in ("agf_gram_linear_i8", "agf_gram_linear_i8t"):
        ws = _engine.workspace(0)
        internal = (_i8_exponents(ws, n_red) if expected == "agf_gram_linear_i8" else _i8t_exponents(ws, n_red))
        order = _engine.GramPlan(col_of_site, n_red, want_i8=True).order
        exps = np.empty(n_red, dtype=np.int64)
        exps[order] = internal
        allow = _allowance(exps, n_frames)
    _assert_gram(got, ref, TOL_I8 if allow is not None else TOL_FP64, f"engine {expected}", allowance=allow,
                 what=name)


def test_device_reference_matches_the_oracle():
    """The device reference of this file (float64 index_add_ group sums, V^T V per slab) against oracle.gram_csr,
    weighted and not, on a mid-size system with sites in no column and an empty column."""
    rng = np.random.default_rng(4)
    sizes, _ = _sizes(rng, 150, top=6)
    s = System(rng, sizes, int(sizes.sum()) + 9)
    f = _forces(4, 3000, s.n_sites, torch.float32)
    w = _weights(rng, 3000)
    host = f.cpu().numpy()
    for weights in (None, w):
        ref = torch.as_tensor(oracle.gram_csr(host, s.ptr, s.sites, None if weights is None else weights.cpu().numpy()),
                              device="cuda")
        got = _reference(s, f, weights)
        scale = _scale(ref)
        assert bool(((got - ref).abs() <= 1e-13 * scale).all())
        assert bool((ref[scale == 0] == 0).all()) and bool((got[scale == 0] == 0).all())
