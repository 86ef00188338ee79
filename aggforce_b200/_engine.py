"""Frame-parallel statistics engine: device plumbing between the Python API and the kernels.

PyTorch is used for device memory, streams and (optionally) ``torch.distributed``; all
arithmetic on trajectory data happens in ``libagf_b200.so``.  Nothing here computes on the CPU
beyond index bookkeeping (CSR lists of constraint groups, the set of unique matrix columns).

Data model
----------
A trajectory array ``(n_frames, n_sites, 3)`` is wrapped in :class:`Frames`:
  * numpy (host) input  -> uploaded in pieces on a side stream; kernels for piece *i* run while
    piece *i+1* is in flight; the device copy is kept for later passes when it fits in HBM;
  * torch CUDA input    -> used in place, results stay on the device.
Frames are independent and every fitted quantity is a sum over frames, so under
``frame_sharding`` each rank passes its own frame slice and the accumulators are combined with
one NCCL all-reduce (SURVEY section 8e).
"""
from __future__ import annotations

import contextlib
import ctypes as C
import hashlib
import warnings
from typing import Iterator, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import F32, F64, AgfError

_PIECE_BYTES = 256 << 20  # host->device upload granularity
_RESIDENT_FRACTION = 0.45  # keep a host array resident on the device if it fits in this share of free HBM


# --------------------------------------------------------------------------------------
# device / stream helpers
# --------------------------------------------------------------------------------------
_CUDA_OK = [False]


def device() -> torch.device:
    if not _CUDA_OK[0]:  # asked once: torch.cuda.is_available() costs microseconds on every call
        if not torch.cuda.is_available():
            raise AgfError("aggforce_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")
        _CUDA_OK[0] = True
    return torch.device("cuda", torch.cuda.current_device())


def stream_ptr() -> C.c_void_p:
    """The current torch stream of the current device as a raw ``cudaStream_t`` (the C-level getter:
    ``torch.cuda.current_stream()`` builds a Python Stream object on every call)."""
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))


def ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise AgfError(f"unsupported dtype {t.dtype}")


_COPY_STREAMS: dict = {}


def _copy_stream() -> torch.cuda.Stream:
    dev = torch.cuda.current_device()
    if dev not in _COPY_STREAMS:
        _COPY_STREAMS[dev] = torch.cuda.Stream(device=dev)
    return _COPY_STREAMS[dev]


def to_host(t: torch.Tensor) -> np.ndarray:
    """Device -> pinned host copy, returned as a numpy array."""
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


def read_many(tensors: Sequence[torch.Tensor]) -> List[np.ndarray]:
    """Several device tensors -> pinned host arrays with ONE synchronisation."""
    hosts = []
    for t in tensors:
        host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        host.copy_(t, non_blocking=True)
        hosts.append(host)
    torch.cuda.current_stream().synchronize()
    return [h.numpy() for h in hosts]


_DEV_CACHE: "dict[tuple, torch.Tensor]" = {}


def _dev_cached(arr: np.ndarray) -> torch.Tensor:
    """Small read-only index / coefficient arrays are re-sent on every API call (CSR lists of the
    same constraints, the same coordinate map ...): keep device copies keyed by content."""
    key = (device().index, arr.dtype.str, arr.shape, hashlib.blake2b(arr.tobytes(), digest_size=16).digest())
    hit = _DEV_CACHE.get(key)
    if hit is None:
        if len(_DEV_CACHE) > 256:
            _DEV_CACHE.clear()
        hit = torch.as_tensor(arr, device=device())
        _DEV_CACHE[key] = hit
    return hit


_D2H_STREAMS: dict = {}


def start_d2h(t: torch.Tensor) -> torch.Tensor:
    """Begin an asynchronous device -> pinned-host copy on a dedicated stream (so that it overlaps
    later uploads on the copy stream: PCIe is full duplex).  Call :func:`finish_d2h` before reading."""
    dev = torch.cuda.current_device()
    if dev not in _D2H_STREAMS:
        _D2H_STREAMS[dev] = torch.cuda.Stream(device=dev)
    ds = _D2H_STREAMS[dev]
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream())
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    with torch.cuda.stream(ds):
        ds.wait_event(ev)
        host.copy_(t, non_blocking=True)
    t.record_stream(ds)
    return host


def start_d2h_piece(host: torch.Tensor, a: int, part: torch.Tensor) -> None:
    """Asynchronous copy of ``part`` (just produced on the current stream) into ``host[a : a + len(part)]``
    on the download stream: the output of one upload piece leaves while the next piece arrives."""
    dev = torch.cuda.current_device()
    if dev not in _D2H_STREAMS:
        _D2H_STREAMS[dev] = torch.cuda.Stream(device=dev)
    ds = _D2H_STREAMS[dev]
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream())
    with torch.cuda.stream(ds):
        ds.wait_event(ev)
        host[a : a + part.shape[0]].copy_(part, non_blocking=True)
    part.record_stream(ds)


def finish_d2h() -> None:
    ds = _D2H_STREAMS.get(torch.cuda.current_device())
    if ds is not None:
        ds.synchronize()


_WORKSPACE: dict = {}


def workspace(nbytes: int) -> torch.Tensor:
    """Scratch buffer for the packed-panel kernels (grow-only, one per device; stream-ordered reuse)."""
    dev = torch.cuda.current_device()
    buf = _WORKSPACE.get(dev)
    if buf is None or buf.numel() < nbytes:
        _WORKSPACE[dev] = None
        buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device())
        _WORKSPACE[dev] = buf
    return buf


# --------------------------------------------------------------------------------------
# deferred launches: work that does not depend on a fit's result (the coordinate-map application
# of project_forces) is enqueued right after the fit's last kernel, so the GPU runs it while the
# host solves the QP instead of idling
# --------------------------------------------------------------------------------------
_DEFERRED: list = []


def defer(fn) -> None:
    _DEFERRED.append(fn)


def run_deferred() -> None:
    while _DEFERRED:
        _DEFERRED.pop(0)()


def clear_deferred() -> None:
    _DEFERRED.clear()


_FITS_DEFERRED = [False]


@contextlib.contextmanager
def deferred_fits():
    """Inside this context a device-side fit may return before its status has been read: the caller
    (``project_forces``) reads it together with the application's status."""
    prev = _FITS_DEFERRED[0]
    _FITS_DEFERRED[0] = True
    try:
        yield
    finally:
        _FITS_DEFERRED[0] = prev


def fits_deferred() -> bool:
    return _FITS_DEFERRED[0]


def to_host_overlapped(t: torch.Tensor) -> np.ndarray:
    """Like :func:`to_host`, but deferred launches are enqueued behind ``t``'s producer and the
    host only waits for the copy of ``t`` (dedicated D2H stream)."""
    if not _DEFERRED:
        return to_host(t)
    host = start_d2h(t)
    run_deferred()
    finish_d2h()
    return host.numpy()


def dev_i32(values: Sequence[int]) -> torch.Tensor:
    return _dev_cached(np.ascontiguousarray(values, dtype=np.int32))


def dev_f64(values) -> torch.Tensor:
    arr = np.ascontiguousarray(values, dtype=np.float64)
    if arr.nbytes <= (1 << 20):
        return _dev_cached(arr)
    return torch.as_tensor(arr, device=device())


# --------------------------------------------------------------------------------------
# frame sharding across ranks
# --------------------------------------------------------------------------------------
class _Sharding:
    enabled = False
    group = None


def _dist():
    import torch.distributed as dist

    return dist


@contextlib.contextmanager
def frame_sharding(enabled: bool = True, group=None):
    """Within this context every fit treats its input as ONE RANK'S SLICE of the frames.

    Partial Grams / pair moments / residual sums are all-reduced over ``group`` (default
    process group) so every rank fits the same map, then applies it to its own frames.
    """
    prev = (_Sharding.enabled, _Sharding.group)
    _Sharding.enabled, _Sharding.group = enabled, group
    try:
        yield
    finally:
        _Sharding.enabled, _Sharding.group = prev


def sharded() -> bool:
    if not _Sharding.enabled:
        return False
    dist = _dist()
    return dist.is_available() and dist.is_initialized() and dist.get_world_size(_Sharding.group) > 1


def shard_rank() -> int:
    return _dist().get_rank(_Sharding.group) if sharded() else 0


class _PeerLink:
    """Symmetric peer-mapped buffers for ``agf_peer_exchange`` (one-shot all-reduce / all-gather of
    small float64 payloads over NVLink, csrc/peer.cu).  ``torch.distributed._symmetric_memory`` only
    does the rendezvous (allocation + exchange of the mappings); the exchange itself is our kernel
    on the caller's stream.  Falls back to the library collectives when the rendezvous is not
    available (decision agreed by all ranks)."""

    SLOT_DOUBLES = 1 << 16  # 512 KiB per slot: the 175 x 175 screening matrix is 245 KB
    links: dict = {}

    def __init__(self, group) -> None:
        import os
        import sys

        dist = _dist()
        self.ok = False
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.seq = 0
        want = (os.environ.get("AGF_PEER_REDUCE", "1") != "0" and dist.get_backend(group) == "nccl"
                and self.world <= 16)
        good = 0
        if want:
            try:
                import torch.distributed._symmetric_memory as symm

                nbytes = int(_lib.lib().agf_peer_buffer_bytes(self.SLOT_DOUBLES))
                self.buf = symm.empty(nbytes, dtype=torch.uint8, device=device())
                self.buf.zero_()
                self.handle = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
                ptrs = [int(v) for v in self.handle.buffer_ptrs]
                self.d_ptrs = torch.tensor(ptrs, dtype=torch.int64, device=device())
                self.err = torch.zeros(1, dtype=torch.int32, device=device())
                good = 1
            except Exception as exc:  # noqa: BLE001  (any failure means: use the library collectives)
                print(f"aggforce_b200: peer-memory exchange unavailable ({type(exc).__name__}: {exc}); "
                      "using NCCL collectives", file=sys.stderr)
        flag = torch.tensor([good], dtype=torch.int32, device=device())
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)  # also orders the zeroing before any signal
        torch.cuda.synchronize()
        self.ok = bool(flag.item())

    def exchange(self, t: torch.Tensor, op: int) -> torch.Tensor:
        """op 0 sum / 1 max: reduced IN PLACE; op 2: returns the gathered ``[world, numel]`` tensor."""
        self.seq += 1
        out = t if (op & 0xff) != 2 else torch.empty((self.world, t.numel()), dtype=torch.float64, device=t.device)
        _lib.call("agf_peer_exchange", ptr(self.d_ptrs), self.rank, self.world, C.c_uint32(self.seq & 0xFFFFFFFF or 1),
                  op, ptr(t), ptr(out), t.numel(), self.SLOT_DOUBLES, ptr(self.err), stream_ptr())
        return out


def _peer_link(t: torch.Tensor) -> Optional[_PeerLink]:
    """The peer link of the active sharding group if ``t`` qualifies (float64, contiguous, fits)."""
    if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and 0 < t.numel() <= _PeerLink.SLOT_DOUBLES):
        return None
    key = id(_Sharding.group)
    link = _PeerLink.links.get(key)
    if link is None:
        link = _PeerLink.links[key] = _PeerLink(_Sharding.group)
    return link if link.ok else None


def peer_exchange_errors() -> int:
    """Non-zero if any one-shot exchange gave up waiting for a peer (tests / bench check this)."""
    return sum(int(link.err.item()) for link in _PeerLink.links.values() if link.ok)


def allreduce_sum_(t: torch.Tensor) -> torch.Tensor:
    if sharded():
        link = _peer_link(t)
        if link is not None:
            return link.exchange(t, 0)
        _dist().all_reduce(t, group=_Sharding.group)
    return t


def allreduce_max_(t: torch.Tensor) -> torch.Tensor:
    if sharded():
        link = _peer_link(t)
        if link is not None:
            return link.exchange(t, 1)
        dist = _dist()
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=_Sharding.group)
    return t


def allreduce_sum_max_(t: torch.Tensor, n_sum: int) -> torch.Tensor:
    """In place: the first ``n_sum`` values are summed over ranks, the rest max-ed (one message)."""
    if sharded():
        link = _peer_link(t)
        if link is not None:
            return link.exchange(t, 3 | (int(n_sum) << 8))
        dist = _dist()
        dist.all_reduce(t[:n_sum], group=_Sharding.group)
        dist.all_reduce(t[n_sum:], op=dist.ReduceOp.MAX, group=_Sharding.group)
    return t


def allgather_dev(t: torch.Tensor) -> torch.Tensor:
    """``[world, numel]`` float64 device tensor holding every rank's ``t``."""
    link = _peer_link(t)
    if link is not None:
        return link.exchange(t, 2)
    dist = _dist()
    outs = [torch.empty_like(t) for _ in range(dist.get_world_size(_Sharding.group))]
    dist.all_gather(outs, t, group=_Sharding.group)
    return torch.stack(outs).reshape(len(outs), -1)


def allreduce_min_(t: torch.Tensor) -> torch.Tensor:
    if sharded():
        dist = _dist()
        dist.all_reduce(t, op=dist.ReduceOp.MIN, group=_Sharding.group)
    return t


def allgather_host(arr: np.ndarray) -> List[np.ndarray]:
    """Gather one small float64 array per rank (same shape everywhere)."""
    if not sharded():
        return [arr]
    dist = _dist()
    on_cuda = dist.get_backend(_Sharding.group) == "nccl"
    t = torch.as_tensor(np.ascontiguousarray(arr, dtype=np.float64))
    if on_cuda:
        t = t.to(device())
    outs = [torch.empty_like(t) for _ in range(dist.get_world_size(_Sharding.group))]
    dist.all_gather(outs, t, group=_Sharding.group)
    return [o.cpu().numpy() for o in outs]


_CHECKED_WEIGHTS: dict = {}  # id -> weakref of device weight tensors this module made and validated


def frame_weights_dev(frame_weights, n_frames: int) -> Optional[torch.Tensor]:
    """Per-frame weights of a fit as a validated float64 device tensor (``None`` stays ``None``).

    ``frame_weights``: 1-D numpy array or tensor, one entry per frame of this rank's slice, any float dtype.
    Raises ``ValueError`` for a wrong length, a negative or non-finite entry, or a sum of zero -- under
    ``frame_sharding`` the global sum, and every rank raises when any rank's slice is invalid (one exchange).
    A tensor returned here is recognised when it is passed again (``project_forces`` forwards it to the
    method), so the weights are uploaded and checked once per call."""
    import weakref

    if frame_weights is None:
        return None
    ref = _CHECKED_WEIGHTS.get(id(frame_weights))
    if ref is not None and ref() is frame_weights and frame_weights.shape[0] == n_frames:
        return frame_weights
    if isinstance(frame_weights, torch.Tensor):
        w = frame_weights.detach().to(device=device(), dtype=torch.float64).contiguous()
    else:
        arr = np.asarray(frame_weights)
        if not (np.issubdtype(arr.dtype, np.floating) or np.issubdtype(arr.dtype, np.integer)):
            raise ValueError(f"frame_weights must be a float array; got dtype {arr.dtype}")
        w = torch.as_tensor(np.ascontiguousarray(arr, dtype=np.float64), device=device())
    good_shape = w.dim() == 1 and int(w.shape[0]) == int(n_frames)
    if good_shape:
        bad = (~torch.isfinite(w) | (w < 0)).any().to(torch.float64)
        local = torch.stack([bad, torch.where(bad > 0, torch.zeros_like(bad), w.sum())])
    else:
        local = torch.tensor([1.0, 0.0], dtype=torch.float64, device=device())
    if sharded():
        dist = _dist()
        if dist.get_backend(_Sharding.group) != "nccl":
            local = local.cpu()
        dist.all_reduce(local, group=_Sharding.group)
    n_bad, total = (float(v) for v in to_host(local.to(device())))
    if not good_shape:
        raise ValueError(f"frame_weights must be a 1-D array with one weight per frame ({n_frames}); "
                         f"got shape {tuple(w.shape)}")
    if n_bad > 0:
        if sharded():
            raise ValueError("frame_weights of some rank have a wrong length or a negative or non-finite entry")
        raise ValueError("frame_weights must be finite and non-negative")
    if not total > 0.0:
        raise ValueError("frame_weights sum to zero" + (" over all ranks" if sharded() else ""))
    if len(_CHECKED_WEIGHTS) > 64:
        _CHECKED_WEIGHTS.clear()
    if w is not frame_weights:
        _CHECKED_WEIGHTS[id(w)] = weakref.ref(w)
    return w


def global_count(local: int) -> int:
    if not sharded():
        return int(local)
    dist = _dist()
    on_cuda = dist.get_backend(_Sharding.group) == "nccl"
    t = torch.tensor([int(local)], dtype=torch.int64, device=device() if on_cuda else "cpu")
    dist.all_reduce(t, group=_Sharding.group)
    return int(t.item())


# --------------------------------------------------------------------------------------
# trajectory arrays
# --------------------------------------------------------------------------------------
_SHARED_UPLOADS: dict = {}


@contextlib.contextmanager
def shared_uploads(*arrays):
    """While the context is open, ``Frames(a)`` of any of ``arrays`` (matched by identity) shares ONE
    upload: ``project_forces`` opens it around constraint detection, the fit and the application, so
    the caller's own arrays -- not a proxy -- can be handed to every ``method`` / featurizer."""
    added = []
    for a in arrays:
        if a is None or isinstance(a, Frames) or id(a) in _SHARED_UPLOADS:
            continue
        _SHARED_UPLOADS[id(a)] = (a, Frames(a))  # the array is kept alive: its id cannot be recycled
        added.append(id(a))
    try:
        yield
    finally:
        for key in added:
            _SHARED_UPLOADS.pop(key, None)


class Frames:
    """A ``(n_frames, n_sites, 3)`` array as the kernels see it (see module docstring)."""

    def __new__(cls, array=None, *args, **kwargs):
        # virtual frame sources (subclasses: Gaussian-augmented frames, synthetic frames) pass through
        # unchanged; their __init__ must tolerate the second call
        if cls is Frames and isinstance(array, Frames) and type(array) is not Frames:
            return array
        return super().__new__(cls)

    def __init__(self, array) -> None:
        if array is self:
            return
        shared = _SHARED_UPLOADS.get(id(array))
        if shared is not None and shared[0] is array:  # upload made once per project_forces call
            array = shared[1]
        if isinstance(array, Frames):
            self.__dict__ = array.__dict__  # share state (and the cached device copy)
            return
        self._dev: Optional[torch.Tensor] = None
        self._host: Optional[np.ndarray] = None
        if isinstance(array, torch.Tensor) and array.is_cuda:
            if array.dtype not in (torch.float32, torch.float64):
                array = array.to(torch.float64)
            self._dev = array.contiguous()
            shape = tuple(self._dev.shape)
        else:
            if isinstance(array, torch.Tensor):
                array = array.numpy()
            host = np.asarray(array)
            if host.dtype not in (np.float32, np.float64):
                host = host.astype(np.float64)
            self._host = np.ascontiguousarray(host)
            shape = self._host.shape
        if len(shape) != 3 or shape[2] != 3:
            raise ValueError(f"expected an array of shape (n_frames, n_sites, 3); got {shape}")
        self.n_frames, self.n_sites = int(shape[0]), int(shape[1])

    @property
    def on_host(self) -> bool:
        return self._host is not None

    @property
    def shape(self) -> Tuple[int, int, int]:
        return (self.n_frames, self.n_sites, 3)

    def __len__(self) -> int:
        return self.n_frames

    @property
    def np_dtype(self):
        if self._host is not None:
            return self._host.dtype
        return np.float32 if self._dev.dtype == torch.float32 else np.float64

    @property
    def torch_dtype(self):
        return torch.float32 if self.np_dtype == np.float32 else torch.float64

    def nbytes(self) -> int:
        return self.n_frames * self.n_sites * 3 * np.dtype(self.np_dtype).itemsize

    def _fits(self) -> bool:
        free, _ = torch.cuda.mem_get_info()
        return self.nbytes() <= _RESIDENT_FRACTION * free

    def piece_frames(self) -> int:
        """Frames per upload piece of a host array (a multiple of 4: 16-byte aligned piece starts)."""
        frame_bytes = max(1, self.n_sites * 3 * np.dtype(self.np_dtype).itemsize)
        return max(4, (_PIECE_BYTES // frame_bytes) // 4 * 4)

    def pieces(self, start: int = 0, stop: Optional[int] = None, per: Optional[int] = None
               ) -> Iterator[Tuple[int, torch.Tensor]]:
        """Yield ``(first_frame, device_tensor)`` pieces covering frames [start, stop).

        Every yielded tensor is safe to use on the current stream.  Host arrays are uploaded
        on a side stream one piece ahead of the consumer, ``per`` frames at a time (default:
        ``piece_frames()``).
        """
        stop = self.n_frames if stop is None else min(stop, self.n_frames)
        if start >= stop:
            return
        if self._dev is not None:
            yield start, self._dev[start:stop]
            return
        device()
        per = self.piece_frames() if per is None else max(4, int(per) // 4 * 4)
        whole = start == 0 and stop == self.n_frames and self._fits()
        cs, cur = _copy_stream(), torch.cuda.current_stream()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            src = torch.from_numpy(self._host)
        if whole:
            full = torch.empty((self.n_frames, self.n_sites, 3), dtype=self.torch_dtype, device=device())
        bounds = list(range(start, stop, per)) + [stop]
        events = []
        views = []

        def launch(i: int) -> None:
            a, b = bounds[i], bounds[i + 1]
            dst = full[a:b] if whole else torch.empty((b - a, self.n_sites, 3), dtype=self.torch_dtype,
                                                      device=device())
            if not whole:
                # a fresh staging block may reuse the memory of piece i-2, already released on the host
                # but possibly still being read by a kernel on the compute stream: order the copy after
                # everything enqueued there so far (kernel i-1 is enqueued after this call, so the
                # upload still overlaps it)
                cs.wait_stream(cur)
            with torch.cuda.stream(cs):
                dst.copy_(src[a:b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cs)
            dst.record_stream(cs)
            events.append(ev)
            views.append(dst)

        cs.wait_stream(cur)
        n_pieces = len(bounds) - 1
        launch(0)
        for i in range(n_pieces):
            if i + 1 < n_pieces:
                launch(i + 1)
            cur.wait_event(events[i])
            yield bounds[i], views[i]
            views[i] = None  # type: ignore[call-overload]
        if whole:
            self._dev = full

    def frame_range(self, t0: int, count: int) -> torch.Tensor:
        """Frames ``[t0, t0 + count)`` as ONE device tensor usable on the current stream."""
        if self._dev is not None:
            return self._dev[t0 : t0 + count]
        parts = [p for _, p in self.pieces(t0, t0 + count)]
        return parts[0] if len(parts) == 1 else torch.cat(parts)

    def resident(self) -> torch.Tensor:
        """The whole array on the device (uploaded once and cached)."""
        if self._dev is None:
            if not self._fits():
                raise AgfError("trajectory array does not fit in device memory; use pieces()")
            for _ in self.pieces():
                pass
        return self._dev  # type: ignore[return-value]

    def gather(self, frame_indices: np.ndarray) -> torch.Tensor:
        """Selected frames ``(len(idx), n_sites, 3)`` on the device."""
        idx = np.asarray(frame_indices, dtype=np.int64)
        if self._dev is not None:
            return self._dev[torch.as_tensor(idx, device=self._dev.device)].contiguous()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return torch.from_numpy(np.ascontiguousarray(self._host[idx])).to(device())

    def prefix(self, n: int) -> torch.Tensor:
        """First ``n`` frames on the device."""
        n = min(n, self.n_frames)
        if self._dev is not None:
            return self._dev[:n]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return torch.from_numpy(self._host[:n]).to(device())


def paired_pieces(a: Frames, b: Frames) -> Iterator[Tuple[int, torch.Tensor, torch.Tensor]]:
    """``(first_frame, piece_of_a, piece_of_b)`` over ONE frame schedule shared by both arrays.

    Each array on its own would be cut by its own rule (a device tensor is one piece, a host array
    is cut by bytes per frame, virtual sources by their slab size), so zipping two ``pieces()``
    generators pairs different frame ranges.  Two plain host arrays are cut with the smaller of
    their piece lengths (uploads of both stay one piece ahead); otherwise ``a`` drives and ``b``
    supplies the matching range."""
    if a.n_frames != b.n_frames:
        raise ValueError(f"paired arrays have {a.n_frames} and {b.n_frames} frames")
    plain = type(a) is Frames and type(b) is Frames
    if plain and a._dev is None and b._dev is None:
        per = min(a.piece_frames(), b.piece_frames())
        ga, gb = a.pieces(per=per), b.pieces(per=per)
        for (t0, pa), (t1, pb) in zip(ga, gb):
            if t0 != t1 or pa.shape[0] != pb.shape[0]:
                raise AgfError(f"paired upload schedules diverged at frames {t0} / {t1}")
            yield t0, pa, pb
        for _ in ga:  # run both generators to their end: that is where the resident copy is kept
            pass
        for _ in gb:
            pass
        return
    if plain and a._dev is not None and b._dev is None:  # let the host array drive its own uploads
        for t0, pb in b.pieces():
            yield t0, a._dev[t0 : t0 + pb.shape[0]], pb
        return
    for t0, pa in a.pieces():
        yield t0, pa, b.frame_range(t0, pa.shape[0])


def allreduce_host_sum(arr: np.ndarray) -> np.ndarray:
    """Sum of one float64 host array over the ranks of the sharding group (same shape everywhere)."""
    if not sharded():
        return arr
    return np.sum(allgather_host(np.ascontiguousarray(arr, dtype=np.float64).reshape(-1)), axis=0).reshape(arr.shape)


def broadcast_host(arr: np.ndarray, src: int = 0) -> np.ndarray:
    """Rank ``src``'s copy of a float64 host array (same shape everywhere)."""
    if not sharded():
        return arr
    return allgather_host(np.ascontiguousarray(arr, dtype=np.float64).reshape(-1))[src].reshape(arr.shape)


# --------------------------------------------------------------------------------------
# index structures
# --------------------------------------------------------------------------------------
def csr_from_labels(labels: np.ndarray, n_groups: int) -> Tuple[np.ndarray, np.ndarray]:
    """CSR (ptr, members) listing, for every group g, the sites with ``labels == g`` in
    increasing site order; negative labels are skipped."""
    labels = np.asarray(labels, dtype=np.int64)
    keep = np.nonzero(labels >= 0)[0]
    order = keep[np.argsort(labels[keep], kind="stable")]
    counts = np.bincount(labels[keep], minlength=n_groups)
    ptr_ = np.zeros(n_groups + 1, dtype=np.int32)
    np.cumsum(counts, out=ptr_[1:])
    return ptr_, order.astype(np.int32)


# --------------------------------------------------------------------------------------
# kernel wrappers
# --------------------------------------------------------------------------------------
import os as _os

# int8 / tcgen05 Gram (csrc/gram_i8.cu, csrc/gram_i8t.cu): on by default for long float32 trajectories;
# AGF_GRAM_I8=0 selects the FP64 DMMA kernel everywhere (A/B measurements, bit-exact FP64 products)
_GRAM_I8 = [_os.environ.get("AGF_GRAM_I8", "1") != "0"]
_GRAM_I8_MIN_FRAMES = 8192
_GRAM_I8T_MIN_FRAMES = int(_os.environ.get("AGF_GRAM_I8T_MIN_FRAMES", "2048"))  # tiled variant, n_red > 97


class GramPlan:
    """Column order and device-side CSR of the constraint groups for kernel (a) -- a function of the
    column table only, so fits over the same constraints build it once."""

    def __init__(self, col_of_site: np.ndarray, n_red: int, want_i8: bool = True) -> None:
        col_of_site = np.asarray(col_of_site, dtype=np.int64)
        sizes = np.bincount(col_of_site[col_of_site >= 0], minlength=n_red)
        # largest groups first: with lane = column in 32-column groups the group holding the few
        # 3- and 4-member columns is then also the one holding pairs, and the ragged last group holds
        # singles -- the number of (warp-wide) f64 additions per frame drops from 33 to 12 at cln025
        order = np.argsort(-sizes, kind="stable")  # internal position -> caller's column
        self.i8_shape = bool(want_i8 and n_red and n_red <= 97 and 1 <= int(sizes.max()) <= 4)
        if self.i8_shape and n_red >= 96:
            # int8 / tcgen05 kernel: a lane owns the column quad 4q..4q+3; slot c of every quad should hold
            # columns of similar group size (uniform member loops): deal the size-sorted columns slot by slot
            slot_major = np.empty(96, dtype=np.int64)
            slot_major[(np.arange(96) % 24) * 4 + np.arange(96) // 24] = order[:96]
            order = np.concatenate([slot_major, order[96:]])
        if n_red > 128:
            # packed-panel path: no per-lane member walk to balance; keep the caller's order (columns follow
            # their first site), so the pack kernel's gathers of neighbouring columns hit neighbouring sites
            order = np.arange(n_red)
        rank = np.empty(n_red, dtype=np.int64)
        rank[order] = np.arange(n_red)
        internal = np.where(col_of_site >= 0, rank[np.maximum(col_of_site, 0)], -1)
        ptr_, sites = csr_from_labels(internal, n_red)
        self.order, self.n_red = order, n_red
        self.d_ptr, self.d_sites = dev_i32(ptr_), dev_i32(sites)
        self.max_group = int(sizes.max()) if n_red else 0
        isz = sizes[order]  # group size of every internal column
        self.slot_members = 0
        for c in range(4):
            members = isz[c:96:4]
            self.slot_members |= (int(members.max()) if members.size else 1) << (8 * c)


def gram_linear_raw(frames: Frames, col_of_site: np.ndarray, n_red: int, plan: Optional[GramPlan] = None,
                    weights: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, np.ndarray]:
    """Kernel (a): accumulated and all-reduced second-moment matrix as the kernels leave it --
    ``(gram f64 [n_red, n_red] with the element-wise UPPER triangle valid, order)`` where
    ``order[p]`` is the caller's column held at internal position ``p``.  ``weights``: per-frame weights
    from :func:`frame_weights_dev`; the weighted Gram runs on the FP64 DMMA kernels (the int8 paths
    take their column scales from a sample of frames, which a heavy frame outside it would defeat)."""
    if plan is None:
        plan = GramPlan(col_of_site, n_red, want_i8=_GRAM_I8[0] and frames.np_dtype == np.float32)
    d_ptr, d_sites, order = plan.d_ptr, plan.d_sites, plan.order
    gram = torch.zeros((n_red, n_red), dtype=torch.float64, device=device())
    for t0, piece in frames.pieces():
        if weights is not None:
            w = weights[t0 : t0 + piece.shape[0]]
            need = int(_lib.lib().agf_gram_linear_workspace_bytes(frames.n_sites, n_red, piece.shape[0]))
            ws = workspace(need) if need > 0 else None
            _lib.call("agf_gram_linear_ws_weighted", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites,
                      ptr(d_ptr), ptr(d_sites), n_red, ptr(gram), ptr(ws), C.c_size_t(0 if ws is None else ws.numel()),
                      ptr(w), stream_ptr())
            continue
        need_i8 = 0
        if (_GRAM_I8[0] and plan.i8_shape and piece.dtype == torch.float32
                and piece.shape[0] >= _GRAM_I8_MIN_FRAMES):
            need_i8 = int(_lib.lib().agf_gram_linear_i8_workspace_bytes(frames.n_sites, n_red, piece.shape[0]))
        if need_i8 > 0:  # tcgen05 int8 slices (Ozaki): the Blackwell tensor-core path
            ws = workspace(need_i8)
            _lib.call("agf_gram_linear_i8", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites, ptr(d_ptr),
                      ptr(d_sites), n_red, plan.max_group, C.c_uint32(plan.slot_members), ptr(gram), ptr(ws),
                      C.c_size_t(ws.numel()), stream_ptr())
            continue
        if (_GRAM_I8[0] and n_red > 97 and piece.dtype == torch.float32
                and piece.shape[0] >= _GRAM_I8T_MIN_FRAMES):
            need_i8 = int(_lib.lib().agf_gram_linear_i8t_workspace_bytes(frames.n_sites, n_red, piece.shape[0]))
            if need_i8 > 0:  # the same digit scheme tiled over the Gram (csrc/gram_i8t.cu)
                ws = workspace(need_i8)
                _lib.call("agf_gram_linear_i8t", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites,
                          ptr(d_ptr), ptr(d_sites), n_red, ptr(gram), ptr(ws), C.c_size_t(ws.numel()), stream_ptr())
                continue
        need = int(_lib.lib().agf_gram_linear_workspace_bytes(frames.n_sites, n_red, piece.shape[0]))
        if need > 0:  # n_red > 128: pack group sums once, TMA-fed SYRK
            ws = workspace(need)
            _lib.call("agf_gram_linear_ws", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites, ptr(d_ptr),
                      ptr(d_sites), n_red, ptr(gram), ptr(ws), C.c_size_t(ws.numel()), stream_ptr())
        else:
            _lib.call("agf_gram_linear", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites, ptr(d_ptr),
                      ptr(d_sites), n_red, ptr(gram), stream_ptr())
    allreduce_sum_(gram)
    return gram, order


def gram_linear(frames: Frames, col_of_site: np.ndarray, n_red: int,
                weights: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Kernel (a): all-reduced, symmetrised second-moment matrix (device f64 [n_red, n_red]) in the
    caller's column order (``weights``: see :func:`gram_linear_raw`)."""
    gram, order = gram_linear_raw(frames, col_of_site, n_red, weights=weights)
    _lib.call("agf_symmetrize", ptr(gram), n_red, stream_ptr())
    if not np.array_equal(order, np.arange(n_red)):
        rank = np.empty(n_red, dtype=np.int64)
        rank[order] = np.arange(n_red)
        back = _dev_cached(np.ascontiguousarray(rank, dtype=np.int64))  # cached: no pageable upload per call
        gram = gram[back][:, back]
    return gram


def weighted_sumsq(x: torch.Tensor, weights: torch.Tensor, out: torch.Tensor) -> None:
    """``out`` (device f64 [1], +=) gets ``sum_t weights[t] * sum(x[t]**2)`` of a device array ``(T, ...)``."""
    x = x.contiguous()
    _lib.call("agf_weighted_sumsq", ptr(x), dtype_code(x), x.shape[0], int(np.prod(x.shape[1:])), ptr(weights),
              ptr(out), stream_ptr())


class CompiledMap:
    """Device-side form of a (n_cg, n_fg) matrix for kernel (d)."""

    def __init__(self, matrix: np.ndarray, keep_zero_columns: bool, column_labels: Optional[np.ndarray] = None) -> None:
        """``column_labels`` (optional, ``int[n_fg]``): a labelling under which equal labels are KNOWN to
        have identical matrix columns (e.g. the reduced columns of a fit) -- skips the column search."""
        m = np.asarray(matrix)
        self.n_cg, self.n_fg = m.shape
        self.out_f32 = m.dtype == np.float32
        m64 = np.ascontiguousarray(m, dtype=np.float64)
        nz_per_row = (m64 != 0).sum(axis=1)
        nnz = int(nz_per_row.sum())
        self.sparse = (not keep_zero_columns) and nnz <= 8 * self.n_cg and np.isfinite(m64).all()
        if self.sparse:
            rows, cols = np.nonzero(m64)
            ptr_ = np.zeros(self.n_cg + 1, dtype=np.int32)
            np.cumsum(np.bincount(rows, minlength=self.n_cg), out=ptr_[1:])
            if nnz == 0:  # degenerate all-zero map: one explicit zero weight keeps the kernel simple
                ptr_[1:] = 1
                cols = np.zeros(1, dtype=np.int64)
                weights = np.zeros(1)
            else:
                weights = m64[rows, cols]
            self.row_ptr, self.row_sites, self.row_w = dev_i32(ptr_), dev_i32(cols), dev_f64(weights)
            self.slice = nnz == self.n_cg and bool((nz_per_row == 1).all())  # one site per bead
            return
        if column_labels is not None:
            inverse = np.asarray(column_labels, dtype=np.int64)
            firsts = np.full(int(inverse.max()) + 1, -1, dtype=np.int64)
            firsts[inverse[::-1]] = np.arange(self.n_fg)[::-1]  # first site of every label
            uniq = np.ascontiguousarray(m64.T[firsts])
        else:
            uniq, inverse = np.unique(m64.T, axis=0, return_inverse=True)
        inverse = np.asarray(inverse).reshape(-1)
        if not keep_zero_columns:
            zero = np.nonzero(~uniq.any(axis=1))[0]
            if zero.size and uniq.shape[0] > 1:
                z = int(zero[0])
                relabel = np.arange(uniq.shape[0])
                relabel[z] = -1
                relabel[z + 1 :] -= 1
                inverse = relabel[inverse]
                uniq = np.delete(uniq, z, axis=0)
        # order unique columns by member count: the lanes of a warp then walk member lists of equal
        # length (f32->f64 conversions issue per warp instruction, divergent lists would serialise)
        sizes = np.bincount(inverse[inverse >= 0], minlength=uniq.shape[0])
        order = np.argsort(sizes, kind="stable")
        if self.n_cg > 64:
            # packed-panel GEMM path: order the unique columns by their first site instead, so the pack
            # kernel's gathers for neighbouring columns hit neighbouring sites of a frame
            live = np.nonzero(inverse >= 0)[0]
            first = np.full(uniq.shape[0], self.n_fg, dtype=np.int64)
            np.minimum.at(first, inverse[live], live)
            order = np.argsort(first, kind="stable")
        rank = np.empty_like(order)
        rank[order] = np.arange(order.size)
        inverse = np.where(inverse >= 0, rank[np.maximum(inverse, 0)], -1)
        uniq = uniq[order]
        ptr_, sites = csr_from_labels(inverse, uniq.shape[0])
        self.n_ucol, self.nnz = int(uniq.shape[0]), int(sites.size)
        self.ucol_ptr, self.ucol_sites = dev_i32(ptr_), dev_i32(sites)
        self.umat_t = dev_f64(uniq)  # [n_ucol, n_cg]
        self._finite = bool(np.isfinite(uniq).all())

    @classmethod
    def from_labels(cls, column_labels: np.ndarray, n_cg: int, n_labels: int) -> Tuple["CompiledMap", np.ndarray]:
        """Dense-small map whose unique columns are KNOWN to be the labels (the reduced columns of a
        fit) and whose values are filled in on the device (``agf_qp_equality_small`` writes ``umat_t``).
        Returns ``(map, ucol_of_label)``; same unique-column order as the value-based constructor."""
        self = cls.__new__(cls)
        labels = np.asarray(column_labels, dtype=np.int64)
        self.n_cg, self.n_fg = int(n_cg), int(labels.size)
        self.out_f32, self.sparse, self.slice = False, False, False
        sizes = np.bincount(labels, minlength=n_labels)
        order = np.argsort(sizes, kind="stable")
        if self.n_cg > 64:  # packed-panel GEMM path: unique columns follow their first site (see __init__)
            first = np.full(n_labels, self.n_fg, dtype=np.int64)
            np.minimum.at(first, labels, np.arange(self.n_fg))
            order = np.argsort(first, kind="stable")
        rank = np.empty_like(order)
        rank[order] = np.arange(order.size)
        ptr_, sites = csr_from_labels(rank[labels], n_labels)
        self.n_ucol, self.nnz = int(n_labels), int(sites.size)
        self.ucol_ptr, self.ucol_sites = dev_i32(ptr_), dev_i32(sites)
        self.umat_t = None  # filled per fit: see with_values
        return self, rank

    def weights_finite(self) -> bool:
        """The int8 application needs finite coefficients (a NaN / inf weight has no fixed-point digits; the
        float64 kernels propagate it like numpy).  Host matrices are checked when compiled; a device fit is
        checked when it is solved (``solve_equality_qp_device`` / ``agf_qp_equality_small`` decline otherwise)."""
        return bool(getattr(self, "_finite", True))

    def with_values(self, umat_t: torch.Tensor) -> "CompiledMap":
        """A map sharing this one's (immutable) structure with its own coefficient operand."""
        import copy

        other = copy.copy(self)
        other.umat_t = umat_t
        return other


def map_apply(frames: Frames, cmap: CompiledMap, nan_mode: int, nan_atol: float, want_sumsq: bool = False,
              start: int = 0, stop: Optional[int] = None, sumsq: Optional[torch.Tensor] = None,
              flags: Optional[torch.Tensor] = None, download: Optional[list] = None
              ) -> Tuple[torch.Tensor, Optional[torch.Tensor], torch.Tensor]:
    """Kernel (d).  Returns ``(out [T, n_cg, 3] device, sumsq device f64[1] | None, nan_flags int32[2])``.
    ``sumsq`` / ``flags``: zeroed slots of a caller-owned status buffer to accumulate into.
    ``download``: an empty list; for a host array the pinned copy of ``out`` is started here -- piece by
    piece behind each piece's kernel when the array is still being uploaded -- and appended to it
    (``finish_d2h`` before reading)."""
    if frames.n_sites != cmap.n_fg:
        raise ValueError(
            f"map expects {cmap.n_fg} fine-grained sites but the array has {frames.n_sites}"
        )
    stop = frames.n_frames if stop is None else stop
    out_dtype = torch.float32 if (cmap.out_f32 and frames.np_dtype == np.float32) else torch.float64
    out = torch.empty((stop - start, cmap.n_cg, 3), dtype=out_dtype, device=device())
    if sumsq is None:
        sumsq = torch.zeros(1, dtype=torch.float64, device=device()) if want_sumsq else None
    if flags is None:
        flags = torch.zeros(2, dtype=torch.int32, device=device())
    host_out = None
    by_piece = download is not None and frames.on_host and frames._dev is None
    if by_piece:
        host_out = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
    for t0, piece in frames.pieces(start, stop):
        o = out[t0 - start : t0 - start + piece.shape[0]]
        if cmap.sparse and cmap.slice:
            _lib.call("agf_map_apply_slice", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites,
                      ptr(cmap.row_sites), ptr(cmap.row_w), cmap.n_cg, ptr(o), dtype_code(o), ptr(sumsq), nan_mode,
                      float(nan_atol), ptr(flags), stream_ptr())
        elif cmap.sparse:
            _lib.call("agf_map_apply_sparse", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites,
                      ptr(cmap.row_ptr), ptr(cmap.row_sites), ptr(cmap.row_w), cmap.n_cg, ptr(o), dtype_code(o),
                      ptr(sumsq), nan_mode, float(nan_atol), ptr(flags), stream_ptr())
        else:
            need = int(_lib.lib().agf_map_apply_workspace_bytes(dtype_code(piece), frames.n_sites, cmap.n_ucol,
                                                                cmap.nnz, cmap.n_cg, piece.shape[0]))
            need_i8 = 0
            if (need > 0 and _GRAM_I8[0] and piece.dtype == torch.float32 and cmap.n_cg > 64
                    and piece.shape[0] >= _GRAM_I8T_MIN_FRAMES and cmap.weights_finite()):
                need_i8 = int(_lib.lib().agf_map_apply_i8_workspace_bytes(frames.n_sites, cmap.n_ucol, cmap.n_cg,
                                                                          piece.shape[0]))
            if need_i8 > 0:  # int8 digit planes on tcgen05 (csrc/apply_i8.cu)
                ws = workspace(need_i8)
                _lib.call("agf_map_apply_i8", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites,
                          ptr(cmap.ucol_ptr), ptr(cmap.ucol_sites), cmap.n_ucol, ptr(cmap.umat_t), cmap.n_cg, ptr(o),
                          dtype_code(o), ptr(sumsq), nan_mode, float(nan_atol), ptr(flags), ptr(ws),
                          C.c_size_t(ws.numel()), stream_ptr())
            elif need > 0:  # too large for the shared-memory resident kernel: packed-panel DMMA GEMM
                ws = workspace(need)
                _lib.call("agf_map_apply_ws", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites,
                          ptr(cmap.ucol_ptr), ptr(cmap.ucol_sites), cmap.n_ucol, cmap.nnz, ptr(cmap.umat_t),
                          cmap.n_cg, ptr(o), dtype_code(o), ptr(sumsq), nan_mode, float(nan_atol), ptr(flags),
                          ptr(ws), C.c_size_t(ws.numel()), stream_ptr())
            else:
                _lib.call("agf_map_apply", ptr(piece), dtype_code(piece), piece.shape[0], frames.n_sites,
                          ptr(cmap.ucol_ptr), ptr(cmap.ucol_sites), cmap.n_ucol, cmap.nnz, ptr(cmap.umat_t),
                          cmap.n_cg, ptr(o), dtype_code(o), ptr(sumsq), nan_mode, float(nan_atol), ptr(flags),
                          stream_ptr())
        if by_piece:
            start_d2h_piece(host_out, t0 - start, o)
    if download is not None and frames.on_host:
        download.append(host_out if by_piece else start_d2h(out))
    return out, sumsq, flags


def merge_moments(parts: Sequence[np.ndarray], n_pairs: int) -> np.ndarray:
    """Population sd per pair from per-rank ``[count, mean(P), M2(P)]`` records (Chan's pairwise
    update in float64); NaN moments stay NaN."""
    cnt, mu, m2t = 0.0, np.zeros(n_pairs), np.zeros(n_pairs)
    for part in parts:
        tb, mb, m2b = part[0], part[1 : 1 + n_pairs], part[1 + n_pairs :]
        if tb == 0:
            continue
        delta = mb - mu
        tot = cnt + tb
        m2t = m2t + m2b + delta * delta * cnt * tb / tot
        mu = mu + delta * tb / tot
        cnt = tot
    with np.errstate(invalid="ignore"):
        sd = np.sqrt(np.maximum(m2t, 0.0) / cnt)
    sd[np.isnan(m2t)] = np.nan
    return sd


_SCREEN_FRAMES = 32
_RESCREEN_FRAMES = 4096
_SELECT_CAP = 8192  # survivor capacity of the one-kernel compaction (small systems)


def _screen_frames(t_est_total: float, threshold: float, t_local: int) -> int:
    """Frames of the literal all-pairs screen.  A flexible pair is pruned once its partial sum of squared
    deviations exceeds threshold^2 * T_total, which grows with the trajectory: 32 frames are enough up
    to about a million frames at the default threshold; longer (e.g. sharded) trajectories get a
    proportionally longer prefix, so that the survivors are the O(n) rigid pairs and no second pruning
    pass (with its extra collective) is needed."""
    want = _SCREEN_FRAMES * max(1.0, threshold * threshold * t_est_total / 1.0)
    return int(min(t_local, min(512, int(np.ceil(want / 32.0)) * 32)))


def pair_constraints(frames: Frames, other: Optional[Frames], threshold: float):
    """Kernel (c) with exact progressive pruning.  Returns ``(pairs int64 [P, 2], sd float64 [P])``
    for every pair that survived pruning (the caller applies ``sd < threshold``)."""
    if other is not None and other.n_frames != frames.n_frames:
        raise ValueError("xyz and cross_xyz must have the same number of frames")
    n, n_o = frames.n_sites, (frames.n_sites if other is None else other.n_sites)
    t_local = frames.n_frames
    empty = (np.zeros((0, 2), dtype=np.int64), np.zeros(0))
    # Under frame sharding with a small pair matrix the global frame count travels with the screening
    # statistics (one MAX exchange of [M2 | per-rank counts], no separate count round trip).
    fused = sharded() and n * n_o <= (1 << 16) - 64 and _dist().get_backend(_Sharding.group) == "nccl"
    t_total = None if fused else global_count(t_local)
    if not fused and (t_total == 0 or t_local == 0 and not sharded()):
        return empty
    # a pair can only be a constraint if  M2_total <= thr^2 * T  (var = M2 / T < thr^2); partial
    # M2 never exceeds the total, so anything above the (slightly widened) bound is pruned for good.
    bound = None if fused else float(threshold) ** 2 * t_total * (1.0 + 1e-6) + 1e-300
    dev = device()
    world = _dist().get_world_size(_Sharding.group) if sharded() else 1

    def other_piece(piece_t0: int, count: int) -> Optional[torch.Tensor]:
        # the frames matching a piece of `frames`: a host cross array too large to keep resident is
        # uploaded range by range, as `frames` itself is
        if other is None:
            return None
        return other.frame_range(piece_t0, count)

    # ---- stage 0: literal all-pairs pass over a short prefix
    n0 = _screen_frames(float(t_total if t_total is not None else world * t_local), float(threshold), t_local)
    x0 = o0 = None
    n_mat = n_o * n
    buf = torch.empty(n_mat + (world if fused else 0), dtype=torch.float64, device=dev)
    m2 = buf[:n_mat].view(n_o, n)
    if n0 > 0:
        x0 = frames.prefix(n0)
        o0 = None if other is None else other.prefix(n0)
        if o0 is not None and o0.dtype != x0.dtype:
            o0 = o0.to(x0.dtype)
        _lib.call("agf_pair_screen", ptr(x0), ptr(o0), dtype_code(x0), n0, n, n_o, ptr(m2), stream_ptr())
    elif fused:  # a rank without frames constrains nothing: zeros under the MAX (inf below the diagonal)
        m2.zero_()
        if other is None:
            m2.copy_(torch.where(torch.triu(torch.ones_like(m2), diagonal=1) > 0, m2, torch.full_like(m2, float("inf"))))
    else:
        m2.fill_(float("inf"))
    counts_dev = None
    if fused:
        rank = _dist().get_rank(_Sharding.group)
        mine = np.zeros(world)
        mine[rank] = float(t_local)
        buf[n_mat:].copy_(_dev_cached(mine))  # cached: the same shard sizes come back every call
        allreduce_max_(buf)
        counts_dev = buf[n_mat:]
    pairs = shift = acc = pairs_host = None
    if n0 > 0 and n_mat <= (1 << 18) and (fused or not sharded()):
        # small systems: ONE kernel turns the screened matrix into the ordered survivor list, their
        # frame-0 distances and zeroed accumulators; one small read returns the count and the list
        cap = min(n_mat, _SELECT_CAP)
        ints = torch.empty(1 + 2 * cap, dtype=torch.int32, device=dev)
        fl = torch.empty(3 * cap, dtype=torch.float64, device=dev)
        _lib.call("agf_pair_select", ptr(m2), float(threshold) ** 2 if fused else bound, ptr(counts_dev), world if fused else 0,
                  ptr(x0), ptr(o0), dtype_code(x0), n, n_o, cap, ptr(ints[1:]), ptr(fl), ptr(fl[cap:]), ptr(ints),
                  stream_ptr())
        host_ints = to_host(ints)
        n_pairs = int(host_ints[0])
        if n_pairs == 0:
            return empty
        if n_pairs > 0:
            pairs_host = host_ints[1 : 1 + 2 * n_pairs].reshape(-1, 2).astype(np.int64)
            pairs = ints[1 : 1 + 2 * n_pairs].view(n_pairs, 2)
            shift, acc = fl[:n_pairs], fl[cap : cap + 2 * n_pairs].view(n_pairs, 2)
    bound_dev = None
    if pairs is None:  # general path (large systems, or more survivors than the capacity)
        if fused:
            bound_dev = (float(threshold) ** 2 * counts_dev.sum() * (1.0 + 1e-6) + 1e-300).reshape(1)
            alive = m2 <= bound_dev
        else:
            if n0 > 0:
                alive = (m2 <= bound).to(torch.uint8)
            else:
                alive = torch.ones((n_o, n), dtype=torch.uint8, device=dev)
                if other is None:
                    alive = torch.triu(alive, diagonal=1)
            allreduce_min_(alive)
        pairs = torch.nonzero(alive).to(torch.int32).contiguous()  # [P, 2] = (i over other, j over xyz)
        del alive
        n_pairs = int(pairs.shape[0])
        if n_pairs == 0:
            return empty
        shift = torch.zeros(n_pairs, dtype=torch.float64, device=dev)
        if t_local > 0:
            xf = frames.prefix(1)
            of_ = None if other is None else other.prefix(1).to(xf.dtype)
            _lib.call("agf_pair_first", ptr(xf), ptr(of_), dtype_code(xf), n, n_o, ptr(pairs), n_pairs, ptr(shift),
                      stream_ptr())
        acc = torch.zeros((n_pairs, 2), dtype=torch.float64, device=dev)

    # ---- stage 1..: stream all frames for the survivors
    def run(a: int, b: int) -> None:
        for t0, piece in frames.pieces(a, b):
            o = other_piece(t0, piece.shape[0])
            if o is not None and o.dtype != piece.dtype:
                o = o.to(piece.dtype)
            _lib.call("agf_pair_moments", ptr(piece), ptr(o), dtype_code(piece), piece.shape[0], n, n_o,
                      ptr(pairs), int(pairs.shape[0]), ptr(shift), ptr(acc), stream_ptr())

    # second pruning point after a few thousand frames: bounds the survivor count for flexible
    # molecules (at n = 5000 the screen leaves ~10^5 pairs, 4096 frames leave the bonded ones).  Under
    # sharding every rank holds the same pair list and a pair dead on any rank is dead globally
    # (M2_global >= M2_rank), so the keep masks are combined with one MIN all-reduce; the branch depends
    # on the (global) pair count only, so all ranks take it together.
    done = 0
    if n_pairs > 4 * max(n, n_o) and (sharded() or t_local > 4 * _RESCREEN_FRAMES):
        done = min(_RESCREEN_FRAMES, t_local)
        run(0, done)
        if fused and bound_dev is None:
            bound_dev = (float(threshold) ** 2 * counts_dev.sum() * (1.0 + 1e-6) + 1e-300).reshape(1)
        if done > 0:
            m2p = acc[:, 1] - acc[:, 0] ** 2 / done
            keep_mask = m2p <= (bound_dev if fused else bound)
        else:
            keep_mask = torch.ones(n_pairs, dtype=torch.bool, device=dev)
        if sharded():
            km = keep_mask.to(torch.uint8)
            allreduce_min_(km)
            keep_mask = km > 0
        keep = torch.nonzero(keep_mask).reshape(-1)
        pairs, shift, acc = pairs[keep].contiguous(), shift[keep].contiguous(), acc[keep].contiguous()
        pairs_host = None
        n_pairs = int(pairs.shape[0])
        if n_pairs == 0:
            return empty
    run(done, t_local)

    # ---- per-rank (count, shift, running sums) go to the host as they are -- gathered across ranks
    #      under sharding -- and the moments are formed and merged (Chan) there in float64; P is O(n).
    #      One synchronising read.
    def record(t_cnt: float, sh: np.ndarray, ac: np.ndarray) -> np.ndarray:
        with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
            d = max(t_cnt, 1.0)
            return np.concatenate([[t_cnt], sh + ac[:, 0] / d, ac[:, 1] - ac[:, 0] ** 2 / d])

    if not sharded():
        want = [shift, acc] if pairs_host is not None else [shift, acc, pairs]
        got = read_many(want)
        if pairs_host is None:
            pairs_host = got[2].astype(np.int64)
        return pairs_host.reshape(-1, 2), merge_moments([record(float(t_local), got[0], got[1])], n_pairs)
    packed = torch.cat([_dev_cached(np.array([float(t_local)])), shift, acc.reshape(-1)])
    gathered = allgather_dev(packed)
    want = [gathered] if pairs_host is not None else [gathered, pairs]
    got = read_many(want)
    if pairs_host is None:
        pairs_host = got[1].astype(np.int64)
    parts = [record(float(row[0]), row[1 : 1 + n_pairs], row[1 + n_pairs :].reshape(n_pairs, 2)) for row in got[0]]
    return pairs_host.reshape(-1, 2), merge_moments(parts, n_pairs)
