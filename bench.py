#!/usr/bin/env python
"""Benchmark of the force-map fit+apply hot path (BASELINE.json metric: frames/s).

Workload (BASELINE.json configs[1]): a synthetic replica of chignolin (cln025: 175 atoms,
10 C-alpha beads, 78 X-H constraints -> 97 reduced columns), 1 M frames per GPU.  One
"step" is one pass of the whole path over those frames:

    constraints = guess_pairwise_constraints(coords)                        # kernel (c), all frames
    project_forces(..., method=constraint_aware_uni_map)                    # kernel (d) x2
    project_forces(..., method=qp_linear_map, l2_regularization=1e3)        # kernel (a) + QP + (d) x2

  value : frames/s with inputs resident in HBM (torch CUDA tensors in, CUDA tensors out)
  e2e   : the same calls on pinned HOST arrays; every step uploads coords+forces once and reads
          all four mapped arrays back (numpy out)
  N > 1 : every rank owns its own 1 M frames (weak scaling); Gram and pair moments are
          all-reduced (NCCL), the map is applied locally.  `parity` compares a sharded fit with the
          single-GPU fit of the same global frames.
  configs : short probes of BASELINE configs 3 (featurised fit), 4 (5 000 atoms / 500 beads /
          n_red 2 600) and 5 (joptgauss_map, 2 000 atoms / 200 beads) with per-kernel times and
          roofline fractions, so that those numbers are taken under the driver's clock too.
  peaks : the FP64 DMMA issue rate and a streaming read bandwidth, measured in this run
          (agf_probe_dmma / agf_probe_read); the HBM copy peak comes from MEASURED_PEAKS.json.

`--impl reference` times the REFERENCE's own code (`oracle/_ref`, an unmodified copy of its Python
package made by `oracle/make_ref.py`, behind the exact-solve `qpsolvers` stand-in) on a bounded frame
sample with all host threads; the float64 numpy port in `oracle/` is the fallback when the copy is
absent.

`--dump-outputs DIR` writes what the last timed step returned (rank 0's share) as `DIR/<name>.npy`, so
that two builds can be compared output for output on the same seeded inputs: the constraint set, both
fitted force maps and residuals, and the four mapped arrays on a fixed sample of frames (`frames.npy`).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from

METRIC = "frames/sec through force-map fit+apply"
UNIT = "frames/s"
L2_REG = 1e3
KBT = 0.6955215
# frames of each mapped array written by --dump-outputs: 4 arrays x 32 768 frames x 10 beads x 3 x 8 B = 31 MB
DUMP_FRAMES = 32_768
DUMP_LIMIT_BYTES = 64 << 20


def _at_least_one(text: str) -> int:
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {n}")
    return n


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_at_least_one, default=5, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=1_000_000, help="frames per GPU")
    ap.add_argument("--cpu-frames", type=int, default=4000, help="frames of the CPU sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the config 3/4/5 probes")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# ----------------------------------------------------------------------------- CPU arm
def _cpu_data(n_frames: int):
    from aggforce_b200.synth import chignolin_topology, synth_trajectory_host

    topo = chignolin_topology()
    coords, forces = synth_trajectory_host(topo, n_frames, seed=1234)
    return topo, coords, forces


def cpu_run(n_frames: int, steps: int, warmup: int):
    """Times the config-2 step on the host cores.  Returns (frames/s, s per step, kind, description)."""
    from oracle import make_ref

    topo, coords, forces = _cpu_data(n_frames)
    ref = make_ref.load()
    if ref is not None:
        # the reference's own functions, float32 input as in its shipped datasets
        from aggforce.qp import constraint_aware_uni_map  # noqa: PLC0415  (oracle/_ref)

        cmap = ref.LinearMap([[i] for i in topo.bead_atoms], n_fg_sites=topo.n_sites)

        def step():
            cons = ref.guess_pairwise_constraints(coords)
            ref.project_forces(coords=coords, forces=forces, coord_map=cmap, constrained_inds=cons,
                               method=constraint_aware_uni_map)
            return ref.project_forces(coords=coords, forces=forces, coord_map=cmap, constrained_inds=cons,
                                      l2_regularization=L2_REG)["residual"]

        kind = "reference"
        what = ("the reference's own guess_pairwise_constraints + project_forces(constraint_aware_uni_map) + "
                "project_forces(qp_linear_map, l2=1e3) from oracle/_ref (unmodified copy of its package; "
                "qpsolvers replaced by the exact equality-QP solve)")
    else:
        import oracle

        cm = np.zeros((len(topo.bead_atoms), topo.n_sites))
        cm[np.arange(len(topo.bead_atoms)), topo.bead_atoms] = 1

        def step():
            cons = oracle.guess_pairwise_constraints_literal(coords)
            uni = oracle.uni_map_matrix(cm, cons)
            oracle.apply_map(coords, cm), oracle.apply_map(forces, uni)
            w = oracle.qp_linear_weights(forces, cm, cons, L2_REG)
            oracle.apply_map(coords, cm)
            return oracle.force_smoothness(oracle.apply_map(forces, w))

        kind = "port"
        what = "float64 numpy port of the reference lines (oracle/; oracle/_ref is absent)"
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(1, steps)
    return n_frames / dt, dt, kind, what


def reference_arm(args) -> None:
    if int(os.environ.get("RANK", "0")) != 0:
        return
    value, dt, kind, what = cpu_run(args.cpu_frames, args.steps, args.warmup)
    cores = os.cpu_count() or 1
    sample = (f"{args.cpu_frames} frames of the same synthetic cln025 workload per step; {what}; "
              "BLAS threads = all cores")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.cpu_frames),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(line)


def workload_config(frames_per_gpu: int) -> dict:
    return {
        "workload": "cln025 (175 atoms, 10 CA beads, 78 X-H constraints -> n_red 97): "
                    "guess_pairwise_constraints(all frames) + constraint_aware_uni_map + optimised "
                    "qp_linear_map(l2=1e3) via project_forces, synthetic replica",
        "frames_per_gpu": frames_per_gpu,
        "cache": "inputs (2.1 GB per array per GPU) are larger than L2; no explicit flush",
    }


def step_outputs(cons, r_uni, r_opt, n_frames: int) -> dict:
    """What one step hands its caller, as host float32 / float64 arrays: the constraint set (sorted site
    pairs), each map's force matrix and residual, and the mapped arrays on a fixed, seeded sample of frames."""
    import torch

    frames = np.sort(np.random.default_rng(0).choice(n_frames, size=min(n_frames, DUMP_FRAMES), replace=False))
    out = {"frames": frames.astype(np.float64),
           "constraints": np.array(sorted(sorted(p) for p in cons), dtype=np.float64).reshape(-1, 2)}
    for tag, res in (("uni", r_uni), ("opt", r_opt)):
        out[f"{tag}_force_map"] = np.asarray(res["tmap"].force_map.standard_matrix, dtype=np.float64)
        out[f"{tag}_residual"] = np.array([res["residual"]], dtype=np.float64)
        for key in ("mapped_coords", "mapped_forces"):
            arr = torch.as_tensor(res[key])
            sample = arr.index_select(0, torch.as_tensor(frames, device=arr.device)).cpu().numpy()
            out[f"{tag}_{key}"] = sample if sample.dtype == np.float32 else sample.astype(np.float64)
    return out


def dump_outputs(outputs: dict, where: Path) -> None:
    total = sum(a.nbytes for a in outputs.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs would write {total} bytes"
    where.mkdir(parents=True, exist_ok=True)
    for name, arr in outputs.items():
        np.save(where / f"{name}.npy", arr)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self) -> None:
        assert self.proc is not None and self.proc.stdout is not None
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- GPU arm
_REAL_STDOUT = None


def _quiet_stdout() -> None:
    """The contract is ONE JSON line on stdout: route everything libraries print to fd 1 (NCCL's
    version banner, ...) to stderr and keep the real stdout for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def _emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def measure_peaks(torch, _lib, _engine) -> dict:
    """FP64 DMMA issue rate and streaming read bandwidth, measured now (CUDA events, best of 5)."""
    import ctypes as C

    sms = int(_lib.lib().agf_device_sm_count())
    sink = torch.empty(sms * 8 * 256, dtype=torch.float64, device="cuda")
    flop = C.c_int64(0)
    buf = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")  # 1 GiB: far larger than L2
    buf.zero_()
    fsink = torch.zeros(4, dtype=torch.float32, device="cuda")

    def best(fn, n=5):
        fn()
        torch.cuda.synchronize()
        out = []
        for _ in range(n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return min(out)

    ms_d = best(lambda: _lib.check(_lib.lib().agf_probe_dmma(20000, _engine.ptr(sink), C.byref(flop),
                                                             _engine.stream_ptr()), "agf_probe_dmma"))
    ms_r = best(lambda: _lib.check(_lib.lib().agf_probe_read(_engine.ptr(buf), buf.numel(), _engine.ptr(fsink),
                                                             _engine.stream_ptr()), "agf_probe_read"))
    del buf
    return {"fp64_dmma_tflops": flop.value / (ms_d * 1e-3) / 1e12, "read_gbs": (1 << 30) / (ms_r * 1e-3) / 1e9,
            "how": "agf_probe_dmma: 8 independent DMMA.8x8x4 accumulator tiles per warp, 8 CTAs x 8 warps per SM, "
                   "20 000 iterations; agf_probe_read: one float4 streaming read of 1 GiB; CUDA events, best of 5"}


def kernel_table(per_kernel: dict, algo: dict, peaks: dict, hbm_peak: float, traffic: dict) -> dict:
    """{entry point: {launches, ms_total, bound, achieved, peak, unit, frac, traffic}}; ``algo`` maps an
    entry point to (bound, algorithmic flop or bytes summed over its launches)."""
    out = {}
    for name, times in per_kernel.items():
        tot = float(np.sum(times))
        entry = {"launches": len(times), "ms_total": tot}
        if name in algo and tot > 0:
            kind, amount = algo[name]
            if kind == "tensor":
                entry.update(bound="tensor", achieved=amount / (tot * 1e-3) / 1e12, peak=peaks["fp64_dmma_tflops"],
                             unit="TFLOP/s")
            else:
                entry.update(bound="hbm", achieved=amount / (tot * 1e-3) / 1e9, peak=hbm_peak, unit="GB/s")
            entry["frac"] = entry["achieved"] / entry["peak"]
        if name in traffic:
            entry["traffic"] = traffic[name]
        out[name] = entry
    return out


INT8_NOMINAL_TOPS = 4500.0  # dense int8 tensor peak of one B200 (datasheet; no int8 probe runs inside the bench)


def tiled_gram_note(entry: dict, n_red: int, n_frames: int, batch: int = 1) -> None:
    """agf_gram_linear_i8t: `achieved` stays the float64-EQUIVALENT rate against the FP64 DMMA peak (the roof
    of the formulation it replaces); the kernel's own roof is the int8 tensor pipe, reported next to it."""
    if not entry or entry.get("ms_total", 0) <= 0:
        return
    n_mb, n_nb = -(-n_red // 128), -(-n_red // 96)
    tiles = sum(n_nb - (128 * mi) // 96 for mi in range(n_mb))
    ops = 2.0 * 15 * batch * tiles * 128 * 96 * 3 * n_frames  # n_frames: all frames of the call, over all its launches
    entry["int8_tops"] = ops / (entry["ms_total"] * 1e-3) / 1e12
    entry["int8_peak_tops"] = INT8_NOMINAL_TOPS
    entry["int8_frac"] = entry["int8_tops"] / INT8_NOMINAL_TOPS
    entry["note"] = ("float64 Gram through five int8 digit planes on tcgen05 (tiled, TMEM accumulators): `achieved` "
                     "is float64-equivalent flop/s against the FP64 DMMA peak of the formulation it replaces (so "
                     "frac > 1 is the point); int8_* is the executed int8 work (15 plane products over the 128 x 96 "
                     "tiles of the upper block-triangle, digit conversion included in the time) against the nominal "
                     "dense int8 peak")


def main() -> None:
    args = parse()
    _quiet_stdout()
    if args.impl == "reference":
        reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    import aggforce_b200 as agf
    from aggforce_b200 import _engine, _lib
    from aggforce_b200.synth import chignolin_topology, protein_like_topology, synth_trajectory_device

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    T = args.frames
    topo = chignolin_topology()
    cmap = agf.LinearMap([[i] for i in topo.bead_atoms], n_fg_sites=topo.n_sites)
    peaks = measure_peaks(torch, _lib, _engine)
    coords, forces = synth_trajectory_device(topo, T, seed=1234, frame0=rank * T)
    torch.cuda.synchronize()

    def step(c, f):
        cons = agf.guess_pairwise_constraints(c)
        r1 = agf.project_forces(coords=c, forces=f, coord_map=cmap, constrained_inds=cons,
                                method=agf.constraint_aware_uni_map)
        r2 = agf.project_forces(coords=c, forces=f, coord_map=cmap, constrained_inds=cons,
                                l2_regularization=L2_REG)
        return cons, r1, r2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sample_clocks=False):
        # the sampler runs across warm-up AND the timed steps: the timed region alone lasts tens of
        # milliseconds, less than one nvidia-smi sampling period
        sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None  # one nvidia-smi poller per box
        done, t_w = 0, time.perf_counter()
        # at least `warmup` steps, and the same load kept up until the poller has delivered its first sample
        # (nvidia-smi needs ~0.1-0.3 s to start), so that the samples bracket the timed steps under load;
        # rank 0 (the one with the poller) decides for everybody: the steps carry collectives
        while True:
            more = done < warmup or (sampler is not None and sampler.proc is not None and not sampler.rows
                                     and time.perf_counter() - t_w < 3.0)
            if world > 1:
                flag = torch.tensor([1 if more else 0], device="cuda", dtype=torch.int32)
                dist.broadcast(flag, 0)
                more = bool(flag.item())
            if not more:
                break
            fn()
            done += 1
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _lib.LAUNCHES["count"]
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()  # what the last timed step returned (earlier results are dropped as they come)
        e1.record()
        barrier()
        launches = _lib.LAUNCHES["count"] - n0
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        clocks = None
        if sampler is not None:
            # the step function does not communicate outside frame_sharding(), so rank 0 may keep its GPU under
            # the same load alone until two more samples have arrived (untimed; at most one second)
            have, t_a = len(sampler.rows), time.perf_counter()
            while (world == 1 and sampler.proc is not None and len(sampler.rows) < have + 2
                   and time.perf_counter() - t_a < 1.0):
                fn()
            clocks = sampler.stop()
        return float(ms.item()) / steps, launches, clocks, last

    def kernel_times(fn):
        """{entry point: [ms per call]} of one extra pass (CUDA events on the launching stream)."""
        _lib.timing(True)
        fn()
        per = {}
        for name, ms in _lib.timing_records():
            per.setdefault(name, []).append(ms)
        _lib.timing(False)
        return per

    peaks_path = ROOT / "MEASURED_PEAKS.json"
    hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    if peaks_path.exists():
        hbm_peak, hbm_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    traffic_path = ROOT / "profiles" / "r02_traffic.json"  # dram bytes per launch from an ncu --set full capture
    traffic = json.loads(traffic_path.read_text()).get("per_launch_bytes", {}) if traffic_path.exists() else {}

    configs, parity, h2d_probe = {}, None, None
    ctx = agf.frame_sharding(world > 1)
    with ctx:
        # ---- device-resident throughput
        ms_dev, launches, clocks, last = timed(lambda: step(coords, forces), args.steps, args.warmup,
                                               sample_clocks=True)
        if args.dump_outputs is not None and rank == 0:
            dump_outputs(step_outputs(*last, T), args.dump_outputs)
        del last
        per_kernel = kernel_times(lambda: step(coords, forces))

        # ---- end to end from pinned host memory
        e2e = None
        if not args.no_e2e:
            hc = torch.empty(coords.shape, dtype=coords.dtype, pin_memory=True)
            hf = torch.empty(forces.shape, dtype=forces.dtype, pin_memory=True)
            hc.copy_(coords)
            hf.copy_(forces)
            torch.cuda.synchronize()
            nc, nf = hc.numpy(), hf.numpy()
            d2h = {"n": 0}

            def host_step():
                c, f = agf.Frames(nc), agf.Frames(nf)  # fresh wrappers: uploaded once per step
                _, r1, r2 = step(c, f)
                d2h["n"] = sum(r[k].nbytes for r in (r1, r2) for k in ("mapped_coords", "mapped_forces"))

            ms_e2e, _, _, _ = timed(host_step, args.steps, 3)
            # what the host side can deliver: all ranks upload their pinned coordinate array at once
            dst = torch.empty_like(coords)

            def upload():
                dst.copy_(hc, non_blocking=True)

            ms_up, _, _, _ = timed(upload, 3, 1)
            h2d_probe = world * hc.numel() * 4 / (ms_up * 1e-3) / 1e9
            del dst
            moved = int(nc.nbytes + nf.nbytes)
            e2e = {"value": world * T / (ms_e2e * 1e-3), "unit": UNIT,
                   "h2d_bytes_per_step": moved, "d2h_bytes_per_step": int(d2h["n"]),
                   "ms_per_step": ms_e2e, "h2d_probe_gbs": h2d_probe,
                   "h2d_gbs_achieved": world * moved / (ms_e2e * 1e-3) / 1e9,
                   "frac_of_h2d_probe": (world * moved / (ms_e2e * 1e-3) / 1e9) / h2d_probe,
                   "h2d_probe": "all ranks copy their pinned 2.1 GB coordinate array to the device at the same "
                                "time (aggregate GB/s): the host-side ceiling of the end-to-end number"}
            del hc, hf, nc, nf

        # ---- probes of BASELINE configs 3, 4, 5 (short, same clock; sharded like the main workload)
        if not args.no_configs:
            configs = config_probes(agf, _engine, _lib, torch, dist, rank, world, peaks, hbm_peak, kernel_times,
                                    topo, cmap, protein_like_topology, synth_trajectory_device)
    if world > 1:
        parity = sharded_parity(agf, torch, dist, rank, world, topo, cmap, synth_trajectory_device)

    # ---- roofline of the dominant kernel (algorithmic work per launch / measured time)
    n, n_red, n_cg = topo.n_sites, 97, len(topo.bead_atoms)
    uni_nnz = 21
    launches_of = {k: len(v) for k, v in per_kernel.items()}
    algo = {  # summed over the launches of one step
        "agf_gram_linear": ("tensor", (3 * n_red * (n_red + 1) + 3 * n) * T * launches_of.get("agf_gram_linear", 1)),
        # the int8 / tcgen05 kernel computes the same float64 Gram: same algorithmic flops, quoted against the
        # FP64 tensor roof it replaces (its own int8 roof, 3.4 POP/s measured by tools/ozaki/i8_syrk_probe.cu,
        # is 40x away; see kernels[...]["note"])
        "agf_gram_linear_i8": ("tensor", (3 * n_red * (n_red + 1) + 3 * n) * T * launches_of.get("agf_gram_linear_i8", 1)),
        "agf_pair_moments": ("hbm", 12 * n * T * launches_of.get("agf_pair_moments", 1)),
        "agf_map_apply": ("hbm", (12 * n + 24 * n_cg) * T * launches_of.get("agf_map_apply", 1)),
        # slice: the coordinate map of both project_forces calls (10 sites); sparse: the uniform force map
        # (21 nnz).  Algorithmic bytes = referenced sites (12 B each) + f64 outputs
        "agf_map_apply_slice": ("hbm", (n_cg * 12 + 24 * n_cg) * T * launches_of.get("agf_map_apply_slice", 1)),
        "agf_map_apply_sparse": ("hbm", (uni_nnz * 12 + 24 * n_cg) * T * launches_of.get("agf_map_apply_sparse", 1)),
    }
    kernels = kernel_table(per_kernel, algo, peaks, hbm_peak, traffic)
    if "agf_gram_linear_i8" in kernels:
        k8 = kernels["agf_gram_linear_i8"]
        k8["hbm_gbs"] = 12 * n * T * k8["launches"] / (k8["ms_total"] * 1e-3) / 1e9
        k8["hbm_frac"] = k8["hbm_gbs"] / hbm_peak
        k8["note"] = ("float64 Gram through int8 digit planes on tcgen05 (TMEM accumulators): `achieved` is "
                      "float64-EQUIVALENT flop/s (algorithmic flops of the float64 Gram / time) against the FP64 "
                      "DMMA peak that bounds the FP64 formulation; the kernel itself is bounded by its digit "
                      "fill, not by the int8 tensor pipe (about 25 % active) nor by HBM (hbm_frac)")
    dominant = max(kernels, key=lambda k: kernels[k]["ms_total"]) if kernels else None
    roofline = None
    if dominant and "frac" in kernels[dominant]:
        k = kernels[dominant]
        roofline = {"kernel": dominant, "bound": k["bound"], "achieved": k["achieved"], "peak": k["peak"],
                    "unit": k["unit"], "frac": k["frac"], "traffic": k.get("traffic"),
                    "peak_source": ("FP64 DMMA issue rate measured in this run (agf_probe_dmma)"
                                    if k["bound"] == "tensor" else hbm_src),
                    "traffic_source": "profiles/r02_traffic.json (ncu --set full, dram__bytes_read.sum + "
                                      "dram__bytes_write.sum per launch)" if k.get("traffic") else None}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, dt, kind, what = cpu_run(args.cpu_frames, 3, 1)
        cpu = {"value": v, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": kind,
               "sample": f"{args.cpu_frames} frames of the same workload, 3 timed steps ({dt:.2f} s each); {what}; "
                         "BLAS threads = all cores"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": world * T / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(T), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "gpu_launches_note": "C-ABI entry calls of libagf_b200.so inside the timed region (each launches "
                                 "one to three kernels)",
            "roofline": roofline, "kernels": kernels, "peaks": dict(peaks, hbm_copy_gbs=hbm_peak, hbm_source=hbm_src),
            "cpu_baseline": cpu, "configs": configs, "parity": parity,
        }
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def config_probes(agf, _engine, _lib, torch, dist, rank, world, peaks, hbm_peak, kernel_times, topo, cmap,
                  protein_like_topology, synth_trajectory_device) -> dict:
    """Short runs of BASELINE configs 3, 4 and 5: wall time of the public call (CUDA events, max over
    ranks, median of three calls after one warm-up call) and the roofline fraction of every kernel with a
    defined algorithmic cost."""
    from aggforce_b200.qp import Multifeaturize, gb_feat, id_feat, qp_feat_linear_map
    from aggforce_b200.qp.qplinear import reduced_columns
    from aggforce_b200.util import Curry

    def wall(fn):
        fn()  # warm-up (workspace allocation, map compilation)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        times, out = [], None
        for _ in range(3):  # median of three timed calls (max over ranks each): one hiccup does not make the number
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            times.append(float(ms.item()))
        return float(np.median(times)), out

    out = {}
    # ---- config 3: featurised fit, cln025, id_feat + gb_feat(0, 8, 1, n_basis=7), l2 = 1e3
    T3 = 50_000
    c3, f3 = synth_trajectory_device(topo, T3, seed=2, frame0=rank * T3)
    feat = Multifeaturize([id_feat, Curry(gb_feat, inner=0, outer=8, width=1, n_basis=7)])

    def run3():
        return agf.project_forces(coords=c3, forces=f3, coord_map=cmap, constrained_inds=topo.xh_constraints,
                                  method=qp_feat_linear_map, featurizer=feat, kbt=KBT, l2_regularization=L2_REG,
                                  constraint_frames=np.arange(20))

    ms3, _ = wall(run3)
    per = kernel_times(run3)
    n_feat, n_cg = 97 + 7 * 96, 10
    algo3 = {"agf_gram_feat_ws": ("tensor", n_cg * 3 * n_feat * (n_feat + 1) * T3),
             "agf_gram_feat_i8": ("tensor", n_cg * 3 * n_feat * (n_feat + 1) * T3)}
    out["cfg3_featurised"] = {
        "workload": f"cln025, qp_feat_linear_map(Multifeaturize([id_feat, gb_feat(0,8,1,n_basis=7)]), l2=1e3), "
                    f"n_feat {n_feat}, {T3} frames per GPU: project_forces = featurised Gram + per-bead device solve "
                    "+ featurised application",
        "frames_per_gpu": T3, "ms_project_forces": ms3, "frames_per_s": world * T3 / (ms3 * 1e-3),
        "kernels": kernel_table(per, algo3, peaks, hbm_peak, {}),
    }
    tiled_gram_note(out["cfg3_featurised"]["kernels"].get("agf_gram_feat_i8"), n_feat, T3, batch=n_cg)
    del c3, f3

    # ---- config 4 shape: 5 000 atoms, 500 beads, n_red 2 600; Gram + constraint detection + apply
    T4 = 20_000
    topo4 = protein_like_topology(500)
    c4, f4 = synth_trajectory_device(topo4, T4, seed=3, frame0=rank * T4)
    cmap4 = agf.LinearMap([[i] for i in topo4.bead_atoms], n_fg_sites=topo4.n_sites)
    n4 = topo4.n_sites
    n_red4 = int(reduced_columns(n4, topo4.xh_constraints).max()) + 1
    found = {}

    def run4():
        res = agf.project_forces(coords=c4, forces=f4, coord_map=cmap4, constrained_inds="auto",
                                 l2_regularization=L2_REG)
        found["ok"] = res["constraints"] == topo4.xh_constraints
        return res

    ms4, _ = wall(run4)
    per = kernel_times(run4)
    algo4 = {
        "agf_gram_linear_ws": ("tensor", (3 * n_red4 * (n_red4 + 1) + 3 * n4) * T4),
        "agf_gram_linear_i8t": ("tensor", (3 * n_red4 * (n_red4 + 1) + 3 * n4) * T4),
        "agf_map_apply_ws": ("tensor", 6 * 500 * n_red4 * T4),
        "agf_map_apply_i8": ("tensor", 6 * 500 * n_red4 * T4),
        "agf_pair_moments": ("hbm", 12 * n4 * T4),
    }
    out["cfg4_shape"] = {
        "workload": f"synthetic {n4}-atom system, 500 beads, 2 400 X-H constraints -> n_red {n_red4}, {T4} frames per "
                    "GPU: project_forces(constrained_inds='auto', qp_linear_map l2=1e3) = constraint detection + "
                    "Gram + device solve + both applications",
        "frames_per_gpu": T4, "ms_project_forces": ms4, "frames_per_s": world * T4 / (ms4 * 1e-3),
        "constraints_recovered": bool(found.get("ok")),
        "kernels": kernel_table(per, algo4, peaks, hbm_peak, {}),
    }
    tiled_gram_note(out["cfg4_shape"]["kernels"].get("agf_gram_linear_i8t"), n_red4, T4)
    del c4, f4

    # ---- config 5 shape: joptgauss_map on 2 000 atoms / 200 beads
    T5 = 200_000
    topo5 = protein_like_topology(200)
    c5, f5 = synth_trajectory_device(topo5, T5, seed=5, frame0=rank * T5)
    cmap5 = agf.LinearMap([[i] for i in topo5.bead_atoms], n_fg_sites=topo5.n_sites)
    traj5 = agf.Trajectory(coords=c5, forces=f5)
    n5, ncg5 = topo5.n_sites, len(topo5.bead_atoms)
    n_red5 = int(reduced_columns(n5 + ncg5, topo5.xh_constraints).max()) + 1
    held = {}

    def fit5():
        held["tmap"] = agf.joptgauss_map(traj5, cmap5, var=0.25, kbt=KBT, constraints=topo5.xh_constraints,
                                         seed=42100, l2_regularization=L2_REG)
        return held["tmap"]

    ms5_fit, _ = wall(fit5)
    per_fit = kernel_times(fit5)
    ms5_apply, _ = wall(lambda: held["tmap"](traj5))
    per_apply = kernel_times(lambda: held["tmap"](traj5))
    aug_bytes = (12 * n5 + 12 * (n5 + ncg5)) * T5
    algo5f = {"agf_gram_linear_ws": ("tensor", (3 * n_red5 * (n_red5 + 1) + 3 * (n5 + ncg5)) * T5),
              "agf_gram_linear_i8t": ("tensor", (3 * n_red5 * (n_red5 + 1) + 3 * (n5 + ncg5)) * T5),
              "agf_gauss_augment": ("hbm", aug_bytes)}
    algo5a = {"agf_map_apply_ws": ("tensor", 6 * ncg5 * n_red5 * T5),
              "agf_map_apply_i8": ("tensor", 6 * ncg5 * n_red5 * T5),
              "agf_gauss_augment": ("hbm", 2 * aug_bytes)}
    out["cfg5_shape"] = {
        "workload": f"synthetic {n5}-atom system, {ncg5} beads (+{ncg5} noise sites), n_red {n_red5}, {T5} frames per "
                    "GPU: joptgauss_map(var=0.25, l2=1e3) fit, then the fitted AugmentedTMap applied to all frames",
        "frames_per_gpu": T5, "ms_fit": ms5_fit, "ms_apply": ms5_apply,
        "frames_per_s_fit": world * T5 / (ms5_fit * 1e-3), "frames_per_s_apply": world * T5 / (ms5_apply * 1e-3),
        "kernels_fit": kernel_table(per_fit, algo5f, peaks, hbm_peak, {}),
        "kernels_apply": kernel_table(per_apply, algo5a, peaks, hbm_peak, {}),
    }
    tiled_gram_note(out["cfg5_shape"]["kernels_fit"].get("agf_gram_linear_i8t"), n_red5, T5)
    return out


def sharded_parity(agf, torch, dist, rank, world, topo, cmap, synth_trajectory_device) -> dict:
    """Sharded fit (ragged, unaligned shards of 60 000 frames) against the single-GPU fit of the same
    global frames, which every rank recomputes: constraint set, weights, this rank's mapped forces and
    the residual.  Errors are the maximum over ranks."""
    T = 60_000
    bounds = np.linspace(0, T, world + 1).astype(int)
    bounds[1:-1] += 3
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    ac, af = synth_trajectory_device(topo, T, seed=99, frame0=0)
    with agf.frame_sharding():
        res = agf.project_forces(coords=ac[lo:hi].contiguous(), forces=af[lo:hi].contiguous(), coord_map=cmap,
                                 constrained_inds="auto", l2_regularization=L2_REG)
    ref = agf.project_forces(coords=ac, forces=af, coord_map=cmap, constrained_inds="auto", l2_regularization=L2_REG)
    w, wr = res["tmap"].force_map.standard_matrix, ref["tmap"].force_map.standard_matrix
    mine = ref["mapped_forces"][lo:hi]
    errs = torch.tensor([
        float(np.linalg.norm(w - wr) / np.linalg.norm(wr)),
        float((res["mapped_forces"] - mine).norm() / mine.norm()),
        abs(res["residual"] / ref["residual"] - 1.0),
        0.0 if res["constraints"] == ref["constraints"] == topo.xh_constraints else 1.0,
    ], device="cuda", dtype=torch.float64)
    dist.all_reduce(errs, op=dist.ReduceOp.MAX)
    e = errs.tolist()
    return {"frames_total": T, "shards": "ragged, not aligned to 4 frames", "weights_rel_err": e[0],
            "mapped_forces_rel_err": e[1], "residual_rel_err": e[2], "constraints_equal": e[3] == 0.0,
            "n_constraints": len(res["constraints"]), "against": "single-GPU project_forces on all frames"}


if __name__ == "__main__":
    main()
