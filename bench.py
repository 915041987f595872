#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 gravitational force engine.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload direct|tree] [--dump-outputs DIR]

Default workload = BASELINE.json configs[1]: DirectForceComputer, 2^20 particles,
softened gravity (eps = 0.01), one force evaluation per step.  Metric: pairwise
interactions/s (N_targets x N_sources per evaluation, self pair included -- it
contributes exactly 0).  At N > 1 the SAME 2^20-particle problem is target-
sharded over the ranks (strong scaling): each step all-gathers the source
positions with NCCL and every rank evaluates its N/G targets against all sources.

`value`  : device-resident throughput (CUDA events on the launching stream,
           max over ranks, L2 flushed between timed steps).
`e2e`    : the same metric through the host-pointer C-ABI call
           (b200_direct_forces_host; pinned host buffers, H2D + D2H inside the
           timed region).  This is the number to hold against --impl reference.
`roofline`: dominant kernel (direct_kernel) against the FP32 FMA peak measured
           in this run by an FFMA probe (MEASURED_PEAKS.json has no FP32 figure).
Sub-lines of the default run, at every N, each ending in its own `parity_check` (a 1 024-target sample per rank
against the CPU oracle; non-local rows are NaN-poisoned before every gather, so a broken exchange cannot pass):
`tree_summary`  BASELINE configs[2]: TreeForceComputer theta = 0.5, leaf 8, the same 2^20 particles -- ms per build +
           walk, interactions/s, roofline = issue fraction + LSU write-back fraction + lane utilisation of the walk.
`tree_box_convention_summary`  the same with positions in [0, 100)^3 (what the reference's generators emit).
`c4_summary`    configs[3]: 2^24-particle Lambda-CDM KDK steps (random index order): Hilbert-stored particles, octant-
           sharded build, table exchange, forest walk; phases leapfrog / allgather / build / publish / walk as the max
           over ranks, the walk kernel's own time, per-rank list.  `c4_summary_replicated_build`: the round-1 scheme.
`c5_summary`    configs[4]: 2^23-particle direct sum (--no-c5 skips it: 24 s on one GPU).
`c1_summary`    configs[0]: 16 384 particles x 10 KDK steps, device-resident.
`leapfrog_roofline`  the fused kick-kick-drift pass at 2^24 / N particles against the measured HBM peak.
`--workload tree` makes the Barnes-Hut step the main line (e2e, CPU reference tree); `--ic zeldovich`,
`--order morton`, `--kdk`, `--c4-mode replicated`, `--sources peer` select other inputs / schemes.
`cpu_baseline` / --impl reference: the reference's own CPU direct sum
           (oracle/_ref = /root/reference sources compiled in place; falls back
           to the restated port) on all host cores, bounded sample.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))

FLOP_PER_INTERACTION = 20          # GPU-Gems-3 convention (SURVEY 8d)
EPS = 0.01


# --------------------------------------------------------------------------- inputs
def make_particles(n, seed=42, order="random"):
    """Uniform in [-50,50)^3, unit masses (what every reference generator emits).  order="morton":
    the same particles stored in Morton (Z-curve) order, the way a production run keeps them, so that a
    contiguous index range -- one rank's shard -- is a compact region of space."""
    rng = np.random.default_rng(seed)
    pos = rng.uniform(-50.0, 50.0, size=(n, 3)).astype(np.float32)
    if order == "morton":
        q = np.clip(((pos + 50.0) * (1024.0 / 100.0)).astype(np.int64), 0, 1023)

        def spread(v):
            v = (v | (v << 16)) & 0x030000FF
            v = (v | (v << 8)) & 0x0300F00F
            v = (v | (v << 4)) & 0x030C30C3
            v = (v | (v << 2)) & 0x09249249
            return v
        key = (spread(q[:, 0]) << 2) | (spread(q[:, 1]) << 1) | spread(q[:, 2])
        pos = np.ascontiguousarray(pos[np.argsort(key, kind="stable")])
    return pos, np.ones(n, np.float32)


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons while the timed region runs."""

    def __init__(self, index=0, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------- CPU baseline
TREE_SAMPLE = 65536          # particles per single-threaded reference tree evaluation (~1 s per core)
DIRECT_SAMPLE = 16384


def _ref_worker(args):
    workload, kind, n, seed, reps = args
    sys.path.insert(0, ROOT)
    from oracle.pyoracle import Oracle, Ref
    pos, mass = make_particles(n, seed)
    if kind != "reference":
        os.environ["OMP_NUM_THREADS"] = "1"
    t0 = time.perf_counter()
    if workload == "direct":
        if kind == "reference":
            r = Ref()
            for _ in range(reps):
                r.direct(pos)                  # TreeForceComputer, one root leaf: the CPU direct sum
        else:
            o = Oracle()
            for _ in range(reps):
                o.direct_f32(pos, None, eps=EPS)
    else:
        if kind == "reference":
            r = Ref()
            for _ in range(reps):
                r.tree_forces(pos, mass, 0.5, 8, 20, 100.0)      # TreeForceComputer::compute_forces: build + walk
        else:
            o = Oracle()
            for _ in range(reps):
                o.tree_forces(o.tree_build(pos, mass), pos, 0.5)
    return time.perf_counter() - t0


def _tree_sample_interactions(n_sample):
    """Cell + pair interactions of ONE reference tree evaluation of an n_sample uniform set (counted
    once, untimed, by the restated oracle whose counters equal the reference walk's by construction)."""
    from oracle.pyoracle import Oracle
    o = Oracle()
    pos, mass = make_particles(n_sample, 1000)
    _, cnt = o.tree_forces(o.tree_build(pos, mass), pos, 0.5, counters=True)
    return float(cnt[1] + cnt[2])


def cpu_reference_batch(cores, n_sample, reps, pool, kind, workload="direct", per_eval=None):
    """One bounded batch: every core runs the reference's single-threaded CPU path on its own
    n_sample-particle subsample.  Returns (interactions, seconds)."""
    t0 = time.perf_counter()
    list(pool.map(_ref_worker, [(workload, kind, n_sample, 1000 + c, reps) for c in range(cores)]))
    dt = time.perf_counter() - t0
    if per_eval is None:
        per_eval = float(n_sample) * float(n_sample)
    return cores * reps * per_eval, dt


def cpu_kind():
    from oracle.pyoracle import Ref
    return "reference" if Ref.available() else "port"


def _cpu_sample(workload):
    if workload == "direct":
        return DIRECT_SAMPLE, None, ("the reference CPU direct sum (TreeForceComputer, leaf_capacity>N => leaf "
                                     "pair loop; its own sources built -O2 -ffp-contract=off by oracle/Makefile, "
                                     "the bit-reproducible flags of the parity oracle, not the reference's -O3 "
                                     "-march=native)")
    return TREE_SAMPLE, _tree_sample_interactions(TREE_SAMPLE), ("the reference CPU TreeForceComputer "
                                                                 "(theta 0.5, leaf 8: build + walk; its own sources "
                                                                 "built -O2 -ffp-contract=off by oracle/Makefile)")


def run_cpu_baseline(workload="direct", target_seconds=12.0):
    from concurrent.futures import ProcessPoolExecutor
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    kind = cpu_kind()
    n_sample, per_eval, what = _cpu_sample(workload)
    with ProcessPoolExecutor(max_workers=cores, mp_context=mp.get_context("spawn")) as pool:
        cpu_reference_batch(cores, 2048, 1, pool, kind, workload)                   # warm: spawn workers, page in
        inter, dt = cpu_reference_batch(cores, n_sample, 1, pool, kind, workload, per_eval)   # calibrate
        reps = max(1, int(round(target_seconds / dt)))
        inter, dt = cpu_reference_batch(cores, n_sample, reps, pool, kind, workload, per_eval)
    return {"value": inter / dt, "unit": "interactions/s", "cores": cores, "kind": kind,
            "sample": f"{cores} independent single-threaded instances of {what}, {n_sample} uniform particles each x "
                      f"{reps} evaluations; {inter:.3e} interactions in {dt:.1f} s"}


def bench_reference(args):
    """--impl reference: the reference's own CPU path, all host cores, bounded steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from concurrent.futures import ProcessPoolExecutor
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    kind = cpu_kind()
    n_sample, per_eval, what = _cpu_sample(args.workload)
    reps = 1
    times, inter = [], 0.0
    with ProcessPoolExecutor(max_workers=cores, mp_context=mp.get_context("spawn")) as pool:
        cpu_reference_batch(cores, 2048, 1, pool, kind, args.workload)
        for _ in range(args.warmup):
            cpu_reference_batch(cores, n_sample, reps, pool, kind, args.workload, per_eval)
        for _ in range(args.steps):
            inter, dt = cpu_reference_batch(cores, n_sample, reps, pool, kind, args.workload, per_eval)
            times.append(dt)
    total = sum(times)
    value = inter * args.steps / total
    sample = (f"each step = {cores} independent single-threaded instances of {what}, "
              f"{n_sample} uniform particles each ({inter:.3e} interactions/step); the rate is per interaction, "
              f"so it transfers to the {args.particles}-particle workload" +
              ("" if args.workload == "direct" else " (a larger tree does more interactions per particle, "
                                                    "at the same cost per interaction)"))
    line = {"impl": "reference", "metric": "pairwise_interactions_per_s", "value": value, "unit": "interactions/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": value, "unit": "interactions/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "interactions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.workload == "tree":
        line["particle_steps_per_s"] = cores * reps * n_sample * args.steps / total
    print(json.dumps(line))


def zeldovich_grid(n):
    """Power-of-two grid with at least n points (SURVEY 8d): 128 for 2^20 (stride-2 subsample of the
    grid, grid_to_particles), 256 for 2^24 (the first n grid points)."""
    g = 4
    while g ** 3 < n:
        g *= 2
    return g


def workload_config(args):
    cfg = _workload_config(args)
    if getattr(args, "order", "random") == "morton" and getattr(args, "ic", "uniform") == "uniform":
        cfg["workload"] = cfg["workload"].replace("uniform [-50,50)^3", "uniform [-50,50)^3 stored in Morton order")
        cfg["order"] = "morton"
    if getattr(args, "ic", "uniform") == "zeldovich":
        cfg["workload"] = cfg["workload"].replace(
            "uniform [-50,50)^3",
            f"Zel'dovich ICs (b200_zeldovich_ics_dev: {zeldovich_grid(args.particles)}^3 grid, 100 Mpc/h box, "
            f"z = {args.z_initial:g}, seed 12345, sigma_8 0.81, origin-centred)")
        cfg["ic"] = "zeldovich"
    if getattr(args, "kdk", False):
        cfg["workload"] += "; each step = full KDK leapfrog step (omega_m 0.31, omega_lambda 0.69, h 0.67, a0 1, dt 1e-4)"
    return cfg


def _workload_config(args):
    n = args.particles
    if args.workload == "direct":
        return {"workload": f"DirectForceComputer, {n} particles (BASELINE configs[1] when n = 2^20), "
                            f"uniform [-50,50)^3, unit masses, eps = {EPS}, one force evaluation per step; "
                            f"targets sharded over {args.gpus} GPU(s), sources all-gathered",
                "particles": n, "eps": EPS, "l2": "flushed between timed steps (512 MB write)",
                "sources": getattr(args, "sources", "allgather")}
    return {"workload": f"TreeForceComputer Barnes-Hut theta=0.5 leaf=8 max_depth=20, {n} particles "
                        f"(BASELINE configs[2] scale), uniform [-50,50)^3, build + walk per step",
            "particles": n, "theta": 0.5, "leaf_capacity": 8, "l2": "flushed between timed steps (512 MB write)"}


# --------------------------------------------------------------------------- GPU arm
NAN = float("nan")


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), \
            "MEASURED_PEAKS.json hbm_gbs (burst copy figure; of measured)"
    except Exception:
        return 6532.2, "fallback 6532.2 GB/s (MEASURED_PEAKS.json not on this box)"


def ncu_static(key, n):
    """Per-launch figures that only a profiler can give (DRAM / L2 / L1 bytes, warp instructions executed) for
    the launch this run repeats -- same inputs, same kernel, hence the same counts.  Captured once per kernel
    revision under ncu (never timed there) and committed in profiles/ncu_traffic.json; null when no capture of
    this size exists."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(key, {}).get(str(n))
    except Exception:
        return None


class Dist:
    """The few collectives the harness needs, no-ops on one GPU."""

    def __init__(self, torch, dist, world, rank, dev):
        self.torch, self.dist, self.world, self.rank, self.dev = torch, dist, world, rank, dev

    def sync(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t)
        return float(t.item())

    def all_ok(self, flag):
        return self.max(0.0 if flag else 1.0) == 0.0


class Sharded:
    """Replicated float4 source array + this rank's target shard (SURVEY 8e): contiguous original-index
    ranges, sources all-gathered with NCCL.  poison() overwrites every row this rank does not own with NaN
    (untimed, before each step), so a step whose all-gather did not deliver produces NaN forces;
    gather_checksums_ok() compares, shard by shard, an integer checksum of the gathered rows with the one
    their owner computed on its own copy."""

    def __init__(self, D, posm_full_host, n):
        torch = D.torch
        self.D, self.n = D, n
        self.lo, self.hi = D.rank * n // D.world, (D.rank + 1) * n // D.world
        self.nl = self.hi - self.lo
        self.posm = torch.from_numpy(posm_full_host).to(D.dev) if isinstance(posm_full_host, np.ndarray) \
            else posm_full_host
        self.shard = self.posm[self.lo:self.hi].clone() if D.world > 1 else self.posm
        self.equal = (n % D.world == 0)

    def poison(self):
        if self.D.world > 1:
            self.posm[:self.lo].fill_(NAN)
            self.posm[self.hi:].fill_(NAN)

    def gather(self):
        D = self.D
        if D.world > 1:
            if self.equal:
                D.dist.all_gather_into_tensor(self.posm.view(-1), self.shard.view(-1))
            else:
                outs = [self.posm[r * self.n // D.world:(r + 1) * self.n // D.world] for r in range(D.world)]
                D.dist.all_gather(outs, self.shard)

    def _checksum(self, rows):
        return rows.contiguous().view(self.D.torch.int32).to(self.D.torch.int64).sum()

    def gather_checksums_ok(self):
        D = self.D
        if D.world == 1:
            return True
        torch = D.torch
        mine = self._checksum(self.shard).reshape(1)
        owners = [torch.zeros(1, dtype=torch.int64, device=D.dev) for _ in range(D.world)]
        D.dist.all_gather(owners, mine)
        ok = True
        for r in range(D.world):
            got = self._checksum(self.posm[r * self.n // D.world:(r + 1) * self.n // D.world])
            ok = ok and bool((got == owners[r][0]).item())
        return D.all_ok(ok)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(D, out_dir, n, rows, scalars=None):
    """--dump-outputs: write what the timed path returned in its last step as <out_dir>/<name>.npy (float32 /
    float64) on rank 0, so that two builds can be compared output for output.  `rows` maps a name to this rank's
    [nl, k] device rows of an n-row result (target order); they are gathered over the ranks.  Above
    DUMP_LIMIT_BYTES in all, the same fixed, seeded sample of rows (sorted row indices) is kept from every array."""
    torch = D.torch
    full = {}
    for name, t in rows.items():
        t = t.contiguous()
        if D.world > 1:
            parts = [torch.empty(((r + 1) * n // D.world - r * n // D.world, t.shape[1]), dtype=t.dtype, device=D.dev)
                     for r in range(D.world)]
            D.dist.all_gather(parts, t)
            t = torch.cat(parts)
        full[name] = t.cpu().numpy()
    if D.rank != 0:
        return
    row_bytes = sum(a.itemsize * a.shape[1] for a in full.values())
    if n * row_bytes > DUMP_LIMIT_BYTES - 4096:
        keep = np.sort(np.random.default_rng(0).choice(n, (DUMP_LIMIT_BYTES - 4096) // row_bytes, replace=False))
        full = {k: a[keep] for k, a in full.items()}
    full.update({k: np.asarray(v, np.float64) for k, v in (scalars or {}).items()})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in full.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def sample_block(lo, nl, want=1024):
    """A contiguous block of `want` targets inside [lo, lo + nl) (the oracle takes target ranges)."""
    cnt = min(want, nl)
    return lo + (nl - cnt) // 3, cnt


def parity_direct(D, S, acc, mass_unit):
    """Untimed: >= 1024 targets per rank against the CPU oracle's FP64 direct sum over the gathered sources."""
    from inputs import rel_l2
    from oracle.pyoracle import Oracle
    o = Oracle()
    host = S.posm.cpu().numpy()
    pos = np.ascontiguousarray(host[:, :3])
    mass = None if mass_unit else np.ascontiguousarray(host[:, 3])
    b0, cnt = sample_block(S.lo, S.nl)
    finite = bool(np.isfinite(host).all())
    ref = o.direct_f64(pos, mass, EPS, i0=b0, n_targets=cnt) if finite else np.full((cnt, 3), np.nan)
    got = acc[b0 - S.lo:b0 - S.lo + cnt].cpu().numpy()
    err = rel_l2(got, ref) if finite and np.isfinite(got).all() else float("inf")
    err = D.max(err)
    return {"rel_l2": err, "gate": 1e-5, "targets_per_rank": cnt, "oracle": "orc_direct_f64 (CPU, all gathered sources)",
            "gather_checksums_ok": S.gather_checksums_ok(), "ok": bool(err <= 1e-5)}


def parity_tree(D, S, acc, box=100.0, theta=0.5, on_rank0_only=False):
    """Untimed: a block of targets per rank against the CPU oracle's tree (restated reference builder + walk) on
    the gathered particles.  on_rank0_only: the oracle tree is built once, on rank 0, which checks every
    rank's block (used at 2^24 particles, where the CPU build takes seconds and gigabytes)."""
    from inputs import rel_l2
    from oracle.pyoracle import Oracle
    torch = D.torch
    b0, cnt = sample_block(S.lo, S.nl)
    got_dev = acc[b0 - S.lo:b0 - S.lo + cnt].contiguous()
    err = 0.0
    if on_rank0_only and D.world > 1:
        blocks = [torch.empty((cnt, 3), dtype=torch.float32, device=D.dev) for _ in range(D.world)]
        D.dist.all_gather(blocks, got_dev)      # every rank's block has the same size only when shards are equal
        starts = [sample_block(r * S.n // D.world, (r + 1) * S.n // D.world - r * S.n // D.world)[0]
                  for r in range(D.world)]
        if D.rank == 0:
            host = S.posm.cpu().numpy()
            pos, mass = np.ascontiguousarray(host[:, :3]), np.ascontiguousarray(host[:, 3])
            if np.isfinite(host).all():
                o = Oracle()
                t = o.tree_build(pos, mass, box=box)
                for r in range(D.world):
                    ref = o.tree_forces(t, pos, theta, i0=starts[r], n_targets=cnt)
                    g = blocks[r].cpu().numpy()
                    err = max(err, rel_l2(g, ref) if np.isfinite(g).all() else float("inf"))
            else:
                err = float("inf")
    else:
        host = S.posm.cpu().numpy()
        pos, mass = np.ascontiguousarray(host[:, :3]), np.ascontiguousarray(host[:, 3])
        got = got_dev.cpu().numpy()
        if np.isfinite(host).all() and np.isfinite(got).all():
            o = Oracle()
            ref = o.tree_forces(o.tree_build(pos, mass, box=box), pos, theta, i0=b0, n_targets=cnt)
            err = rel_l2(got, ref)
        else:
            err = float("inf")
    err = D.max(err)
    return {"rel_l2": err, "gate": 1e-3, "targets_per_rank": cnt,
            "oracle": "orc_tree_build_levels + orc_tree_forces (CPU restatement of TreeForceComputer, all gathered particles)",
            "gather_checksums_ok": S.gather_checksums_ok(), "ok": bool(err <= 1e-3)}


def walk_roofline(eng, D, n_total, nl, cnt6, walk_s, clocks, static_ok):
    """What bounds the walk (walk_warp2_kernel): instruction issue on L1/L2-resident data, with the L1 -> register
    write-back of its warp-wide broadcast loads (128 B per clock and SM) as the second ceiling -- the one-target
    kernel it replaced ran that path at 0.76.  No HBM fraction is quoted -- the algorithmic byte count of SURVEY 8d
    (32 B per node visit, 16 B per pair source, per LANE) is served by broadcast loads and exceeds what any memory
    level moves by 10-1000x."""
    vis, pc, pp, slots, nlanes, nawake = [float(x) for x in cnt6]
    # instruction-weighted lane utilisation: one node visit of a warp costs ~47 instructions for its 64 target slots
    # (23.5 per 32), a packed pair row ~18 for 32 lanes x 2 source slots (9 per slot); SASS of the shipped kernel,
    # profiles/r2_sass_excerpts.md
    issued = 23.5 * nlanes + 9.0 * slots
    useful = 23.5 * nawake + 9.0 * pp
    inst = ncu_static("tree_walk_inst_executed", n_total) if static_ok else None
    wb = ncu_static("tree_walk_lsu_writeback_cycles", n_total) if static_ok else None
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    issue_peak = eng.sm_count * 4 * sm_mhz * 1e6            # warp instructions per second, 4 schedulers per SM
    out = {
        "bound": "issue",
        "kernel": "walk_warp2_kernel (a warp walks the union of the traversals of 64 Hilbert-adjacent targets, two per "
                  "lane in the halves of packed-FP32 operands; per-target accept test; depth-first walk records; leaf "
                  "particles grouped per parent, packed-FP32 pair rows)",
        "kernel_ms": 1e3 * walk_s,
        "interactions_per_s_walk_only": (pc + pp) / walk_s,
        "fp32_tflops_at_20_flop": 20.0 * (pc + pp) / walk_s / 1e12,
        "pair_row_lane_frac": pp / slots if slots else None,
        "node_visit_lane_frac": nawake / nlanes if nlanes else None,
        "useful_lane_frac": useful / issued if issued else None,
        "lane_frac_weights": "47 instructions per node visit of 64 target slots, 9 per pair-row source slot (SASS counts)",
        "walk_counters_nodes_cells_pairs": [int(vis), int(pc), int(pp)],
        "warp_instructions": inst,
        "issue_frac": (inst / walk_s / issue_peak) if inst else None,
        "issue_peak": f"{eng.sm_count} SMs x 4 schedulers x {sm_mhz:.0f} MHz (median SM clock sampled in this run)",
        "warp_instructions_source": "ncu smsp__inst_executed.sum of this launch (profiles/ncu_traffic.json; same inputs, "
                                    "same kernel => same count); time and clock are live",
        # second ceiling: cycles the L1's LSU write-back port was busy (ncu l1tex__lsu_writeback_active.sum over the
        # SMs; a warp-wide 256-bit broadcast load takes 8) against the cycles of this run's launch
        "lsu_writeback_frac": (wb / (eng.sm_count * walk_s * sm_mhz * 1e6)) if wb else None,
        "traffic": ncu_static("tree", n_total) if static_ok else None,
        "ncu_l2_bytes": ncu_static("tree_l2_bytes", n_total) if static_ok else None,
        "ncu_l1_bytes": ncu_static("tree_l1_bytes", n_total) if static_ok else None,
    }
    if out["issue_frac"] is not None:
        out.update({"achieved": inst / walk_s / 1e9, "peak": issue_peak / 1e9, "unit": "G warp-instructions/s",
                    "frac": out["issue_frac"]})
    return out


def tree_summary(eng, D, S, flush, steps=5, box=100.0, label="centred [-50,50)^3", with_parity=True, clocks=None,
                 static_ok=False):
    """BASELINE configs[2] on the device-resident particles: (all-gather +) build + walk per step, theta 0.5,
    leaf 8, max_depth 20.  CUDA events around each step and around build / walk, L2 flushed between steps."""
    torch = D.torch
    n, lo, nl = S.n, S.lo, S.nl
    acc = torch.empty((nl, 3), dtype=torch.float32, device=D.dev)

    def step(ev=None):
        S.gather()
        if ev:
            ev[1].record()
        eng.tree_build_dev(S.posm, n, box, 8, 20)
        if ev:
            ev[2].record()
        eng.tree_walk_dev(acc, lo, nl, theta=0.5)

    for _ in range(3):
        S.poison()
        step()
    D.sync()
    tot, gat, bld, wlk = [], [], [], []
    for _ in range(steps):
        flush.zero_()
        S.poison()
        D.sync()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        step(ev)
        ev[3].record()
        torch.cuda.synchronize()
        tot.append(ev[0].elapsed_time(ev[3])); gat.append(ev[0].elapsed_time(ev[1]))
        bld.append(ev[1].elapsed_time(ev[2])); wlk.append(ev[2].elapsed_time(ev[3]))
    D.sync()
    eng.tree_set_counting(True)
    eng.tree_walk_dev(acc, lo, nl, theta=0.5)
    torch.cuda.synchronize()
    cnt6 = eng.tree_walk_stats()
    eng.tree_set_counting(False)
    eng.tree_walk_dev(acc, lo, nl, theta=0.5)      # the parity block comes from the shipped (non-counting) instance
    torch.cuda.synchronize()
    step_s = D.max(float(np.mean(tot))) * 1e-3
    walk_s = D.max(float(np.mean(wlk))) * 1e-3
    inter = D.sum(float(cnt6[1] + cnt6[2]))
    out = {"workload": f"TreeForceComputer theta=0.5 leaf=8 max_depth=20, {n} uniform particles {label}, root cube "
                       f"[-{box / 2:g},{box / 2:g})^3; step = "
                       + ("NCCL all-gather of the shards + replicated build + walk of this rank's targets" if D.world > 1
                          else "build + walk"),
           "ms_per_step": 1e3 * step_s, "allgather_ms": D.max(float(np.mean(gat))),
           "build_ms": D.max(float(np.mean(bld))), "walk_kernel_ms": 1e3 * walk_s,
           "interactions_per_s": inter / step_s, "particle_steps_per_s": n / step_s, "steps": steps,
           "roofline": walk_roofline(eng, D, n, nl, cnt6, walk_s, clocks, static_ok and D.world == 1)}
    if with_parity:
        out["parity_check"] = parity_tree(D, S, acc, box=box)
    return out


def leapfrog_roofline(eng, D, n, reps=10):
    """leapfrog_kernel alone on n particles (the fused kick-kick-drift pass of a KDK step): 16 + 12 + 12 B read,
    12 + 16 B written per particle; the arrays (68 B x n) are far larger than L2, so no flush is needed."""
    torch = D.torch
    posm = torch.rand((n, 4), device=D.dev) + 0.5
    vel = torch.zeros((n, 3), device=D.dev)
    acc = torch.rand((n, 3), device=D.dev)
    for _ in range(3):
        eng.leapfrog_dev(posm, vel, acc, n, 2, np.float32(5e-5), 1.0, np.float32(1e-4), 0.0)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):            # 4 launches back to back per event pair: the ~5 us of event + launch overhead
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)      # would be 3 % of one
        e0.record()
        for _ in range(4):
            eng.leapfrog_dev(posm, vel, acc, n, 2, np.float32(5e-5), 1.0, np.float32(1e-4), 0.0)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / 4)
    t = float(np.mean(ms)) * 1e-3
    peak, src = hbm_peak()
    gbs = 68.0 * n / t / 1e9
    del posm, vel, acc
    return {"bound": "hbm", "kernel": "leapfrog_kernel (kick + kick + drift fused, 1024-particle tiles, coalesced 128-bit "
                                      "accesses, velocities/accelerations transposed through shared memory)",
            "particles": n, "kernel_ms": 1e3 * t, "bytes_per_particle": 68, "achieved": gbs, "peak": peak,
            "unit": "GB/s", "frac": gbs / peak, "peak_source": src,
            "traffic": ncu_static("leapfrog", n), "particle_steps_per_s": n / t}


def c4_summary(eng, D, flush, n, steps, mode):
    """BASELINE configs[3]: TreeForceComputer + Lambda-CDM leapfrog (omega_m 0.31, omega_lambda 0.69, h 0.67,
    a0 = 1, dt = 1e-4), n particles uniform in [-50,50)^3 in RANDOM index order with N(0,100) velocities,
    sharded over the ranks.  Every step = fused kick-kick-drift of the local particles, scale-factor update,
    exchange, octree build, theta = 0.5 walk of the local targets.  Phases are timed with CUDA events on the
    launching stream; every figure is the max over ranks."""
    torch, dist = D.torch, D.dist
    g = torch.Generator(device=D.dev)
    g.manual_seed(4242)
    posm = torch.empty((n, 4), dtype=torch.float32, device=D.dev)
    velf = torch.empty((n, 3), dtype=torch.float32, device=D.dev)
    if D.rank == 0:
        posm[:, :3] = torch.rand((n, 3), generator=g, device=D.dev) * 100.0 - 50.0
        posm[:, 3] = 1.0
        velf.normal_(0.0, 100.0, generator=g)
    if D.world > 1:
        dist.broadcast(posm, 0)
        dist.broadcast(velf, 0)
    dt = 1e-4
    run = (C4RunSharded if mode == "sharded" else C4Run)(eng, D, posm, velf, n, mode)
    del velf
    a = 1.0
    run.forces()                         # forces at the initial positions (first half-kick)
    for _ in range(3):
        a = run.step(a, dt)
    D.sync()
    sampler = ClockSampler(D.dev.index, period=0.005)
    sampler.start()
    names = run.phase_names
    acc_ms = {k: [] for k in names}
    tot, kern = [], []
    eng.set_timing(True)                 # the walk kernel's own events (inside b200_tree_walk_dev)
    for _ in range(steps):
        flush.zero_()
        run.poison()
        D.sync()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record()
        a = run.step(a, dt, ev)
        torch.cuda.synchronize()
        tot.append(ev[0].elapsed_time(ev[-1]))
        kern.append(eng.last_kernel_ms())
        for i, k in enumerate(names):
            acc_ms[k].append(ev[i].elapsed_time(ev[i + 1]))
    # the same walk once more on its own (tables and target order as the last step left them, L2 flushed, no
    # collective in front of it): what the kernel costs when nothing else has just used the GPU's memory system
    alone = []
    for _ in range(3):
        flush.zero_()
        D.sync()
        run.walk_only()
        torch.cuda.synchronize()
        alone.append(eng.last_kernel_ms())
    D.sync()
    sampler.stop()
    step_s = D.max(float(np.sum(tot))) * 1e-3 / steps
    out = {"workload": f"TreeForceComputer theta=0.5 leaf=8 max_depth=20 + Lambda-CDM KDK leapfrog (omega_m 0.31, "
                       f"omega_lambda 0.69, h 0.67, a0 1, dt 1e-4), {n} particles uniform [-50,50)^3 in random index "
                       f"order, N(0,100) velocities, {D.world} GPU(s)",
           "mode": run.mode_text, "ms_per_step": 1e3 * step_s, "particle_steps_per_s": n / step_s, "steps": steps,
           "scale_factor_after": a}
    for k in names:
        out[k + "_ms"] = D.max(float(np.mean(acc_ms[k])))
    out["walk_kernel_ms"] = D.max(float(np.mean(kern)))          # the rest of walk_ms: target order (every 8th step), launch
    out["walk_kernel_ms_min_rank"] = -D.max(-float(np.mean(kern)))
    out["walk_kernel_alone_ms"] = D.max(float(np.min(alone)))
    if D.world > 1:                      # per-rank view: which GPU is the slow one, and at what clock
        mine = {"rank": D.rank, "gpu": D.dev.index, "walk_kernel_ms": float(np.mean(kern)),
                "walk_kernel_alone_ms": float(np.min(alone)), "sm_mhz": sampler.summary().get("sm_mhz")}
        if os.environ.get("B200_BENCH_WALK_MATRIX"):       # diagnosis: every rank walks every rank's range on its own
            row = []
            for rr in range(D.world):
                best = 1e30
                for _ in range(2):
                    flush.zero_()
                    D.sync()
                    eng.tree_walk_dev(run.acc, rr * run.nl, run.nl, theta=0.5)
                    torch.cuda.synchronize()
                    best = min(best, eng.last_kernel_ms())
                row.append(round(best, 3))
            mine["walk_of_range_ms"] = row
        per_rank = [None] * D.world
        dist.all_gather_object(per_rank, mine)
        out["per_rank"] = per_rank
    eng.set_timing(False)
    out["clocks"] = sampler.summary()
    peak, _ = hbm_peak()
    out["leapfrog_hbm_frac"] = 68.0 * run.nl / (out["leapfrog_ms"] * 1e-3) / 1e9 / peak if out.get("leapfrog_ms") else None
    out["parity_check"] = run.parity()
    run.close()
    return out


class C4Run:
    """One rank's state of the C4 run.  mode "replicated": contiguous index shards, positions all-gathered in
    place, every rank builds the whole octree (round-1 scheme)."""

    def __init__(self, eng, D, posm, velf, n, mode):
        torch = D.torch
        self.eng, self.D, self.n, self.mode = eng, D, n, mode
        self.S = Sharded(D, posm, n)
        self.lo, self.nl = self.S.lo, self.S.nl
        self.vel = velf[self.lo:self.lo + self.nl].clone()
        self.acc = torch.zeros((self.nl, 3), dtype=torch.float32, device=D.dev)
        self.phase_names = ["leapfrog", "allgather", "build", "walk"]
        self.mode_text = ("contiguous index shards; NCCL all-gather of the float4 shards; every rank builds the whole "
                          "octree (graph replay) and walks its own targets")

    def poison(self):
        self.S.poison()

    def forces(self, ev=None):
        S, eng = self.S, self.eng
        S.gather()
        if ev:
            ev[2].record()
        eng.tree_build_dev(S.posm, self.n, 100.0, 8, 20)
        if ev:
            ev[3].record()
        eng.tree_walk_dev(self.acc, self.lo, self.nl, theta=0.5)
        if ev:
            ev[4].record()

    def walk_only(self):
        self.eng.tree_walk_dev(self.acc, self.lo, self.nl, theta=0.5)

    def step(self, a, dt, ev=None):
        eng = self.eng
        # closing half-kick of the previous step + opening half-kick + drift: one pass (b200_leapfrog_dev, n_kicks = 2)
        eng.leapfrog_dev(self.S.shard, self.vel, self.acc, self.nl, 2, np.float32(dt * 0.5), a, np.float32(dt), 0.0)
        a = eng.scale_factor_step(a, dt)
        if ev:
            ev[1].record()
        self.forces(ev)
        return a

    def parity(self):
        return parity_tree(self.D, self.S, self.acc, on_rank0_only=True)

    def close(self):
        pass


class C4RunSharded:
    """mode "sharded": (1) STORAGE along a space-filling curve -- the particles are ordered once along a Hilbert curve
    (b200_spatial_order_dev) and kept in that order for the whole run; rank r owns the r-th N/G run of slots, a
    compact region whatever the original index order, and the per-step exchange is the plain in-place NCCL
    all-gather of the float4 shards.  The octree is still the reference's: the build receives the ARRIVAL order
    (arrival[k] = slot of original particle k), so particles are inserted in original index order.
    (2) OCTANT-SHARDED BUILD -- rank r builds only the subtrees of its octants of the root
    (b200_tree_build_part_dev) and the ranks exchange their walk tables (b200_tree_forest_publish: NCCL broadcasts
    on the context's own communicator).  (3) The walk of the rank's slots runs over the forest."""

    def __init__(self, eng, D, posm, velf, n, mode):
        torch, dist = D.torch, D.dist
        self.eng, self.D, self.n = eng, D, n
        if n % D.world or D.world > 8:
            raise SystemExit("c4 sharded mode needs n divisible by the rank count and at most 8 ranks")
        if D.world > 1:
            box = [eng.shard_unique_id() if D.rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            eng.shard_init(box[0], D.rank, D.world)
        self.perm = torch.empty(n, dtype=torch.int32, device=D.dev)          # perm[slot] = original index
        eng.spatial_order_dev(posm, n, 100.0, self.perm)
        stored = torch.empty_like(posm)
        vel_all = torch.empty_like(velf)
        eng.gather_rows_dev(posm, velf, self.perm, n, stored, vel_all)
        self.arrival = torch.empty_like(self.perm)                            # arrival[original index] = slot
        self.arrival[self.perm.long()] = torch.arange(n, dtype=torch.int32, device=D.dev)
        self.S = Sharded(D, stored, n)
        self.lo, self.nl = self.S.lo, self.S.nl
        self.vel = vel_all[self.lo:self.lo + self.nl].clone()
        del vel_all
        self.acc = torch.zeros((self.nl, 3), dtype=torch.float32, device=D.dev)
        self.phase_names = ["leapfrog", "allgather", "build", "publish", "walk"]
        self.mode_text = ("particles stored in Hilbert-curve order fixed at step 0 (contiguous slot shards), arrival order "
                          "= original index order handed to the build; per step: in-place NCCL all-gather of the float4 "
                          "shards, octant-sharded octree build (each rank its own octants of the root) + NCCL exchange of "
                          "the walk tables (b200_tree_forest_publish), forest walk of the rank's slots")

    def poison(self):
        self.S.poison()

    def forces(self, ev=None):
        D, eng, S = self.D, self.eng, self.S
        S.gather()
        if ev:
            ev[2].record()
        eng.tree_build_part_dev(S.posm, self.n, D.rank, D.world, 100.0, 8, 20, arrival=self.arrival)
        if ev:
            ev[3].record()
        if D.world > 1:
            eng.tree_forest_publish()
        if ev:
            ev[4].record()
        eng.tree_walk_dev(self.acc, self.lo, self.nl, theta=0.5)
        if ev:
            ev[5].record()

    def walk_only(self):
        self.eng.tree_walk_dev(self.acc, self.lo, self.nl, theta=0.5)

    def step(self, a, dt, ev=None):
        eng = self.eng
        eng.leapfrog_dev(self.S.shard, self.vel, self.acc, self.nl, 2, np.float32(dt * 0.5), a, np.float32(dt), 0.0)
        a = eng.scale_factor_step(a, dt)
        if ev:
            ev[1].record()
        self.forces(ev)
        return a

    def parity(self, per_rank=1024):
        """Untimed.  Rank 0 puts the particles it holds after the all-gather back in original index order, builds the
        CPU oracle's tree from them and walks a block of every rank's targets."""
        from inputs import rel_l2
        from oracle.pyoracle import Oracle
        D, torch = self.D, self.D.torch
        b0, cnt = sample_block(self.lo, self.nl, per_rank)
        got = self.acc[b0 - self.lo:b0 - self.lo + cnt].contiguous()
        gots = [torch.empty_like(got) for _ in range(D.world)]
        if D.world > 1:
            D.dist.all_gather(gots, got)
        else:
            gots = [got]
        err = 0.0
        if D.rank == 0:
            perm = self.perm.cpu().numpy()
            host = np.empty((self.n, 4), np.float32)
            host[perm] = self.S.posm.cpu().numpy()                     # original index order
            if np.isfinite(host).all():
                pos, mass = np.ascontiguousarray(host[:, :3]), np.ascontiguousarray(host[:, 3])
                o = Oracle()
                t = o.tree_build(pos, mass)
                for r in range(D.world):
                    s0 = sample_block(r * self.nl, self.nl, per_rank)[0]
                    ref = np.concatenate([o.tree_forces(t, pos, 0.5, i0=int(i), n_targets=1) for i in perm[s0:s0 + cnt]], 0)
                    g = gots[r].cpu().numpy()
                    err = max(err, rel_l2(g, ref) if np.isfinite(g).all() else float("inf"))
            else:
                err = float("inf")
        err = D.max(err)
        return {"rel_l2": err, "gate": 1e-3, "targets_per_rank": cnt,
                "oracle": "orc_tree_build_levels + orc_tree_forces on rank 0 (CPU restatement of TreeForceComputer; all "
                          "particles as gathered, put back in original index order)",
                "gather_checksums_ok": self.S.gather_checksums_ok(), "ok": bool(err <= 1e-3)}

    def close(self):
        if self.D.world > 1:
            self.eng.shard_finalize()


def c1_summary(eng, D, steps=10):
    """BASELINE configs[0]: DirectForceComputer, 16 384 uniform particles, 10 KDK leapfrog steps (dt 1e-3, eps
    0.01), device-resident between steps; wall clock around the 10 steps with a synchronise on both sides."""
    import b200grav
    from inputs import uniform_mt
    n = 16384
    pos = uniform_mt(n, seed=42)
    rng = np.random.default_rng(12345)
    vel = rng.normal(0.0, 100.0, size=(n, 3)).astype(np.float32)
    sim = b200grav.LambdaCDMSimulation(eng, pos, vel, np.ones(n, np.float32), force="direct", wrap=False)
    sim.step(1e-3)
    D.torch.cuda.synchronize()
    e0, e1 = D.torch.cuda.Event(enable_timing=True), D.torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sim.step(1e-3)
    e1.record()
    D.torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"workload": f"DirectForceComputer, {n} uniform particles, {steps} KDK leapfrog steps, dt 1e-3, eps 0.01, "
                        "open boundary, state device-resident (b200grav.LambdaCDMSimulation)",
            "ms_per_step": ms, "particle_steps_per_s": n / (ms * 1e-3),
            "interactions_per_s": float(n) * n / (ms * 1e-3), "steps": steps}


def c5_summary(eng, D, flush, n=1 << 23):
    """BASELINE configs[4]: DirectForceComputer 2^23 particles, strong scaling; ONE timed evaluation (24 s on one
    GPU) after a warm-up on 1/16 of the targets; NCCL all-gather of the shards inside the timed region."""
    torch = D.torch
    pos, mass = make_particles(n, seed=7)
    S = Sharded(D, np.ascontiguousarray(np.concatenate([pos, mass[:, None]], 1), np.float32), n)
    acc = torch.zeros((S.nl, 3), dtype=torch.float32, device=D.dev)
    S.gather()
    eng.direct_forces_dev(S.posm, acc, S.lo, max(1, S.nl // 16), eps=EPS)
    flush.zero_()
    S.poison()
    D.sync()
    eng.set_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    S.gather()
    eng.direct_forces_dev(S.posm, acc, S.lo, S.nl, eps=EPS)
    e1.record()
    torch.cuda.synchronize()
    kern_s = D.max(eng.last_kernel_ms()) * 1e-3
    eng.set_timing(False)
    t = D.max(e0.elapsed_time(e1)) * 1e-3
    out = {"workload": f"DirectForceComputer, {n} particles, uniform, unit masses, eps {EPS}, one evaluation; targets "
                       f"sharded over {D.world} GPU(s), sources all-gathered (NCCL)",
           "ms_per_step": 1e3 * t, "kernel_ms": 1e3 * kern_s, "interactions_per_s": float(n) * n / t, "steps": 1,
           "fp32_tflops_per_gpu_at_20_flop": 20.0 * float(S.nl) * n / kern_s / 1e12,
           "parity_check": parity_direct(D, S, acc, True)}
    del S, acc
    return out


def bench_gpu(args):
    import torch
    import torch.distributed as dist
    import b200grav

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly one JSON line: libraries that print there (NCCL's version banner) are
    # pointed at stderr for the whole run; the line itself goes to the saved descriptor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    D = Dist(torch, dist, world, rank, dev)
    eng = b200grav.Engine(local)

    n = args.particles
    if args.ic == "zeldovich":
        # generated on the device by the engine's own IC step (b200_zeldovich_ics_dev): every rank
        # produces the same replicated particle set (counter-based RNG), origin-centred convention
        posm0 = torch.empty((n, 4), dtype=torch.float32, device=dev)
        vel_ic = torch.empty((n, 3), dtype=torch.float32, device=dev)
        eng.zeldovich_ics_dev(posm0, vel_ic, n_particles=n, grid=zeldovich_grid(n), box=100.0,
                              z_initial=args.z_initial, seed=12345, origin_shift=50.0)
        del vel_ic
        torch.cuda.synchronize()
        posm_host = posm0.cpu().numpy()
        del posm0
        pos, mass = np.ascontiguousarray(posm_host[:, :3]), np.ascontiguousarray(posm_host[:, 3])
    else:
        pos, mass = make_particles(n, order=args.order)
        posm_host = np.ascontiguousarray(np.concatenate([pos, mass[:, None]], 1), np.float32)
    S = Sharded(D, posm_host, n)                            # full source set resident in HBM + this rank's shard
    posm, shard, lo, hi, nl = S.posm, S.shard, S.lo, S.hi, S.nl
    acc = torch.zeros((nl, 3), dtype=torch.float32, device=dev)
    vel = torch.zeros((nl, 3), dtype=torch.float32, device=dev)
    kdk = {"a": 1.0, "dt": 1e-4}                           # C4: a0 = 1, dt = 1e-4 (SURVEY 8d)
    flush = torch.empty(128 * 1024 * 1024, dtype=torch.float32, device=dev)   # 512 MB > 126 MB L2

    masses_equal = bool((mass == mass[0]).all())    # every rank holds the same (replicated) initial masses
    peers = None
    if world > 1 and args.sources == "peer" and args.workload == "direct":
        def _exchange(mine):
            out = [None] * world
            dist.all_gather_object(out, mine)
            return out
        _tok = torch.zeros(1, device=dev)
        peers = b200grav.PeerSources(eng, n, rank, world, lambda: dist.all_reduce(_tok), _exchange)

    def step():
        if peers is not None:       # fused: no all-gather, source tiles are pulled from peer HBM over NVLink
            if args.kdk:
                eng.leapfrog_dev(shard, vel, acc, nl, 2, np.float32(kdk["dt"] * 0.5), kdk["a"], np.float32(kdk["dt"]), 0.0)
                kdk["a"] = eng.scale_factor_step(kdk["a"], kdk["dt"])
            parts = peers.publish(shard)
            eng.direct_forces_parts_dev(parts, peers.lens, shard, nl, acc, eps=EPS, all_masses_equal=masses_equal)
            return
        if args.kdk:    # closing half-kick of the previous step + opening half-kick + drift, one pass
            eng.leapfrog_dev(shard, vel, acc, nl, 2, np.float32(kdk["dt"] * 0.5), kdk["a"], np.float32(kdk["dt"]), 0.0)
            kdk["a"] = eng.scale_factor_step(kdk["a"], kdk["dt"])
        S.gather()
        if args.workload == "direct":
            eng.direct_forces_dev(posm, acc, lo, nl, eps=EPS)
        else:
            eng.tree_build_dev(posm, n, 100.0, 8, 20)
            eng.tree_walk_dev(acc, lo, nl, theta=0.5)

    sync_all = D.sync

    # FP32 peak of this GPU, measured now (the roofline denominator)
    peak_ffma, _ = eng.fp32_peak_probe(0, 4000)
    peak_ffma2, _ = eng.fp32_peak_probe(1, 4000)
    peak = max(peak_ffma, peak_ffma2)

    for _ in range(max(args.warmup, 3)):
        S.poison()
        step()
    sync_all()

    sampler = ClockSampler(local)
    sampler.start()
    eng.set_timing(True)
    launches0 = eng.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms = []
    for k in range(args.steps):
        flush.zero_()                                      # evict L2 (untimed)
        S.poison()                                         # rows this rank does not own: NaN until the step's all-gather
        sync_all()
        ev[k][0].record()
        step()
        ev[k][1].record()
        torch.cuda.synchronize()
        kernel_ms.append(eng.last_kernel_ms())
    sync_all()
    launches = eng.launches - launches0
    eng.set_timing(False)
    sampler.stop()
    if args.dump_outputs:           # before anything below runs the step again
        rows, scalars = {"acc": acc}, None
        if args.kdk:
            rows.update(pos=shard[:, :3], vel=vel)
            scalars = {"scale_factor": kdk["a"]}
        dump_outputs(D, args.dump_outputs, n, rows, scalars)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_s = D.max(sum(step_ms)) * 1e-3
    kern_s = D.max(float(np.mean(kernel_ms))) * 1e-3
    clocks = sampler.summary()

    # ---- untimed: is the result of the last timed step right, and did the all-gather deliver? ----
    if args.workload == "direct":
        parity = parity_direct(D, S, acc, masses_equal) if peers is None else None
    else:
        parity = parity_tree(D, S, acc)

    # ---- end-to-end through the host-pointer C ABI ----
    pin_pos = torch.from_numpy(pos).pin_memory()
    pin_mass = torch.from_numpy(mass).pin_memory()
    pin_out = torch.empty((n if world == 1 else nl, 3), dtype=torch.float32).pin_memory()
    pin_shard = torch.from_numpy(posm_host[lo:hi].copy()).pin_memory()
    page_pos, page_mass = pos.copy(), mass.copy()           # plain malloc'd arrays: what the engine's unique_ptr<float[]> is
    page_out = np.empty((n, 3), np.float32)

    def e2e_step(pageable=False):
        if world == 1:
            p, m, o = (page_pos, page_mass, page_out) if pageable else (pin_pos.numpy(), pin_mass.numpy(), pin_out.numpy())
            if args.workload == "direct":
                eng.direct_forces_host(p, m, eps=EPS, out=o)
            else:
                eng.tree_forces_host(p, m, 0.5, 8, 20, 100.0, out=o)
        else:   # each rank owns its shard on the host: H2D shard, all-gather, kernels, D2H shard result
            shard.copy_(pin_shard, non_blocking=True)
            step()
            pin_out.copy_(acc, non_blocking=True)
            torch.cuda.synchronize()

    def e2e_time(pageable):
        e2e_step(pageable)
        sync_all()
        ts = []
        for _ in range(e2e_steps):
            flush.zero_()
            S.poison()
            sync_all()
            t0 = time.perf_counter()
            e2e_step(pageable)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return D.max(sum(ts))

    e2e_steps = max(2, min(args.steps, 5))
    e2e_s = e2e_time(False)
    e2e_page_s = e2e_time(True) if world == 1 and not args.kdk else None
    e2e_reg_s = None
    if e2e_page_s is not None:      # the same plain arrays, page-locked in place once (b200_host_register: what the
        for a in (page_pos, page_mass, page_out):       # plugin's set_pin_host_arrays(true) does on first sight)
            eng.host_register(a)
        e2e_reg_s = e2e_time(True)
        for a in (page_pos, page_mass, page_out):
            eng.host_unregister(a)

    tree_counts = None
    if args.workload == "direct":
        per_step = float(n) * float(n)                      # whole job: all targets x all sources
        per_launch = float(nl) * float(n)                   # this rank's main kernel
    else:
        eng.tree_set_counting(True)
        eng.tree_walk_dev(acc, lo, nl, theta=0.5)
        torch.cuda.synchronize()
        tree_counts = eng.tree_walk_stats()
        eng.tree_set_counting(False)
        per_launch = float(tree_counts[1] + tree_counts[2])
        per_step = D.sum(per_launch)

    line = None
    if rank == 0:
        value = per_step * args.steps / total_s
        e2e_value = per_step * e2e_steps / e2e_s
        line = {
            "metric": "pairwise_interactions_per_s", "value": value, "unit": "interactions/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": 1e3 * total_s / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args),
            "particle_steps_per_s": float(n) * args.steps / total_s,
            "e2e": {"value": e2e_value, "unit": "interactions/s",
                    "h2d_bytes_per_step": int(16 * n) if world == 1 else int(16 * nl) * world,
                    "d2h_bytes_per_step": int(12 * n), "ms_per_step": 1e3 * e2e_s / e2e_steps,
                    "api": (("b200_direct_forces_host" if args.workload == "direct" else "b200_tree_forces_host") +
                            " (pinned host buffers)") if world == 1 else
                           "per-rank pinned shard H2D + NCCL all-gather + b200_*_dev + D2H"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "parity_check": parity,
        }
        if e2e_page_s is not None:
            line["e2e_pageable"] = {
                "value": per_step * e2e_steps / e2e_page_s, "unit": "interactions/s",
                "ms_per_step": 1e3 * e2e_page_s / e2e_steps,
                "api": "the same call on plain (pageable) host arrays -- what IForceComputer::compute_forces receives "
                       "from the engine's unique_ptr<float[]> (simulation_engine.hpp:60-63)"}
            line["e2e_registered"] = {
                "value": per_step * e2e_steps / e2e_reg_s, "unit": "interactions/s",
                "ms_per_step": 1e3 * e2e_reg_s / e2e_steps,
                "api": "the same plain arrays after one b200_host_register (cudaHostRegister in place; the plugin's opt-in "
                       "set_pin_host_arrays(true), switched on by integration/engine_wiring.patch for the engine's arrays)"}
    if args.workload == "direct":
        if rank == 0:
            achieved = FLOP_PER_INTERACTION * per_launch / kern_s / 1e12
            line["roofline"] = {
                "bound": "fp32_fma",
                "kernel": ("direct_kernel<R=8,THREADS=256,1 CTA/SM,open,equal-mass> (11 FP32 lane-ops + 1 MUFU per "
                           "interaction; unequal masses run the 12-op instance)"),
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": ncu_static("direct", n) if world == 1 and args.ic == "uniform" else None,
                "peak_source": "FFMA/FFMA2 register-chain probe run in this process (b200_fp32_peak_probe: the builder's "
                               "own probe); MEASURED_PEAKS.json has no FP32 figure",
                "peak_ffma": peak_ffma, "peak_ffma2": peak_ffma2,
                "nominal_peak": 148 * 128 * 2 * (clocks.get("sm_max_mhz") or 1965) * 1e6 / 1e12,
                "flop_per_interaction": FLOP_PER_INTERACTION,
                "kernel_ms": 1e3 * kern_s,
            }
    else:
        rl = walk_roofline(eng, D, n, nl, tree_counts, kern_s, clocks, world == 1 and args.ic == "uniform"
                           and args.order == "random")
        if rank == 0:
            line["roofline"] = rl

    # ---- the other BASELINE configs, each a short measurement of its own (collective: every rank takes part) ----
    extras = args.workload == "direct" and not args.kdk and not args.no_extras and args.ic == "uniform" \
        and peers is None and n == (1 << 20)
    if extras:
        del pin_pos, pin_mass, pin_out, pin_shard
        ts = tree_summary(eng, D, S, flush, clocks=clocks, static_ok=(args.order == "random"))
        lf = leapfrog_roofline(eng, D, (1 << 24) // world)
        c4 = c4_summary(eng, D, flush, 1 << 24, 8, args.c4_mode)
        # the round-1 scheme (index shards, every rank builds the whole tree) beside it, where the two differ
        c4_rep = c4_summary(eng, D, flush, 1 << 24, 4, "replicated") if world > 1 and args.c4_mode == "sharded" else None
        c5 = c5_summary(eng, D, flush) if not args.no_c5 else None
        box_line = c1 = None
        if world == 1:
            # the [0,100) convention the reference's generators emit (initial_conditions.cpp:808-820): 7/8 of the
            # particles lie outside the origin-centred root cube and end in max-depth overflow leaves
            pb, mb = make_particles(n, seed=43)
            Sb = Sharded(D, np.ascontiguousarray(np.concatenate([pb + np.float32(50.0), mb[:, None]], 1), np.float32), n)
            box_line = tree_summary(eng, D, Sb, flush, steps=3, label="box convention [0,100)^3", clocks=clocks)
            del Sb
            c1 = c1_summary(eng, D)
        if rank == 0:
            line["tree_summary"] = ts
            line["leapfrog_roofline"] = lf
            line["c4_summary"] = c4
            if c4_rep is not None:
                line["c4_summary_replicated_build"] = c4_rep
            if c5 is not None:
                line["c5_summary"] = c5
            if box_line is not None:
                line["tree_box_convention_summary"] = box_line
                line["c1_summary"] = c1
    if rank == 0:
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = run_cpu_baseline(args.workload)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        if peers is not None:
            peers.close()
        dist.destroy_process_group()
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="direct", choices=["direct", "tree"])
    ap.add_argument("--particles", type=int, default=1 << 20)
    ap.add_argument("--ic", default="uniform", choices=["uniform", "zeldovich"],
                    help="synthetic inputs: uniform random (default) or Zel'dovich initial conditions generated on "
                         "the device")
    ap.add_argument("--z-initial", type=float, default=49.0, help="redshift of the Zel'dovich ICs")
    ap.add_argument("--order", default="random", choices=["random", "morton"],
                    help="index order of the uniform particles: as drawn (default) or sorted along a Morton curve")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", "--no-tree-summary", dest="no_extras", action="store_true",
                    help="default (direct, 2^20) run: skip the short measurements of the other BASELINE configs "
                         "(tree_summary, c4_summary, c5_summary, c1_summary, leapfrog_roofline)")
    ap.add_argument("--no-c5", action="store_true", help="skip c5_summary (2^23-particle direct sum: 24 s on one GPU)")
    ap.add_argument("--c4-mode", default="sharded", choices=["replicated", "sharded"],
                    help="c4_summary: every rank builds the whole octree on contiguous index shards (round-1 scheme), "
                         "or octant-sharded build + Hilbert-owned targets")
    ap.add_argument("--sources", default="allgather", choices=["allgather", "peer"],
                    help="N>1 direct sum: NCCL all-gather of the shards (default) or peer-mapped source tiles "
                         "pulled over NVLink by the force kernel itself")
    ap.add_argument("--kdk", action="store_true",
                    help="each step is a full Lambda-CDM KDK leapfrog step (fused kick-kick-drift pass, scale-factor "
                         "update, source all-gather, force evaluation) instead of a bare force evaluation")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the last timed step computed (forces; with --kdk "
                         "also positions, velocities and the scale factor) as DIR/<name>.npy, at most 64 MB in all "
                         "(a fixed, seeded sample of rows beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl b200)")
    if args.impl == "reference":
        bench_reference(args)
    else:
        bench_gpu(args)


if __name__ == "__main__":
    main()
