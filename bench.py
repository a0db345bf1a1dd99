#!/usr/bin/env python
"""bench.py — million particle-updates/s of the MLS-MPM substep hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload sand256]

A "step" is one substep (sort -> P2G -> grid update -> G2P+constitutive -> delete) over the whole
synthetic particle set.  Workload = BASELINE config 3 (256^3 grid, 8 M Drucker-Prager sand), the config
the metric is quoted on; --gpus N cuts the SAME scene into N z-slabs (strong scaling, the metric's
"1/2/4/8 GPU"; `weak_scaling` is reported beside it).  Prints ONE JSON line (rank 0).

  value     whole-job M particle-updates/s, state resident in HBM, CUDA-event timed, max over ranks:
            the SLOWER of two states of the same scene — the column at rest and a developed collapse
            (`states`: movers per substep, active tiles, hole fraction of each)
  parity_check (N > 1)  a reduced scene on the N-rank exchange path against one engine, per particle id,
            BEFORE any timing; a mismatch ends the run with rc 3
  e2e       same metric through the drop-in's own calls with HOST buffers: one frame = mpmb_upload_aos of
            the reference's 320-byte-slot pool from pinned host memory + frame_substeps substeps +
            mpmb_download_aos back into it (the adapter's per-frame contract, INTEGRATION.md §2)
  roofline  dominant kernel: algorithmic bytes / CUDA-event duration vs measured HBM peak
  cpu_baseline  the OpenMP restatement of the reference's optimized CPU path (oracle "port"),
            timed on this box's host cores on a bounded sample
  --impl reference  times that CPU path alone (the reference cannot be built here: DESIGN.md §2)
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from taichi_mpm_b200 import scenes  # noqa: E402

BYTES_PER_UPDATE = {scenes.MAT_LINEAR: 208, scenes.MAT_JELLY: 208, scenes.MAT_SAND: 216, scenes.MAT_SNOW: 216, scenes.MAT_WATER: 144}
# split of the per-update figure between the two hot kernels (DESIGN.md §5): P2G reads the state
# (+mass, vol) and writes half of the grid traffic, G2P writes the state and reads the other half.
P2G_BYTES = {scenes.MAT_LINEAR: 108, scenes.MAT_JELLY: 108, scenes.MAT_SAND: 112, scenes.MAT_SNOW: 112, scenes.MAT_WATER: 76}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {}
        for n in dir(nv):
            if n.startswith("nvmlClocksEventReason") or n.startswith("nvmlClocksThrottleReason"):
                v = getattr(nv, n)
                if isinstance(v, int) and v and n not in ("nvmlClocksEventReasonAll", "nvmlClocksThrottleReasonAll"):
                    names.setdefault(v, n.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", ""))
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit and "None" not in name and "Idle" not in name:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# the reference re-packs its particle pool in sorted order every `reorder_interval` substeps, the first
# time at substep 0 (src/mpm.cpp:45,811-813); the CPU arms keep that default
REORDER_INTERVAL = 1000


def usable_cpus():
    """Host threads this process can really use: affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return max(1, n)


def best_thread_count(sc, probe):
    """Oversubscribed OpenMP teams collapse on shared boxes (measured: 128 threads were 200x slower
    than 64 here), so the CPU arm probes a few team sizes on a small sample and keeps the fastest."""
    from oracle import pyoracle as O
    cand = sorted({max(1, usable_cpus() // d) for d in (1, 2, 4, 8)}, reverse=True)
    best, best_rate = cand[-1], 0.0
    for t in cand:
        f = O.FastOracle(sc, probe, threads=t, reorder_interval=REORDER_INTERVAL)
        f.substeps(2)  # team start-up, first touch and the storage re-order are not part of the rate
        rate = 0.0
        for _ in range(3):  # best of three short runs: the probe must not be decided by one hiccup
            t0 = time.perf_counter()
            upd, tm = f.substeps(2)
            rate = max(rate, upd / (time.perf_counter() - t0 - tm[4]))
        del f
        if rate > best_rate:
            best, best_rate = t, rate
    return best, best_rate


def build_workload(name, scale, state=True):
    cfg = scenes.config(name, scale, state=state)
    sc = cfg["scene"]
    if sc["planes"] is not None:
        sc["sdf"] = None  # engine builds the dense level set on the device from the planes
    return cfg


# slot layout of the reference's particle pool: offsetof() on MPMParticle<3> / SandParticle<3> ... in the in-place build
# of the reference sources (oracle/transfer_ref.cpp: reft_aos_layout; INTEGRATION.md §2) — stride, pos, v_and_m, dg_e,
# apic_b, column pitch, vol, plastic scalar per kind
AOS_SLOT = dict(stride=320, off_pos=32, off_v_and_m=16, off_dg_e=48, off_apic_b=96, col_pitch=16, off_vol=164)
AOS_SCALAR = {scenes.MAT_LINEAR: -1, scenes.MAT_JELLY: -1, scenes.MAT_SNOW: 196, scenes.MAT_WATER: 204, scenes.MAT_SAND: 216}

# --dump-outputs: particles written per run (120 bytes each: 31 MB for 262144) and the seed that picks them
OUTPUT_SAMPLE = 262144
OUTPUT_SEED = 20240917


def dump_outputs(directory, arrays):
    """One DIR/<name>.npy per array (float32 / float64)."""
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a)


def slab_cuts(meta, res_z, world, weak):
    """Tile-layer cuts [(z0, z1)] * world by particle count: 1-D histogram of the base tile layer of the block's cell
    layers (all columns are statistically identical).  weak: the block is `world` times longer along z."""
    from taichi_mpm_b200 import slab
    dx = 1.0 / meta["res"]
    lo_z, hi_z = meta["lo"][2], meta["hi"][2]
    zs = (np.arange(lo_z, hi_z)[:, None] + 0.5 + np.array([-0.25, 0.25])[None]).reshape(-1) * dx
    return slab.slab_partition(slab.base_tile_z(zs, dx), slab.tile_layers(res_z), world)


def weak_variant(cfg, world):
    """The weak-scaling version of a config: grid res x res x (res*world), block cells x cells x (cells_z*world)."""
    cfg = dict(scene=dict(cfg["scene"]), state=None, meta=dict(cfg["meta"]))
    res = cfg["meta"]["res"]
    lo, hi = list(cfg["meta"]["lo"]), list(cfg["meta"]["hi"])
    cells_z = hi[2] - lo[2]
    lo[2] = (res * world - cells_z * world) // 2
    hi[2] = lo[2] + cells_z * world
    cfg["scene"]["res"] = (res, res, res * world)
    cfg["meta"]["lo"], cfg["meta"]["hi"] = tuple(lo), tuple(hi)
    cfg["meta"]["n"] = cfg["meta"]["n"] * world
    return cfg


def cpu_run(cfg, n_particles_cap, budget_s, min_substeps=1, threads=None):
    """Times the oracle's OpenMP fast path on (a sub-block of) the workload."""
    from oracle import pyoracle as O
    st, sc = cfg["state"], dict(cfg["scene"])
    n = len(st["x"])
    if n > n_particles_cap:
        # bounded sample: the lowest layers of the column (keeps the floor contact), contiguous in y
        order = np.argsort(st["x"][:, 1], kind="stable")[:n_particles_cap]
        st = {k: v[order] for k, v in st.items()}
    if sc.get("planes") is not None:
        sc["sdf"] = scenes.planes_sdf(sc["res"], sc["planes"])
    if threads is None:
        probe = {k: v[: min(len(v), 300_000)] for k, v in st.items()}
        threads, _ = best_thread_count(sc, probe)
    fast = O.FastOracle(sc, st, threads=threads, reorder_interval=REORDER_INTERVAL)
    t0 = time.perf_counter()
    upd, tm = fast.substeps(1)  # first substep also pays first-touch of the buffers: untimed warm-up
    warm = time.perf_counter() - t0
    nsub = max(min_substeps, int(min(50, budget_s / max(warm, 1e-3))))
    t0 = time.perf_counter()
    upd, tm = fast.substeps(nsub)
    dt = time.perf_counter() - t0 - tm[4]  # minus the harness' copy between caller arrays and the pool
    # one-thread figure, as the reference's own benchmark script runs (scripts/benchmark/benchmark_3d.py:17)
    single = None
    try:
        small = {k: v[: min(len(v), 200_000)] for k, v in st.items()}
        f1 = O.FastOracle(sc, small, threads=1, reorder_interval=REORDER_INTERVAL)
        f1.substeps(1)
        t0 = time.perf_counter()
        u1, tm1 = f1.substeps(2)
        single = u1 / (time.perf_counter() - t0 - tm1[4]) / 1e6
        del f1
    except Exception:
        pass
    return dict(value=upd / dt / 1e6, seconds=dt, substeps=nsub, particles=len(st["x"]), threads=fast.threads, single_thread=single,
                ns_per_particle=dict(sort=tm[0] / upd * 1e9, p2g=tm[1] / upd * 1e9, grid=tm[2] / upd * 1e9, g2p=tm[3] / upd * 1e9))


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path = the oracle port
    (the taichi-legacy core is not vendored, so the reference binary cannot be built)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = build_workload(args.workload, args.scale)
    n_full = len(cfg["state"]["x"])
    from oracle import pyoracle as O
    st, sc = cfg["state"], dict(cfg["scene"])
    if sc.get("planes") is not None:
        sc["sdf"] = scenes.planes_sdf(sc["res"], sc["planes"])
    # pick the team size, then calibrate the sample so that (steps+warmup) substeps take about a minute
    probe_n = min(n_full, 300_000)
    order = np.argsort(st["x"][:, 1], kind="stable")
    probe = {k: v[order[:probe_n]] for k, v in st.items()}
    threads, rate = best_thread_count(sc, probe)
    per_particle = 1.0 / rate
    total = args.steps + args.warmup
    n_sample = int(min(n_full, max(50_000, 60.0 / (per_particle * total))))
    sample = {k: v[order[:n_sample]] for k, v in st.items()}
    fast = O.FastOracle(sc, sample, threads=threads, reorder_interval=REORDER_INTERVAL)
    fast.substeps(args.warmup)
    t0 = time.perf_counter()
    upd, tm = fast.substeps(args.steps)
    dt = time.perf_counter() - t0 - tm[4]  # minus the harness' copy between caller arrays and the pool
    val = upd / dt / 1e6
    sample_txt = "%d of %d particles (lowest layers of the column), every substep over the sample, %d OpenMP threads" % (
        n_sample, n_full, fast.threads)
    line = {
        "impl": "reference", "metric": "million particle-updates/s", "value": val, "unit": "M particle-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, cfg, n_full, args.gpus, args.scaling == "weak"),
        "cpu_baseline": {"value": val, "unit": "M particle-updates/s", "cores": fast.threads, "kind": "port", "sample": sample_txt,
                         "ns_per_particle": {"sort": tm[0] / upd * 1e9, "p2g": tm[1] / upd * 1e9, "grid": tm[2] / upd * 1e9,
                                             "g2p": tm[3] / upd * 1e9}},
        "e2e": {"value": val, "unit": "M particle-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    rb = reference_build_rate(sc, sample, fast.threads)
    if rb is not None:
        line["cpu_baseline"]["reference_build"] = rb
    emit(line)


def reference_build_rate(sc, sample, threads, n=400_000, substeps=3):
    """The reference's OWN solver sources compiled in place (oracle/_ref/libtransfer_ref.so, DESIGN.md §2), timed on
    a sample with the same number of threads as the port: MPM<3>::substep() itself, its 8-colour P2G and block-parallel
    G2P running on the stand-in's OpenMP task loops.  It is the parity checker, not a tuned build (stand-in core:
    double-precision SVD, generic matrix code), so it is slower than the port; the port stays the quoted baseline."""
    try:
        from oracle import pyoracle as O
        if not O.ref_transfer_available():
            return None
        small = {k: v[:n] for k, v in sample.items()}
        s = O.RefSolver(sc, small)
        try:
            s.set_threads(threads)
            s.substep(1)
            t0 = time.perf_counter()
            alive = s.substep(substeps)
            dt = time.perf_counter() - t0
        finally:
            s.set_threads(1)
            s.close()
        return {"value": alive * substeps / dt / 1e6, "unit": "M particle-updates/s", "cores": int(threads), "kind": "reference",
                "sample": "%d particles, %d substeps of MPM<3>::substep()" % (len(small["x"]), substeps),
                "note": "reference sources compiled in place against the stand-in core (checker build, not the baseline)"}
    except Exception as ex:  # the checker build is optional for the bench
        return {"unavailable": str(ex)[:200]}


def workload_config(args, cfg, n_particles, world=1, weak=False):
    m = cfg["meta"]
    if world == 1:
        par = "1 GPU"
    elif weak:
        par = "z-slab x%d (weak scaling: block and grid extended along z, one config-sized share per GPU)" % world
    else:
        par = "z-slab x%d (strong scaling: the SAME %d-particle scene cut into %d slabs of equal particle count)" % (world, n_particles, world)
    return {"workload": "%s: %s grid, %d particles, %s, dt=%g, floor plane friction %g" % (
        m["name"], "x".join(str(r) for r in cfg["scene"]["res"]), n_particles, ["linear", "jelly", "snow", "water", "sand"][m["kind"]], cfg["scene"]["dt"],
        cfg["scene"]["friction"]),
        "l2": "inputs larger than L2 (particle state %.0f MB per buffer per GPU vs 126 MB L2)" % (n_particles * 112 / 1e6 / world),
        "parallelism": par}


class SlabJob:
    """One rank's engine over (its slab of) a config, seeded on the device (mpmb_seed_lattice): no host particle arrays."""

    def __init__(self, args, cfg, rank, world, local, dist, weak=False, v0=(0.0, 0.0, 0.0)):
        import torch
        from taichi_mpm_b200 import capi, slab
        self.torch, self.dist, self.rank, self.world = torch, dist, rank, world
        self.cfg = weak_variant(cfg, world) if (weak and world > 1) else cfg
        sc, m = self.cfg["scene"], self.cfg["meta"]
        self.dev = torch.device("cuda", local)
        self.stream = torch.cuda.current_stream(self.dev)
        if world == 1:
            self.eng = capi.Engine(sc["res"], sc["dx"], sc["dt"], sc["gravity"], sc["particle_gravity"], True, device=local)
        else:
            z0, z1 = slab_cuts(m, sc["res"][2], world, weak)[rank]
            self.eng = capi.Engine(sc["res"], sc["dx"], sc["dt"], sc["gravity"], sc["particle_gravity"], True, device=local, rank=rank, world=world,
                                   tile_z0=z0, tile_z1=z1, migrate_capacity=args.migrate_capacity, halo_capacity=args.halo_capacity)
        e = self.eng
        e.set_stream(self.stream.cuda_stream)
        if world > 1:
            if args.exchange == "peer":
                slab.connect_peers(e, rank, world, dist)  # neighbours' receive buffers mapped over NVLink (CUDA IPC)
            else:
                self.runner = slab.SlabRunner(slab.EngineAdapter(e), rank, world, self.dev, dist=dist)
        self.peer = world == 1 or args.exchange == "peer"
        e.set_material(0, m["kind"], sc["mat_params"][0])
        if sc["planes"] is not None:
            e.set_planes(sc["planes"], sc["friction"])
        self.n_local = e.seed_lattice(m["lo"], m["hi"], m["vol"], m["mass"], jitter=m["jitter"], seed=m["seed"], v0=v0)
        self.n_total = int(self.allsum([self.n_local])[0])
        self.barrier()  # peer-memory waits are bounded: start the ranks together

    def allsum(self, vals, op=None):
        t = self.torch.tensor([float(v) for v in vals], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=op or self.dist.ReduceOp.SUM)
        return [float(v) for v in t.cpu()]

    def allmax(self, vals):
        return self.allsum(vals, op=self.dist.ReduceOp.MAX if self.world > 1 else None)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def substep(self, k):
        if k <= 0:
            return
        if self.peer:
            self.eng.substep(k)
        else:
            self.runner.substep(k)

    def timed(self, steps, warmup, sample_clocks=True, keep_outputs=False):
        """W untimed + K timed substeps, barrier + synchronize on both sides, CUDA events, max over ranks.
        keep_outputs: the particle state right after the K-th timed substep is kept in self.outputs (a sample, see
        sample_outputs) before the per-stage pass below moves the scene on."""
        torch, e = self.torch, self.eng
        self.substep(warmup)
        self.barrier()
        c0 = e.get_counters()
        sampler = ClockSampler(self.dev.index)
        if sample_clocks:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record(self.stream)
        self.substep(steps)          # THE timed region: K substeps, one C-ABI call, no per-stage events inside
        ev1.record(self.stream)
        self.barrier()
        clocks = sampler.stop() if sample_clocks else None
        ms_local = ev0.elapsed_time(ev1)
        c1 = e.get_counters()
        if keep_outputs:
            self.outputs = self.sample_outputs()
        # per-stage split: the same K substeps once more with CUDA events around every stage (untimed for `value`:
        # the event records cost a few microseconds per stage and switch the graph replay off)
        e.set_profiling(True)
        e.get_profile(reset=True)
        self.substep(steps)
        stage_ms, _ = e.get_profile(reset=True)
        e.set_profiling(False)
        st = e.get_ordering_stats()
        ms = self.allmax([ms_local])[0]
        alive, launches, tiles, movers, rows = self.allsum([c1["alive"], c1["kernel_launches"] - c0["kernel_launches"], c1["active_tiles"], st["movers"], st["rows"]])
        per = [v / max(steps, 1) for v in stage_ms]
        return dict(ms=ms, ms_per_step=ms / steps, value=alive * steps / (ms * 1e-3) / 1e6, alive=int(alive), alive_local=c1["alive"], launches=int(launches),
                    active_tiles=int(tiles), movers_per_substep=int(movers), hole_fraction=movers / max(rows, 1.0),
                    stage_ms_per_step={"sort+tiles": per[0], "p2g": per[1], "g2p": per[2], "exchange": per[3], "grid": per[4]}, clocks=clocks)

    def gather_particles(self, keys=("id", "x", "v", "F", "ps")):
        d = self.eng.download(sort_by_id=False)
        mine = {k: d[k] for k in keys}
        if self.world == 1:
            return mine
        parts = [None] * self.world
        self.dist.all_gather_object(parts, mine)
        return {k: np.concatenate([p[k] for p in parts]) for k in keys} if self.rank == 0 else None

    def sample_outputs(self, count=OUTPUT_SAMPLE):
        """What mpmb_download_particles hands a caller, for a fixed seeded sample of particle ids (the whole set when it is
        smaller), in id order, gathered on rank 0.  Particle ids are the seeding order, so two builds sample the same particles."""
        keys = ("id", "x", "v", "F", "b", "mass", "vol", "ps", "group")
        d = self.eng.download(sort_by_id=False)
        if self.n_total > count:
            want = np.sort(np.random.default_rng(OUTPUT_SEED).choice(self.n_total, count, replace=False))
            keep = np.isin(d["id"], want)
            d = {k: d[k][keep] for k in keys}
        mine = {k: d[k] for k in keys}
        if self.world > 1:
            parts = [None] * self.world
            self.dist.all_gather_object(parts, mine)
            if self.rank != 0:
                return None
            mine = {k: np.concatenate([p[k] for p in parts]) for k in keys}
        o = np.argsort(mine["id"], kind="stable")
        return {k: mine[k][o].astype(np.float64 if k == "id" else np.float32) for k in keys}

    def close(self):
        self.eng.close()


def multi_gpu_parity_check(args, rank, world, local, dist):
    """Before any timing at N > 1: a reduced scene on the N-rank path (halo exchange + migration, the transport the bench
    times) against ONE engine on rank 0, per particle id.  Uniform initial velocity along +z so that particles cross
    every slab face.  Tolerances = tests/test_gpu_slab.py (the visiting order of arrivals differs between partitions)."""
    scale, nsub = 0.5, 60
    cfg = build_workload(args.workload, scale, state=False)
    v0 = (0.5, 0.0, 12.0)
    job = SlabJob(args, cfg, rank, world, local, dist, weak=False, v0=v0)
    n0 = job.n_local
    job.substep(nsub)
    got = job.gather_particles()
    n1 = job.eng.num_particles()
    crossed = job.allsum([abs(n1 - n0)])[0]
    job.close()
    res = None
    if rank == 0:
        one = SlabJob(args, cfg, 0, 1, local, None, v0=v0)
        one.substep(nsub)
        ref = one.gather_particles()
        one.close()
        o, r = np.argsort(got["id"], kind="stable"), np.argsort(ref["id"], kind="stable")
        same_ids = len(o) == len(r) and np.array_equal(got["id"][o], ref["id"][r])
        err = {}
        if same_ids:
            vmax = max(float(np.abs(ref["v"]).max()), 1e-30)
            err = {"x": float(np.abs(got["x"][o] - ref["x"][r]).max()), "v_rel": float(np.abs(got["v"][o] - ref["v"][r]).max() / vmax),
                   "F": float(np.abs(got["F"][o] - ref["F"][r]).max()), "ps": float(np.abs(got["ps"][o] - ref["ps"][r]).max())}
        tol = {"x": 2e-6, "v_rel": 5e-4, "F": 5e-5, "ps": 1e-5}
        ok = bool(same_ids and all(err[k] <= tol[k] for k in tol) and crossed > 0)
        res = {"ok": ok, "particles": int(len(r)), "substeps": nsub, "ranks": world, "same_ids": bool(same_ids), "max_err": err, "tol": tol,
               "net_particles_exchanged": int(crossed), "scene": "%s x%g, v0=%s, %s exchange vs one engine on rank 0" % (args.workload, scale, v0, args.exchange)}
    flag = job.torch.tensor([1.0 if (res is None or res["ok"]) else 0.0], device=job.dev)
    dist.broadcast(flag, 0)
    return res, bool(flag.item() > 0)


def aos_e2e(job, args, kind):
    """End to end through the drop-in's own calls (N = 1): the reference's 320-byte-slot pool in pinned host memory,
    mpmb_upload_aos -> frame_substeps substeps -> mpmb_download_aos per frame (INTEGRATION.md §2)."""
    import torch
    from taichi_mpm_b200 import capi
    e = job.eng
    n = e.num_particles()
    L = capi.MpmbAosLayout()
    for k, v in AOS_SLOT.items():
        setattr(L, k, v)
    L.off_scalar = AOS_SCALAR[kind]
    pool_t = torch.zeros(n * L.stride, dtype=torch.uint8, pin_memory=True)
    idx_t = torch.empty(n, dtype=torch.int32, pin_memory=True)
    pool, idx = pool_t.numpy(), idx_t.numpy().view(np.uint32)
    # the host pool starts as the engine's current state: ids -> slots 0..n-1 in id order
    d_id = np.sort(e.download(sort_by_id=False)["id"])
    remap = np.full(int(d_id.max()) + 1 if n else 1, 0, np.uint32)
    remap[d_id] = np.arange(n, dtype=np.uint32)
    idx_full = remap            # id -> slot
    nn = e.download_aos(pool, idx_full, L)  # (not resident: reads the zero pool, scatters, returns it)
    assert nn == n
    idx[:] = np.arange(n, dtype=np.uint32)
    times = []
    alive = n
    for f in range(args.frames + 1):
        job.barrier()
        t0 = time.perf_counter()
        e.upload_aos(pool, idx[:alive], L)
        e.substep(args.frame_substeps)
        alive = e.download_aos(pool, idx[:alive], L)
        job.barrier()
        if f > 0:   # frame 0 warms the staging buffers
            times.append(time.perf_counter() - t0)
    sec = float(np.median(times))
    return dict(value=alive * args.frame_substeps / sec / 1e6, frame_seconds=sec, frame_seconds_all=[float(t) for t in times],
                h2d=n * (L.stride + 4), d2h=n * (L.stride + 4), alive=alive,
                path="mpmb_upload_aos -> mpmb_substep(%d) -> mpmb_download_aos on a pinned pool of %d-byte slots" % (args.frame_substeps, L.stride))


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    weak = args.scaling == "weak"
    cfg = build_workload(args.workload, args.scale, state=False)
    kind = cfg["meta"]["kind"]

    parity = None
    if world > 1 and not args.no_parity_check:
        parity, ok = multi_gpu_parity_check(args, rank, world, local, dist)
        if not ok:
            if rank == 0:
                emit({"error": "multi-GPU parity check failed", "parity_check": parity})
            dist.barrier()
            dist.destroy_process_group()
            sys.exit(3)

    job = SlabJob(args, cfg, rank, world, local, dist if world > 1 else None, weak=weak)
    n_total = job.n_total
    # ---- device-resident throughput, column at rest (the round-1 regime) ...
    dump = args.dump_outputs is not None
    quiet = job.timed(args.steps, args.warmup, keep_outputs=dump and args.develop <= 0)
    # ---- ... and in a developed collapse: advance the same engine `develop` substeps, then time again
    flowing = None
    if args.develop > 0:
        job.substep(args.develop)
        flowing = job.timed(args.steps, args.warmup, keep_outputs=dump)
        flowing["developed_substeps"] = 2 * (args.warmup + args.steps) + args.steps + args.develop   # substeps behind the scene when its timed region starts
    head = quiet if (flowing is None or quiet["value"] <= flowing["value"]) else flowing
    head_name = "quiescent" if head is quiet else "flowing"

    # ---- end to end through host buffers
    e2e = None
    if args.frames > 0:
        if world == 1:
            r = aos_e2e(job, args, kind)
            e2e = {"value": r["value"], "unit": "M particle-updates/s", "h2d_bytes_per_step": r["h2d"] / args.frame_substeps,
                   "d2h_bytes_per_step": r["d2h"] / args.frame_substeps, "frame_substeps": args.frame_substeps, "frames": args.frames,
                   "frame_seconds": r["frame_seconds"], "frame_seconds_all": r["frame_seconds_all"], "path": r["path"],
                   "state": "flowing" if flowing else "quiescent"}
        else:
            e2e = soa_e2e(job, args)

    # ---- secondary: weak scaling of the same config (N > 1, default run only)
    weak_line = None
    if world > 1 and not weak and args.also_weak:
        wjob = SlabJob(args, cfg, rank, world, local, dist, weak=True)
        w = wjob.timed(args.steps, args.warmup, sample_clocks=False)
        weak_line = {"value": w["value"], "ms_per_step": w["ms_per_step"], "particles": wjob.n_total, "stage_ms_per_step": w["stage_ms_per_step"],
                     "config": workload_config(args, wjob.cfg, wjob.n_total, world, True)["workload"]}
        wjob.close()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    if dump:
        dump_outputs(args.dump_outputs, job.outputs)
    peaks, peak_kind = measured_peaks()
    peak = float(peaks["hbm_gbs"])
    # dominant kernel of the (headline state's) substep on rank 0
    kms = {"p2g": head["stage_ms_per_step"]["p2g"], "g2p": head["stage_ms_per_step"]["g2p"]}
    dom = max(kms, key=kms.get)
    kb = P2G_BYTES[kind] if dom == "p2g" else BYTES_PER_UPDATE[kind] - P2G_BYTES[kind]
    achieved = kb * head["alive_local"] / (kms[dom] * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get(dom)
        except Exception:
            traffic = None
    value = head["value"]
    roofline = {"bound": "hbm", "kernel": "k_" + dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)" if peak_kind == "measured" else "fallback 6650",
                "algorithmic_bytes_per_launch": kb * head["alive_local"], "kernel_ms": kms[dom],
                "substep": {"bytes_per_update": BYTES_PER_UPDATE[kind], "achieved": BYTES_PER_UPDATE[kind] * value * 1e6 / 1e9 / world,
                            "frac": BYTES_PER_UPDATE[kind] * value * 1e6 / 1e9 / world / peak, "note": "per GPU"},
                "stage_ms_per_step": head["stage_ms_per_step"], "state": head_name}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        hcfg = build_workload(args.workload, args.scale, state=True)
        r = cpu_run(hcfg, args.cpu_sample, budget_s=15.0)
        cpu = {"value": r["value"], "unit": "M particle-updates/s", "cores": r["threads"], "kind": "port",
               "sample": "%d of %d particles (lowest layers of the column), %d substeps, %.1f s" % (r["particles"], n_total, r["substeps"], r["seconds"]),
               "ns_per_particle": r["ns_per_particle"], "single_thread_value": r["single_thread"]}

    def state_line(t):
        return {k: t[k] for k in ("value", "ms_per_step", "alive", "active_tiles", "movers_per_substep", "hole_fraction", "stage_ms_per_step") if k in t} | (
            {"developed_substeps": t["developed_substeps"]} if "developed_substeps" in t else {})

    line = {
        "metric": "million particle-updates/s", "value": value, "unit": "M particle-updates/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (device-seeded lattice, mpmb_seed_lattice)",
        "config": workload_config(args, job.cfg, n_total, world, weak),
        "roofline": roofline, "cpu_baseline": cpu, "clocks": head["clocks"], "e2e": e2e,
        "gpu_launches": head["launches"], "alive_particles": head["alive"], "active_tiles": head["active_tiles"],
        "states": {"headline": head_name + " (the slower of the two)", "quiescent": state_line(quiet), "flowing": state_line(flowing) if flowing else None},
    }
    if parity is not None:
        line["parity_check"] = parity
    if weak_line is not None:
        line["weak_scaling"] = weak_line
    if world > 1:
        line["exchange"] = {"transport": "peer memory over NVLink (CUDA IPC): pack kernels store into the neighbour GPU, seq flag release/acquire, "
                                         "substeps run inside the C-ABI" if args.exchange == "peer" else "torch.distributed NCCL point-to-point"}
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def soa_e2e(job, args):
    """N > 1: per-rank frames of field-wise upload + substeps + download through pinned host buffers (the AoS pool
    adapter is the single-process drop-in; z-slab ranks hold sparse subsets of the ids)."""
    import torch
    e = job.eng
    d = e.download(sort_by_id=False)
    n = len(d["id"])
    cap = n + n // 4 + 65536     # a rank's population changes during a frame (migration): room for the download
    host = {}
    for k, shape, dt_ in (("x", (cap, 3), torch.float32), ("v", (cap, 3), torch.float32), ("F", (cap, 9), torch.float32), ("b", (cap, 9), torch.float32),
                          ("mass", (cap,), torch.float32), ("vol", (cap,), torch.float32), ("ps", (cap,), torch.float32), ("group", (cap,), torch.int32)):
        t = torch.empty(shape, dtype=dt_, pin_memory=True)
        t.numpy()[:n] = d[k]
        host[k] = t
    host["id"] = torch.empty((cap,), dtype=torch.int32, pin_memory=True)
    times, alive = [], n
    # NB ids are renumbered by the field-wise upload (id_base + row); the frames below only time the path
    for f in range(args.frames + 1):
        job.barrier()
        t0 = time.perf_counter()
        e.upload_ptrs(n, host["x"].data_ptr(), host["v"].data_ptr(), host["F"].data_ptr(), host["b"].data_ptr(), host["mass"].data_ptr(),
                      host["vol"].data_ptr(), host["ps"].data_ptr(), host["group"].data_ptr())
        job.barrier()
        job.substep(args.frame_substeps)
        alive = e.download_ptrs(cap, host["id"].data_ptr(), host["x"].data_ptr(), host["v"].data_ptr(), host["F"].data_ptr(), host["b"].data_ptr(), 0, 0,
                                host["ps"].data_ptr(), 0)
        job.barrier()
        if f > 0:
            times.append(time.perf_counter() - t0)
    tmax = [job.allmax([t])[0] for t in times]
    tot = job.allsum([alive])[0]
    sec = float(np.median(tmax))
    h2d = job.allsum([n * 28 * 4])[0]
    d2h = job.allsum([n * 26 * 4])[0]
    return {"value": tot * args.frame_substeps / sec / 1e6, "unit": "M particle-updates/s", "h2d_bytes_per_step": h2d / args.frame_substeps,
            "d2h_bytes_per_step": d2h / args.frame_substeps, "frame_substeps": args.frame_substeps, "frames": args.frames, "frame_seconds": sec,
            "frame_seconds_all": tmax, "path": "per rank: mpmb_upload_particles -> substeps -> mpmb_download_particles (pinned field arrays)"}


_REAL_STDOUT = None


def _quiet_stdout():
    """Everything libraries print to fd 1 (e.g. the NCCL version banner) goes to stderr; the ONE JSON
    line is written to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    # OpenMP workers of the CPU arms: spin briefly between the (many, short) parallel regions, then
    # sleep.  Unbounded spinning collapsed oversubscribed teams on a shared box (200x), a purely passive
    # wait made the colour loops wake-up bound here (5x); measured with /tmp probes, see profiles/README.md
    os.environ.setdefault("GOMP_SPINCOUNT", "20000")
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sand256")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink grid and block together (debug only)")
    ap.add_argument("--frame-substeps", type=int, default=500, help="substeps per e2e frame (frame_dt/base_delta_t = 0.01/2e-5)")
    ap.add_argument("--frames", type=int, default=3, help="e2e frames; the median frame time is reported (host-side noise on shared boxes)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: strong = the SAME scene cut into N z-slabs (what the metric quotes), weak = block and grid extended along z")
    ap.add_argument("--also-weak", type=int, default=1, help="N > 1 strong runs also report the weak-scaling figure as `weak_scaling`")
    ap.add_argument("--develop", type=int, default=-1, help="substeps run before the `flowing` measurement (0 = quiescent only; "
                    "default 20000 for sand256 = 0.4 s of collapse, 2000 for the other workloads)")
    ap.add_argument("--no-parity-check", action="store_true", help="N > 1: skip the reduced-scene comparison with one engine")
    ap.add_argument("--cpu-sample", type=int, default=2_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--migrate-capacity", type=int, default=65536, help="particles per face per substep (z-slab message size)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="z-slab transport: NVLink peer memory (default) or NCCL send/recv")
    ap.add_argument("--halo-capacity", type=int, default=0, help="active tiles per boundary layer (z-slab message size); 0 = the whole cross-section")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the particle state after the last timed substep as DIR/<field>.npy "
                    "(a fixed seeded sample of %d particles, id order), for comparing two builds output for output" % OUTPUT_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        # the CPU arm times a particle sample sized by a speed probe: its outputs are not the same particles from run to run
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.develop < 0:
        args.develop = 20000 if args.workload == "sand256" else 2000
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
