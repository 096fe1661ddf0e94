#!/usr/bin/env python
"""bench.py — measurement-update throughput of the B200 engine (and, with --impl reference, of the
reference's own CPU path) on BASELINE.json's configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one measurement update (the hot path) over one batch: every particle x every sampled
scan point.  Prints ONE JSON line on rank 0 (see the contract in the task statement):
  value     whole-job particle x point evals/s with all inputs resident in HBM (CUDA events, max over ranks).
            N > 1: one process per GPU, particles sharded, map replicated; the ONE exchange of the path (the gather
            of the 24-byte records) is folded into the measurement kernels, which store every record into every
            rank's array over NVLink peer memory (csrc/kernels.cuh: RecordSink + exchange_signal_kernel).
            --exchange nccl keeps the NCCL all-gather for comparison.
            Timing (--l2 rotate, default): all K steps are ONE CUDA graph between one pair of events, step i on input
            set i mod 32 (32 places of the map with their own scan and particles: inputs larger than L2).  --l2 flush:
            a 256 MiB L2 flush before every step and an event pair around each (also always reported, in
            device_step.flushed_step_ms_min_med_max; an event pair + graph launch alone read ~6 us there).
  e2e       same metric through the host-array C-ABI call mcl3dl_measure (H2D + kernels + D2H inside; pose / record
            arrays page-locked via mcl3dl_host_alloc, scans in ordinary memory; L2 flushed before every call).
            N > 1: ONE host process (rank 0) drives all N GPUs through the in-process multi-device engine
            (mcl3dl_create with N device ids) and receives every record in one host array — what a ROS node would do.
  roofline  dominant kernel: algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the reference CPU path (oracle/_ref if present, else the port) on a bounded sample, 1 thread
  workloads driver-run secondaries: c3 (beam DDA), c3_kd (the node's default raycaster), c5 (65 536 spread particles,
            strong scaling at N > 1), each with value / kernel times / counted roofline
Workloads (BASELINE.json configs): c1 64x(96+3)/50k map, c2 1024x512 likelihood/1M map (default, the
metric's config), c3 4096x256 beam DDA/1M map, c4 16384x1024 lik+beam/10M map, c5 65536 spread lik+beam.
"""
import argparse
import functools
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from mcl_3dl_b200 import synth  # noqa: E402

WORKLOADS = {
    #        map pts   P      n_lik n_beam spread dda   scaling
    "c1": (50_000, 64, 96, 3, False, 0.2, "weak"),
    "c2": (1_000_000, 1024, 512, 0, False, 0.2, "weak"),
    "c3": (1_000_000, 4096, 0, 256, False, 0.2, "weak"),
    "c4": (10_000_000, 16384, 1024, 1024, False, 0.1, "strong"),
    "c5": (1_000_000, 65536, 64, 8, True, 0.2, "strong"),
    "c5e": (1_000_000, 8192, 64, 8, True, 0.2, "weak"),   # one GPU's share of c5 at 8 GPUs (kernel experiments)
}
FORCE_SPREAD = False
DIST_WEIGHT = (1.0, 1.0, 5.0)  # the node's default metric (src/parameters.cpp:108-111)
MAP_VOXEL = 0.1
USE_DDA = True
L2_MODE = "rotate"  # how consecutive timed steps are kept from reusing each other's L2 lines (--l2)
L2_TEXT = {
    "rotate": "inputs larger than L2: the timed steps run back to back (one CUDA graph, one event pair) on rotating input "
              "sets - 32 distinct places of the map with their own scan and particle cloud; spread workloads: fresh particle "
              "draws, every step alone reads more map than L2 holds.  device_step.flushed_step_ms_min_med_max is the same step "
              "under the flush-before-every-step protocol (per-step event pairs); e2e: L2 flushed before every call",
    "flush": "flushed (256 MiB write) before every timed step; N > 1: ranks re-aligned (untimed) after the flush",
}

# the synthetic map depends on (n_target, seed) only: c2 / c3 / c5 share one 1 M-point map
synth.warehouse_map = functools.lru_cache(maxsize=2)(synth.warehouse_map)


def bytes_per_eval_model(match_dist_min=0.2, w=DIST_WEIGHT, h=MAP_VOXEL):
    """SURVEY.md §8(d), exact mode: 16 B x cells of the h-lattice inside the search ellipsoid's box."""
    cells = 1
    for k in range(3):
        cells *= 2 * math.ceil(match_dist_min / (w[k] * h) - 1e-9) + 1
    return 16 * cells, cells


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "span": "warm-up, timed steps, ~0.5 s of the same step untimed, roofline and e2e loops (100 ms period)"}


def as_u8(a):
    return np.ascontiguousarray(a).view(np.uint8).reshape(-1)


def build_scene(workload, rank, world, all_ranks=False):
    """The rank's {map, scan, particle shard}.  all_ranks: the particles of every rank concatenated (rank 0's
    in-process multi-device e2e leg needs the whole job on one host)."""
    n_map, P, n_lik, n_beam, spread, dda, scaling = WORKLOADS[workload]
    spread = spread or FORCE_SPREAD
    P_rank = P if scaling == "weak" else P // world
    s = synth.scene(n_map, P, n_lik, n_beam, spread=spread, n_origins=2, seed=1000)

    def draw(r):
        # weak scaling: same map and scan, every rank its own particle draw
        if spread:
            return synth.spread_particles(P, s["info"], seed=2000 + r)
        return synth.tracking_particles(P, s["truth_pos"], s["truth_rpy"], seed=2000 + r)
    if scaling == "weak":
        s["particles"] = np.concatenate([draw(r) for r in range(world)]) if all_ranks else draw(rank)
    elif not all_ranks:
        s["particles"] = s["particles"][rank * P_rank:(rank + 1) * P_rank]
    else:
        s["particles"] = s["particles"][:P_rank * world]
    return s, dda, scaling, P_rank


def build_stations(workload, rank, world, s, n_stations):
    """Input sets for the back-to-back protocol (--l2 rotate): the same map, `n_stations` different places.

    Tracking workloads: every station is another place of the floor plan (a jittered grid, visited in a fixed random
    order) with its own scan and its own particle cloud, so that consecutive steps read different parts of the map's
    search structure and, over one round of the stations, far more of it than L2 holds.  Spread workloads read the whole
    map in every step (each step alone exceeds L2): the stations are fresh particle draws.  Station 0 is the scene."""
    n_map, P, n_lik, n_beam, spread, dda, scaling = WORKLOADS[workload]
    spread = spread or FORCE_SPREAD
    P_rank = P if scaling == "weak" else P // world
    info = s["info"]
    out = [{"particles": s["particles"], "lik": s["lik"], "beam": s["beam"]}]
    # station places: a jittered grid over the floor plan, at least 2 m from every box centre (boxes are box_size wide,
    # centred at (i + 0.5) * pitch), visited in a fixed random order so that consecutive steps are far apart
    L, pitch = info["L"], info["box_pitch"]
    side = int(math.ceil(math.sqrt(2 * n_stations)))
    grng = np.random.default_rng(4242)
    places = []
    for c in grng.permutation(side * side):
        x = 2.0 + (L - 4.0) * ((c // side) + grng.uniform(0.2, 0.8)) / side
        y = 2.0 + (L - 4.0) * ((c % side) + grng.uniform(0.2, 0.8)) / side
        bx, by = (math.floor(x / pitch) + 0.5) * pitch, (math.floor(y / pitch) + 0.5) * pitch
        if max(abs(x - bx), abs(y - by)) >= 2.0:
            places.append((x, y))
    for m in range(1, n_stations):
        if spread:
            parts = synth.spread_particles(P, info, seed=3000 + 17 * m)
            parts = parts if scaling == "weak" else parts[rank * P_rank:(rank + 1) * P_rank]
            out.append({"particles": parts, "lik": s["lik"], "beam": s["beam"]})
            continue
        rng = np.random.default_rng(5000 + m)
        pos = np.array([places[m % len(places)][0], places[m % len(places)][1], 0.6])
        rpy = np.array([0.0, 0.0, rng.uniform(-math.pi, math.pi)])
        q = synth.quat_from_rpy(rpy)[0]
        lik = synth.make_scan(s["map"], pos, q, n_lik, 0.5, 10.0, seed=6000 + m) if n_lik else s["lik"]
        beam = synth.make_scan(s["map"], pos, q, n_beam, 0.5, 4.0, n_origins=2, seed=7000 + m) if n_beam else s["beam"]
        # weak scaling: every rank its own draw around the station; strong (tracking): the rank's slice of one draw
        if scaling == "weak":
            parts = synth.tracking_particles(P, pos, rpy, seed=8000 + 64 * m + rank)
        else:
            parts = synth.tracking_particles(P, pos, rpy, seed=8000 + 64 * m)[rank * P_rank:(rank + 1) * P_rank]
        out.append({"particles": parts, "lik": lik, "beam": beam})
    return out


def host_threads():
    """Threads this process may really use (the lease's CPU set, not the machine's core count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def cpu_arm(workload, s, dda, n_lik, n_beam, target_s, threads, want_kind=None):
    """Time the reference CPU path on a bounded particle sample.  Returns (n_sample, s per pass, handle, meta)."""
    from oracle import cpu_checker as cc
    kind = "reference" if cc.available("reference") else "port"
    if want_kind:
        kind = want_kind
    if kind == "port":
        cc.build("port")
    chk = cc.CpuChecker(kind)
    t0 = time.perf_counter()
    cpu = chk.create(s["map"], cc.lik_params(dist_weight=DIST_WEIGHT),
                     cc.beam_raw(num_points_default=max(n_beam, 1), dda_grid_size=dda, use_raycast_using_dda=USE_DDA),
                     20.0, 0.4)
    build_s = time.perf_counter() - t0
    cpu.set_tally(False)
    per_particle = max(n_lik + n_beam, 1)
    probe = s["particles"][:max(threads, 4)]
    t0 = time.perf_counter()
    cpu.measure(probe, s["lik"], s["beam"], s["origins"], n_threads=threads)  # also builds the lazy DDA grid
    t0 = time.perf_counter()
    cpu.measure(probe, s["lik"], s["beam"], s["origins"], n_threads=threads)
    dt = max(time.perf_counter() - t0, 1e-6)
    rate = len(probe) * per_particle / dt
    n_sample = int(min(len(s["particles"]), max(len(probe), rate * target_s / per_particle)))
    sample = s["particles"][:n_sample]
    reps = int(max(1, min(200, round(target_s / max(n_sample * per_particle / rate, 1e-6)))))
    t0 = time.perf_counter()
    for _ in range(reps):
        cpu.measure(sample, s["lik"], s["beam"], s["origins"], n_threads=threads)
    dt = (time.perf_counter() - t0) / reps
    meta = {"kind": kind, "cores": threads, "index_build_s": round(build_s, 3), "seconds": round(dt * reps, 3),
            "sample": "%d of %d particles x (%d lik + %d beam) pts x %d repeats, same map/scan, %d thread(s)"
                      % (n_sample, len(s["particles"]), n_lik, n_beam, reps, threads)}
    return n_sample, dt, cpu, meta


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on the host threads this process may use
    (the cgroup / affinity set, not os.cpu_count()); the 1-thread figure — what the node really does, it is
    single-threaded by construction — is printed in the same line."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_map, P, n_lik, n_beam, spread, dda, scaling = WORKLOADS[args.workload]
    s, dda, scaling, P_rank = build_scene(args.workload, 0, 1)
    threads = host_threads()
    unit_pts = n_lik if n_lik else n_beam
    workload_particles = s["particles"]
    # give every thread enough particles to amortise its start-up: tile the particle set to >= 64 per thread
    need = threads * 64
    if len(s["particles"]) < need:
        s["particles"] = np.tile(s["particles"], (need + len(s["particles"]) - 1) // len(s["particles"]))
    n_sample, dt, cpu, meta = cpu_arm(args.workload, s, dda, n_lik, n_beam, 2.0, threads)
    sample = s["particles"][:n_sample]
    for _ in range(args.warmup):
        cpu.measure(sample, s["lik"], s["beam"], s["origins"], n_threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu.measure(sample, s["lik"], s["beam"], s["origins"], n_threads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        # the timed sample's size follows this host's speed; records are per particle, so the workload's own particle
        # set (untimed) gives the same records for every particle the timed step covered, at a size fixed by the workload
        dump_outputs(args.dump_outputs, cpu.measure(workload_particles, s["lik"], s["beam"], s["origins"], n_threads=threads))
    value = n_sample * unit_pts * args.steps / dt
    meta["value"] = value
    meta["unit"] = "evals/s"
    # the node's real path: one thread (serial loop pf.h:256, ros::spin mcl_3dl.cpp:1466), ~2 s sample
    n1 = max(4, min(n_sample, int(n_sample / max(threads, 1)) + 1))
    one = s["particles"][:n1]
    cpu.measure(one, s["lik"], s["beam"], s["origins"], n_threads=1)
    reps = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < 2.0:
        cpu.measure(one, s["lik"], s["beam"], s["origins"], n_threads=1)
        reps += 1
    meta["value_1_thread"] = n1 * unit_pts * reps / (time.perf_counter() - t0)
    meta["cores_machine"] = os.cpu_count()
    line = {"impl": "reference", "metric": metric_name(n_lik), "value": value, "unit": "evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.workload, s, P * args.gpus if scaling == "weak" else P, n_lik, n_beam, spread, dda),
            "cpu_baseline": meta,
            "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def dump_outputs(out_dir, recs):
    """--dump-outputs: every field of the last timed step's records as DIR/<field>.npy (float32 scores, float64
    counts), so that two builds can be compared output for output on the same seeded inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for f in recs.dtype.names:
        np.save(os.path.join(out_dir, f + ".npy"), recs[f].astype(np.float32 if recs[f].dtype.kind == "f" else np.float64))


def metric_name(n_lik):
    return "particle x point likelihood evals/s" if n_lik else "particle x ray beam-model evals/s"


def config_dict(workload, s, P, n_lik, n_beam, spread, dda):
    """Identical keys on both arms (the engine-side map figures live in the line's `map` object)."""
    return {"workload": "%s: %d particles x (%d likelihood pts + %d beam rays), %d-pt map @%.1f m voxel, %s particles"
                        % (workload, P, n_lik, n_beam, len(s["map"]), MAP_VOXEL, "spread" if spread else "tracking"),
            "dist_weight": list(DIST_WEIGHT), "dda_grid_size": dda, "match_dist_min": 0.2,
            "raycaster": "RaycastUsingDDA" if USE_DDA else "RaycastUsingKDTree",
            "l2": L2_TEXT[L2_MODE]}


class Ctx:
    """Process-wide state of the b200 arm (torch, distributed ranks, flush buffer)."""
    pass


def device_leg(cx, workload, raycaster, steps, warmup, exchange="peer", graph=True, keep_spinning=False, field=False,
               keep_records=False):
    """Device-resident leg of one workload on every rank: value (CUDA events, max over ranks), per-model kernel
    times, counted roofline.  Returns (result dict, live objects for the e2e leg).  keep_records: live["last_records"]
    holds the records of the last timed step of the headline protocol, as the caller of measure_device receives them."""
    import torch
    import torch.distributed as dist
    from mcl_3dl_b200 import engine, sharding
    global USE_DDA
    USE_DDA = raycaster == "dda"
    world, rank, dev = cx.world, cx.rank, cx.dev
    n_map, P, n_lik, n_beam, spread, _, _ = WORKLOADS[workload]
    spread = spread or FORCE_SPREAD
    s, dda, scaling, P_rank = build_scene(workload, rank, world)
    eng = engine.Engine((cx.local,))  # no fallback: raises without the CUDA library / device
    lik = engine.LikParams(dist_weight=DIST_WEIGHT)
    beam = engine.beam_params_from_reference(num_points_default=max(n_beam, 1), dda_grid_size=dda,
                                             use_raycast_using_dda=USE_DDA)
    eng.set_map(s["map"], lik if (n_lik or not USE_DDA) else None, beam if n_beam else None)
    info = eng.map_info()
    particles = s["particles"]
    n_org = len(s["origins"])
    d_p = torch.from_numpy(as_u8(particles)).to(dev)
    d_l = torch.from_numpy(as_u8(s["lik"])).to(dev) if n_lik else torch.zeros(16, dtype=torch.uint8, device=dev)
    d_b = torch.from_numpy(as_u8(s["beam"])).to(dev) if n_beam else torch.zeros(16, dtype=torch.uint8, device=dev)
    d_o = torch.from_numpy(np.ascontiguousarray(s["origins"], dtype=np.float32)).to(dev)
    d_out = torch.zeros(P_rank * 24, dtype=torch.uint8, device=dev)
    d_all = torch.zeros(world * P_rank * 24, dtype=torch.uint8, device=dev) if world > 1 else None
    flush = cx.flush

    peer = world > 1 and exchange == "peer"
    if peer:
        # the CUDA IPC handles of the exchange buffers are the only thing that goes through torch.distributed
        handle = eng.exchange_create(P_rank, world, rank)
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=dev)
        gathered = torch.empty(world * len(handle), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(gathered, mine)
        eng.exchange_open(bytes(gathered.cpu().numpy().tobytes()))
        dist.barrier()

    def plain_measure(st):
        eng.measure_device(d_p.data_ptr(), P_rank, d_l.data_ptr(), n_lik, d_b.data_ptr(), n_beam,
                           d_o.data_ptr(), n_org, d_out.data_ptr(), st)

    field_info = None
    if field:
        # the opt-in, inexact field mode (dense distance volume + trilinear lookup, north_star's literal kernel): its
        # records against the exact ones of the same engine (which are oracle-checked), then everything below runs in it
        st0 = torch.cuda.current_stream().cuda_stream
        plain_measure(st0)
        torch.cuda.synchronize()
        exact = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=synth.RESULT).copy()
        t0 = time.perf_counter()
        eng.field_mode(True)
        stage_s = time.perf_counter() - t0
        plain_measure(st0)
        torch.cuda.synchronize()
        got = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=synth.RESULT).copy()
        rel = np.abs(got["score_like"] - exact["score_like"]) / np.maximum(np.abs(exact["score_like"]), 1e-3)
        nodes, _, edge, dims = eng.field_nodes(download=False)
        field_info = {"score_like_rel_err_vs_exact": {"mean": float(rel.mean()), "p99": float(np.quantile(rel, 0.99)),
                                                      "max": float(rel.max())},
                      "match_cnt_mismatch_fraction": float(np.mean(got["match_cnt"] != exact["match_cnt"])),
                      "match_cnt_mean_abs_diff": float(np.mean(np.abs(got["match_cnt"].astype(np.int64)
                                                                      - exact["match_cnt"].astype(np.int64)))),
                      "lattice_nodes": list(dims), "lattice_edge": edge,
                      "volume_bytes": int((dims[0] - 1) * (dims[1] - 1) * (dims[2] - 1) * 32),
                      "stage_ms": round(1e3 * stage_s, 2),
                      "note": "exact = this engine's NN-field search (oracle-checked by the -m gpu tests); the field mode "
                              "is reported, not gated: interpolating a distance field at this lattice cannot meet 1e-4"}

    def step_eager():
        st = torch.cuda.current_stream().cuda_stream
        if peer:
            # both models + the record exchange: the kernels store into every rank's array, one signal kernel follows
            eng.measure_exchange_device(d_p.data_ptr(), P_rank, d_l.data_ptr(), n_lik, d_b.data_ptr(), n_beam,
                                        d_o.data_ptr(), n_org, st)
        else:
            plain_measure(st)
            if world > 1:
                sharding.gather_records_device(d_out, d_all)  # comparison arm: NCCL all-gather of the records

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    l0 = eng.kernel_launches()
    for _ in range(3):
        step_eager()
    barrier()
    launches_per_step = (eng.kernel_launches() - l0) // 3
    step, graphed = step_eager, False
    if graph:
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                step_eager()
            step, graphed = g.replay, True
        except Exception as exc:  # keep measuring eagerly, and say so
            cx.notes.append("CUDA graph capture failed for %s: %s" % (workload, exc))
            barrier()

    align = torch.zeros(1, device=dev)

    def timed(fn, k):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        barrier()
        for a, b in evs:
            flush.fill_(1)          # L2 flush, outside the timed span
            if world > 1:
                # the 256 MiB flush does not take the same time on every rank: line the ranks up again (a tiny NCCL
                # all-reduce on the stream, untimed) so that a timed step does not include waiting for a peer's flush
                dist.all_reduce(align)
            a.record()
            fn()
            b.record()
        barrier()
        per = [a.elapsed_time(b) for a, b in evs]
        t = torch.tensor([sum(per)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), per

    def records():
        """The records the step left on the device: this rank's array, or every rank's after the exchange."""
        buf = d_all if world > 1 else d_out
        if peer:
            ptr, _ = eng.exchange_current(torch.cuda.current_stream().cuda_stream)
            cai = {"shape": (world * P_rank * 24,), "typestr": "|u1", "data": (ptr, False), "version": 3}
            buf = torch.as_tensor(type("DeviceBytes", (), {"__cuda_array_interface__": cai})(), device=dev)
        torch.cuda.synchronize()
        return np.frombuffer(buf.cpu().numpy().tobytes(), dtype=synth.RESULT).copy()

    for _ in range(warmup):
        step()
    barrier()
    total_ms, per_step = timed(step, steps)
    last_records = records() if keep_records else None
    if keep_spinning:
        # the timed region lasts a few milliseconds, shorter than one nvidia-smi period: keep the same step running
        # (untimed, same count on every rank) for ~0.5 s so that the clock record holds samples taken under this load
        for _ in range(int(min(20000, max(0, 500.0 / max(total_ms / steps, 1e-3))))):
            step()
        barrier()

    # ---- the back-to-back protocol: ALL `steps` steps in one CUDA graph, one event pair around the replay, consecutive
    # steps on different input sets ("inputs larger than L2" instead of a flush before every step).  A pair of events
    # around one launch costs ~5 us on this system and a graph launch ~3 us (profiles/r02z_cold.txt): per-step event
    # pairs add that to every step, which is most of a 20 us step and none of the kernel's work.
    b2b = None
    if graph and graphed:
        n_st = 4 if spread else 32
        stations = build_stations(workload, rank, world, s, n_st)
        dst = []
        for stn in stations:
            dst.append((torch.from_numpy(as_u8(stn["particles"])).to(dev),
                        torch.from_numpy(as_u8(stn["lik"])).to(dev) if n_lik else d_l,
                        torch.from_numpy(as_u8(stn["beam"])).to(dev) if n_beam else d_b))

        def step_on(i):
            sp, sl, sb = dst[i % len(dst)]
            st = torch.cuda.current_stream().cuda_stream
            if peer:
                eng.measure_exchange_device(sp.data_ptr(), P_rank, sl.data_ptr(), n_lik, sb.data_ptr(), n_beam,
                                            d_o.data_ptr(), n_org, st)
            else:
                eng.measure_device(sp.data_ptr(), P_rank, sl.data_ptr(), n_lik, sb.data_ptr(), n_beam,
                                   d_o.data_ptr(), n_org, d_out.data_ptr(), st)
                if world > 1:
                    sharding.gather_records_device(d_out, d_all)

        def capture(pick):
            for i in range(min(3, steps)):
                step_on(pick(i))
            barrier()
            gk = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gk):
                for i in range(steps):
                    step_on(pick(i))
            return gk

        def replay_ms(gk):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            if world > 1:
                dist.all_reduce(align)  # ranks leave the barrier together (untimed)
            a.record()
            gk.replay()
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        try:
            g_rot = capture(lambda i: i)
            for _ in range(max(1, -(-warmup // max(steps, 1)))):  # >= `warmup` untimed steps
                g_rot.replay()
            barrier()
            official = replay_ms(g_rot)                       # the timed region: exactly `steps` steps
            if keep_records and L2_MODE == "rotate":
                last_records = records()
            repeats = [replay_ms(g_rot) for _ in range(4)]
            g_same = capture(lambda i: 0)                     # comparison: every step on the same inputs (L2-warm)
            g_same.replay()
            same = sorted(replay_ms(g_same) for _ in range(3))[1]
            b2b = {"ms_total": official, "ms_per_step": official / steps, "stations": len(dst),
                   "repeats_ms_per_step": [r / steps for r in repeats],
                   "same_station_every_step_ms_per_step": same / steps,
                   "flushed_with_per_step_events_ms_per_step": total_ms / steps,
                   "note": "one CUDA graph of all timed steps, one event pair around its replay, max over ranks; step i "
                           "runs on station i mod %d (%s); the same graph on ONE station (L2-warm) and the per-step-flush "
                           "protocol are listed beside it" % (
                               len(dst), "fresh spread particle draws: every step alone reads more map than L2 holds"
                               if spread else "distinct places of the floor plan, own scan and particle cloud each")}
            del g_same
        except Exception as exc:
            cx.notes.append("back-to-back protocol failed for %s: %s" % (workload, exc))
            barrier()

    exchange_info = None
    if world > 1:
        exchange_info = {"mode": "peer-memory stores in the kernels' epilogues + signal kernel" if peer else "nccl all_gather",
                         "graph": graphed, "bytes_per_rank_per_step": P_rank * 24 * (world if peer else 1)}
        if peer:
            # the folded exchange against NCCL on the same inputs (outside every timed region), byte for byte
            class _DevView:  # raw device memory as a torch tensor (CUDA array interface)
                def __init__(self, ptr, nbytes):
                    self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
            st = torch.cuda.current_stream().cuda_stream
            plain_measure(st)
            sharding.gather_records_device(d_out, d_all)
            ptr, failed = eng.exchange_current(st)
            t_peer = torch.as_tensor(_DevView(ptr, world * P_rank * 24), device=dev)
            ok = torch.tensor([int(torch.equal(t_peer, d_all))], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            exchange_info["matches_nccl_on_every_rank"] = bool(ok.item())
            exchange_info["peer_wait_timed_out"] = failed

    unit_pts = n_lik if n_lik else n_beam
    evals_step = world * P_rank * unit_pts
    ms_per_step = total_ms / steps
    l2_used = "flush"
    if b2b and L2_MODE == "rotate":
        ms_per_step, l2_used = b2b["ms_per_step"], "rotate"
    elif L2_MODE == "rotate":
        cx.notes.append("%s: no CUDA graph of the timed steps - value is from the flush-before-every-step protocol" % workload)
    res = {"value": evals_step / (ms_per_step * 1e-3), "ms_per_step": ms_per_step, "scaling": scaling,
           "graph": graphed, "launches_per_step": int(launches_per_step), "l2": l2_used,
           "flushed_step_ms_min_med_max": [float(np.min(per_step)), float(np.median(per_step)), float(np.max(per_step))],
           "back_to_back": b2b, "exchange": exchange_info}
    if field_info:
        res["field_mode"] = field_info

    # ---- each model's kernel alone (one launch per call): the dominant kernel's roofline
    stream = torch.cuda.current_stream().cuda_stream
    kern = {}
    if n_lik:
        def lik_only():
            eng.measure_device(d_p.data_ptr(), P_rank, d_l.data_ptr(), n_lik, 0, 0, 0, 0, d_out.data_ptr(), stream)
        kern["lik"] = timed(lik_only, steps)[0] / steps
    if n_beam:
        def beam_only():
            eng.measure_device(d_p.data_ptr(), P_rank, 0, 0, d_b.data_ptr(), n_beam, d_o.data_ptr(), n_org,
                               d_out.data_ptr(), stream)
        kern["beam"] = timed(beam_only, steps)[0] / steps
    kern_src = "flush before every launch, CUDA event pair around each (includes ~5 us of event-pair cost)"
    if l2_used == "rotate" and len(kern) == 1:
        # one kernel per step: the step time of the headline protocol IS the kernel's average launch duration
        kern = {next(iter(kern)): ms_per_step}
        kern_src = "the timed region itself: back-to-back launches on rotating inputs, total / steps"
    peak, peak_src = peaks()
    dom = max(kern, key=kern.get)
    # exact work counters of one (untimed) step: what this layout's algorithm must read, no reuse assumed
    eng.collect_stats(True)
    plain_measure(stream)
    ws = eng.read_stats()
    eng.collect_stats(False)
    io_bytes = P_rank * 32 + P_rank * 24
    bpe, cells = bytes_per_eval_model()
    near = eng.near_field_info()  # [(k, bytes)] likelihood / KD-caster screens; k = 0: not staged
    if dom == "lik":
        alg_bytes = ws["lik_index_rows"] * 8 + ws["lik_points_scanned"] * 16 + io_bytes + n_lik * 16
        note = ("counted: %.1f index entries x 8 B + %.1f map points x 16 B per eval (+ poses/scan/records)"
                % (ws["lik_index_rows"] / max(P_rank * n_lik, 1), ws["lik_points_scanned"] / max(P_rank * n_lik, 1)))
        nnf = eng.nn_field_info()
        if nnf["bytes"]:
            note += "; NN field %.0f MB, %.1f M candidates, %d wide / %d overflow cells" % (
                nnf["bytes"] / 1e6, nnf["candidates"] / 1e6, nnf["wide_cells"], nnf["overflow_cells"])
        elif near[0][0]:
            alg_bytes += P_rank * n_lik * 4
            note += " + one 4 B near-field word per eval (k=%d, %.0f MB)" % (near[0][0], near[0][1] / 1e6)
        survey_bytes = P_rank * n_lik * bpe + io_bytes + n_lik * 16
        survey_note = "SURVEY 8d exact mode, dense float4 voxel grid: %d B/eval = 16 B x %d cells" % (bpe, cells)
    else:
        alg_bytes = (ws["beam_cells_stepped"] * 4 + ws["beam_cells_occupied"] * 8 + ws["beam_points_tested"] * 16
                     + io_bytes + n_beam * 16)
        note = ("counted: %.1f cells stepped x 4 B occupancy word + %.2f occupied x 8 B CSR + %.2f pts x 16 B per ray"
                % (ws["beam_cells_stepped"] / max(P_rank * n_beam, 1), ws["beam_cells_occupied"] / max(P_rank * n_beam, 1),
                   ws["beam_points_tested"] / max(P_rank * n_beam, 1)))
        survey_bytes = (ws["beam_cells_stepped"] * 1 + ws["beam_cells_occupied"] * 8 + ws["beam_points_tested"] * 16
                        + io_bytes + n_beam * 16)
        survey_note = "SURVEY 8d beam: 1 B per cell stepped + 8 B CSR + 16 B per point tested"
    achieved = alg_bytes / (kern[dom] * 1e-3) / 1e9
    traffic, traffic_src, binding = None, None, None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            ncu = json.load(f)
        key = (workload + ("" if raycaster == "dda" or not n_beam else "_kd") + ("_spread" if FORCE_SPREAD else "")
               + ("_field" if field else ""))
        ent = ncu.get(key, {})
        traffic = ent.get(dom + "_dram_bytes_per_launch")
        traffic_src = ent.get(dom + "_source")
        binding = ent.get(dom + "_binding_resource")
    except Exception:
        pass
    res["roofline"] = {"bound": "hbm", "kernel": dom + "_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                       "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                       "binding_resource_ncu": binding,
                       "dram_frac": (traffic / (kern[dom] * 1e-3) / 1e9 / peak) if traffic else None,
                       "kernel_ms": kern[dom], "kernel_ms_source": kern_src, "algorithmic_bytes_per_launch": alg_bytes,
                       "model": note,
                       "kernel_ms_all": kern, "work_counters_per_step": ws,
                       "survey_8d_model": {"bytes_per_launch": survey_bytes,
                                           "achieved": survey_bytes / (kern[dom] * 1e-3) / 1e9,
                                           "frac": survey_bytes / (kern[dom] * 1e-3) / 1e9 / peak, "note": survey_note}}
    res["map"] = {"nn_grid": list(info.nn_dims), "dda_grid": list(info.dda_dims), "device_bytes": int(info.device_bytes),
                  "build_ms": round(info.build_ms, 3)}
    live = {"eng": eng, "scene": s, "dda": dda, "P_rank": P_rank, "d_out": d_out, "plain_measure": plain_measure,
            "n_lik": n_lik, "n_beam": n_beam, "spread": spread, "P": P, "scaling": scaling, "unit_pts": unit_pts,
            "last_records": last_records}
    return res, live


def _e2e_rank0(cx, workload, raycaster, steps, live, fused, pinned):
    """Rank 0's part of e2e_leg.  pinned: the caller's pose / record arrays come from mcl3dl_host_alloc."""
    import torch
    from mcl_3dl_b200 import engine
    world, rank, dev = cx.world, cx.rank, cx.dev
    n_lik, n_beam, unit_pts = live["n_lik"], live["n_beam"], live["unit_pts"]
    if world == 1:
        eng, s = live["eng"], live["scene"]
    else:
        s, dda, _, _ = build_scene(workload, 0, world, all_ranks=True)
        eng = engine.Engine(tuple(range(world)))
        lik = engine.LikParams(dist_weight=DIST_WEIGHT)
        beam = engine.beam_params_from_reference(num_points_default=max(n_beam, 1), dda_grid_size=dda,
                                                 use_raycast_using_dda=(raycaster == "dda"))
        eng.set_map(s["map"], lik if (n_lik or raycaster != "dda") else None, beam if n_beam else None)
    particles = s["particles"]
    n_total = len(particles)
    # the buffer addresses are resolved once (Engine.bind_measure), as a C++ caller's would be: every timed call is
    # exactly one mcl3dl_measure(host pointers) = staging + H2D + kernels + D2H + synchronise
    # the caller's pose and record arrays live in page-locked memory (mcl3dl_host_alloc), as the adapter's do: they
    # are transferred in place; the scans and origins are ordinary memory and go through the engine's staging block
    if pinned:
        h_poses = eng.host_array(n_total, synth.POSE)
        h_poses[...] = np.ascontiguousarray(particles, dtype=synth.POSE)
        out_host = eng.host_array(n_total, synth.RESULT)
    else:
        h_poses = np.ascontiguousarray(particles, dtype=synth.POSE)
        out_host = np.zeros(n_total, dtype=synth.RESULT)
    h_in = [h_poses] + [np.ascontiguousarray(a, dtype=dt) for a, dt in ((s["lik"], synth.POINT), (s["beam"], synth.POINT))]
    h_org = np.ascontiguousarray(s["origins"], dtype=np.float32).reshape(-1, 3)
    call = eng.bind_measure(h_in[0], h_in[1], h_in[2], h_org, out_host)
    flushes = [cx.flush] + [torch.empty(256 << 20, dtype=torch.uint8, device=torch.device("cuda", d))
                            for d in range(world) if d != cx.local]

    def flush_all():
        for f in flushes:
            f.fill_(1)
        for d in range(world if world > 1 else 1):
            torch.cuda.synchronize(d if world > 1 else dev)
    for _ in range(3):
        call()
    tot = 0.0
    for _ in range(steps):
        flush_all()
        t0 = time.perf_counter()
        call()
        tot += time.perf_counter() - t0
    eng.collect_timing(True)   # device-side breakdown of one extra, untimed call (the events cost ~28 us per call,
    call()                     # so they are off while the loop above is timed)
    last = eng.last_timing()
    eng.collect_timing(False)
    evals = n_total * unit_pts
    n_org = len(s["origins"])
    out = {"value": evals * steps / tot, "unit": "evals/s", "ms_per_step": 1e3 * tot / steps,
           "h2d_bytes_per_step": n_total * 32 + world * (n_lik * 16 + n_beam * 16 + n_org * 16),
           "d2h_bytes_per_step": n_total * 24,
           "timing": "host wall clock around the synchronous call, L2 of every device flushed before it",
           "host_buffers": ("poses and records in page-locked memory from mcl3dl_host_alloc (transferred in place); scans "
                            "and origins in ordinary memory (staged)" if pinned else
                            "ordinary memory: everything goes through the engine's page-locked staging block"),
           "last_call_device_ms": last,
           "path": ("mcl3dl_measure on this process' one-device engine" if world == 1 else
                    "mcl3dl_measure on ONE in-process engine over %d devices (rank 0; one host thread, every record "
                    "lands in one host array — the gather is the D2H of each shard)" % world),
           "d2h_mode": ("kernels store the records straight into the caller's page-locked array" if n_total // world <= 8192
                        else "one D2H copy of the records per device")}
    if fused:
        # the fused weight update (scope row f2): priors up, posteriors (4 B/particle) back
        prior = np.full(n_total, 1.0 / max(n_total, 1), dtype=np.float32)
        for _ in range(3):
            eng.measure_update(particles, s["lik"], s["beam"], s["origins"], prior)
        ftot = 0.0
        for _ in range(steps):
            flush_all()
            t0 = time.perf_counter()
            post, summ, _ = eng.measure_update(particles, s["lik"], s["beam"], s["origins"], prior)
            ftot += time.perf_counter() - t0
        out["fused_weight_update"] = {"value": evals * steps / ftot, "unit": "evals/s", "ms_per_step": 1e3 * ftot / steps,
                                      "h2d_bytes_per_step": out["h2d_bytes_per_step"] + n_total * 4,
                                      "d2h_bytes_per_step": n_total * 4, "entropy": summ["entropy"], "kept": summ["kept"]}
    out_host = out_host.copy()  # (the page-locked block goes away with the engine)
    live["out_host"] = out_host
    if world > 1:
        # the in-process N-device engine against this rank's own device-resident shard (first shard of the job)
        live["plain_measure"](torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = np.frombuffer(live["d_out"].cpu().numpy().tobytes(), dtype=synth.RESULT)
        out["shard0_equals_device_resident"] = bool(np.array_equal(got, out_host[:live["P_rank"]]))
        eng.close()
    return out


def e2e_leg(cx, workload, raycaster, steps, live, fused=True):
    """End to end through the host-buffer C-ABI call (pinned staging + H2D + kernels + D2H + synchronise inside).
    N == 1: this process' engine.  N > 1: rank 0 alone drives ALL N GPUs through the in-process multi-device engine and
    receives every record in one host array; the other ranks wait at the barrier."""
    import torch
    import torch.distributed as dist
    from mcl_3dl_b200 import engine
    world, rank, dev = cx.world, cx.rank, cx.dev
    n_lik, n_beam, unit_pts = live["n_lik"], live["n_beam"], live["unit_pts"]
    out = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=cx.cpu_group)  # gloo: the waiting ranks leave their GPUs idle
    if rank == 0:
        # pose / record arrays page-locked through mcl3dl_host_alloc; should that path fail on this box, the same call on
        # ordinary arrays (the engine's own staging block) is measured instead and the line says so
        try:
            out = _e2e_rank0(cx, workload, raycaster, steps, live, fused, True)
        except Exception as exc:
            cx.notes.append("%s e2e with page-locked caller arrays failed (%s: %s); ordinary arrays measured instead"
                            % (workload, type(exc).__name__, exc))
            out = _e2e_rank0(cx, workload, raycaster, steps, live, fused, False)
    if world > 1:
        dist.barrier(group=cx.cpu_group)
    return out


def resident_leg(cx, workload, steps):
    """Scope row f3: whole localisation cycles on the engine's RESIDENT particle set (N = 1).  Every cycle = predict
    (odometry step) + measurement update of both models with the weight update + pose estimate (biased mean, max,
    covariance) + resampling, all on the device: only the scans and an odometry pair go in, only summaries come out.
    Host wall clock around the four C-ABI calls, L2 flushed before every cycle."""
    import torch
    from mcl_3dl_b200 import engine
    global USE_DDA
    USE_DDA = True
    n_map, P, n_lik, n_beam, spread, dda, _ = WORKLOADS[workload]
    s, dda, _, _ = build_scene(workload, 0, 1)
    eng = engine.Engine((cx.local,))
    eng.set_map(s["map"], engine.LikParams(dist_weight=DIST_WEIGHT),
                engine.beam_params_from_reference(num_points_default=max(n_beam, 1), dda_grid_size=dda))
    st = np.zeros(P, dtype=synth.STATE)
    st["pos"] = np.stack([s["particles"]["px"], s["particles"]["py"], s["particles"]["pz"]], axis=1)
    st["rot"] = np.stack([s["particles"][k] for k in ("qx", "qy", "qz", "qw")], axis=1)
    eng.particles_set(st, np.full(P, 1.0 / P, np.float32))
    a = synth.make_poses([[0, 0, 0]], [[0, 0, 0, 1]])
    b = synth.make_poses([[0.02, 0, 0]], synth.quat_from_rpy([[0, 0, 0.01]]))
    sp, sr = np.array([0.05, 0.05, 0.01], np.float32), np.array([0.005, 0.005, 0.02], np.float32)
    parts = {"predict": 0.0, "measure_update": 0.0, "estimate": 0.0, "resample": 0.0}

    def cycle(k, timed):
        t0 = time.perf_counter()
        eng.particles_predict(a, b, 0.1, 10.0, 10.0)
        t1 = time.perf_counter()
        summ = eng.particles_measure_update(s["lik"], s["beam"], s["origins"], 0.05)
        t2 = time.perf_counter()
        est = eng.particles_estimate(None)
        t3 = time.perf_counter()
        eng.particles_resample(sp, sr, 0.5, seed=1000 + k)
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        if timed:
            for name, dt in zip(parts, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                parts[name] += dt
        return summ, est, t4 - t0
    for k in range(3):
        cycle(k, False)
    tot = 0.0
    for k in range(steps):
        cx.flush.fill_(1)
        torch.cuda.synchronize()
        summ, est, dt = cycle(10 + k, True)
        tot += dt
    eng.close()
    n_org = len(s["origins"])
    return {"metric": metric_name(n_lik), "value": P * n_lik * steps / tot, "unit": "evals/s", "ms_per_cycle": 1e3 * tot / steps,
            "ms_per_call": {k: 1e3 * v / steps for k, v in parts.items()}, "steps": steps,
            "h2d_bytes_per_cycle": n_lik * 16 + n_beam * 16 + n_org * 12 + 64, "d2h_bytes_per_cycle": 24 + 256 + 68,
            "cycle": "mcl3dl_particles_predict + _measure_update (both models, odometry-error term, normalise, entropy) + "
                     "_estimate (biased mean, max, 6x6 covariance) + _resample, %d particles resident on the device" % P,
            "last_summary": {"entropy": summ["entropy"], "kept": summ["kept"], "mean_xy": [float(est["mean_biased"]["px"][0]),
                                                                                           float(est["mean_biased"]["py"][0])]},
            "config": config_dict(workload, s, P, n_lik, n_beam, spread, dda)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline sample budget")
    ap.add_argument("--exchange", default="peer", choices=["nccl", "peer"],
                    help="N > 1: how the records are gathered: stores into peer memory from the kernels' epilogues "
                         "(default, the product) or an NCCL all-gather after the kernels (comparison)")
    ap.add_argument("--l2", default="rotate", choices=["rotate", "flush"],
                    help="device-resident leg: how consecutive timed steps are kept from reusing each other's L2 lines: "
                         "back to back on rotating input sets larger than L2 (default), or a 256 MiB flush before every "
                         "step with a CUDA event pair around each step")
    ap.add_argument("--no-graph", action="store_true", help="launch the device-resident step eagerly instead of as one CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondaries", action="store_true", help="only the primary workload (profiling runs)")
    ap.add_argument("--raycaster", default="dda", choices=["dda", "kd"],
                    help="beam raycaster: RaycastUsingDDA (north_star) or RaycastUsingKDTree (the node's default)")
    ap.add_argument("--spread", action="store_true", help="spread (global-localisation style) particles: the HBM-bound variant")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the records of the last timed step (one .npy per field, seeded inputs) into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    global FORCE_SPREAD, USE_DDA, L2_MODE
    L2_MODE = "flush" if args.no_graph else args.l2
    FORCE_SPREAD = args.spread
    USE_DDA = args.raycaster == "dda"
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    cx = Ctx()
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.rank = int(os.environ.get("RANK", "0"))
    cx.local = int(os.environ.get("LOCAL_RANK", "0"))
    cx.notes = []
    if cx.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the launcher set it (the driver reads the communicator's rank count from NCCL's own log)
        dist.init_process_group("nccl", device_id=torch.device("cuda", cx.local))
        # host-side waits (a rank that idles while rank 0 drives every GPU must not park an NCCL kernel on its device)
        cx.cpu_group = dist.new_group(backend="gloo")
    torch.cuda.set_device(cx.local)
    cx.dev = torch.device("cuda", cx.local)
    cx.flush = torch.empty(256 << 20, dtype=torch.uint8, device=cx.dev)
    world, rank = cx.world, cx.rank

    # clocks are sampled from the warm-up to the end of the e2e loop: the timed region alone lasts a few
    # milliseconds, shorter than one nvidia-smi sampling period
    clocks = ClockSampler(cx.local)
    if rank == 0:
        clocks.start()
    graph = not args.no_graph
    res, live = device_leg(cx, args.workload, args.raycaster, args.steps, args.warmup, args.exchange, graph, keep_spinning=True,
                           keep_records=bool(args.dump_outputs))
    e2e = e2e_leg(cx, args.workload, args.raycaster, args.steps, live)
    clk = clocks.stop() if rank == 0 else None
    n_lik, n_beam, P_rank, s = live["n_lik"], live["n_beam"], live["P_rank"], live["scene"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, live["last_records"])

    # ---- sanity: device-resident records == host-path records (N == 1; at N > 1 the e2e leg checked shard 0)
    if rank == 0 and world == 1 and n_lik and n_beam:
        live["plain_measure"](torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = np.frombuffer(live["d_out"].cpu().numpy().tobytes(), dtype=synth.RESULT)
        assert np.array_equal(got, live["out_host"]), "device-resident and host entry points disagree"

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            USE_DDA = args.raycaster == "dda"
            out_host = live["out_host"]
            n_sample, dt, cpu, meta = cpu_arm(args.workload, s, live["dda"], n_lik, n_beam, args.cpu_seconds, 1)
            meta["value"] = n_sample * live["unit_pts"] / dt
            meta["unit"] = "evals/s"
            # parity spot check of this very workload against the checker (first particles of rank 0)
            cpu.set_tally(True)
            chk = cpu.measure(s["particles"][:16], s["lik"], s["beam"], s["origins"])
            ok = all(np.array_equal(chk[f], out_host[:16][f]) for f in ("match_cnt", "n_short", "n_hit", "n_long"))
            ok = ok and np.allclose(chk["score_like"], out_host[:16]["score_like"], rtol=1e-4, atol=1e-6)
            meta["parity_spot_check"] = bool(ok)
            cpu_baseline = meta
        except Exception as exc:  # the GPU line must still be printed if the checker cannot be built / loaded
            cpu_baseline = {"error": "%s: %s" % (type(exc).__name__, exc)}
    live["eng"].close()
    out_host = live.get("out_host")
    del live

    # ---- driver-run secondaries (no CPU leg): what north_star names besides the primary metric
    secondaries = {}
    if not args.no_secondaries and args.workload == "c2" and not args.spread:
        sec = ([("c5", "c5", "dda")] if world > 1 else
               [("c3", "c3", "dda"), ("c3_kd", "c3", "kd"), ("c5", "c5", "dda"), ("c5_field", "c5", "dda")])
        k = args.steps
        for name, wl, caster in sec:
            try:
                r2, live2 = device_leg(cx, wl, caster, k, 3, args.exchange, graph, field=name.endswith("_field"))
                r2["metric"] = metric_name(live2["n_lik"])
                r2["unit"] = "evals/s"
                r2["steps"] = k
                r2["config"] = config_dict(wl, live2["scene"], live2["P"] if live2["scaling"] == "strong" else live2["P_rank"] * world,
                                           live2["n_lik"], live2["n_beam"], live2["spread"], live2["dda"])
                e2 = e2e_leg(cx, wl, caster, k, live2, fused=False)
                if e2 is not None:
                    r2["e2e"] = e2
                live2["eng"].close()
                del live2
                secondaries[name] = r2
            except Exception as exc:
                secondaries[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        if world == 1:
            try:
                secondaries["c5_resident"] = resident_leg(cx, "c5", args.steps)
            except Exception as exc:
                secondaries["c5_resident"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        USE_DDA = args.raycaster == "dda"

    if rank == 0:
        scaling = res.pop("scaling")
        P = WORKLOADS[args.workload][1]
        spread = WORKLOADS[args.workload][4] or args.spread
        line = {"metric": metric_name(n_lik), "value": res.pop("value"), "unit": "evals/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": res.pop("ms_per_step"), "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(args.workload, s, P if scaling == "strong" else P_rank * world, n_lik, n_beam,
                                      spread, WORKLOADS[args.workload][5]),
                "clocks": clk, "e2e": e2e, "gpu_launches": int(res["launches_per_step"] * args.steps),
                "roofline": res.pop("roofline"), "cpu_baseline": cpu_baseline, "exchange": res.pop("exchange"),
                "device_step": res, "workloads": secondaries, "notes": cx.notes,
                "match_ratio_mean": float(out_host["match_cnt"].mean() / max(n_lik, 1)) if out_host is not None else None,
                "beam_tallies_mean": ([float(out_host[f].mean()) for f in ("n_short", "n_hit", "n_long")]
                                      if out_host is not None else None)}
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
