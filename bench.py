#!/usr/bin/env python
"""bench.py — scans/s of the FAST-LIO2 per-scan hot path (BASELINE.json metric) on N B200s.

One "step" = one scan through the timed region of SURVEY.md §8d / laserMapping.cpp:2320,2380,2401:
lasermap_fov_segment -> update_iterated_dyn_share_modified (h_share_model 5-NN + plane + Jacobian, <=4 passes)
-> map_incremental, through the C ABI (libfastlio_b200.so).  Workload = BASELINE.json configs[1]:
64-line 120k-ray scans (all returns are queries, "Q-raw"), 0.2 m voxels, ~5M-point map, max_iteration = 3.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                     (the reference CPU path on the host cores)
  python bench.py --config cfg3|cfg4 ...                   (BASELINE configs[2], configs[3]: separate lines, kept in profiles/)

Prints ONE JSON line (rank 0).  PyTorch is used only for pinned/device buffers, stream events and the NCCL barrier.

Frame schedule (identical for both arms, independent of --steps): the workload is N_SCANS scans generated once from the
seed; frames 0..max(PARITY_FRAMES, W)-1 are replayed first, in order, from the freshly built map (the GPU posteriors of
frames 0..PARITY_FRAMES-1 are compared with the CPU replay of the same frames: the `parity` key); the K timed steps follow
in frame order (wrapping around the scan list when K is larger).  The other timed rows (e2e, sequential) each start from
a rebuilt map (untimed) with W warm-up frames and time K steps too.

  --dump-outputs DIR   after the timed steps, write what the last timed step computed (posterior state, covariance,
                       counters, the map it left) as DIR/<name>.npy, for output-for-output comparison of two builds
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scans/s (120k-pt, 3 ESIKF iters) at 1xB200; kNN+Jacobian HBM GB/s vs peak"
ALG_BYTES_PER_QUERY_SEARCH = 176  # SURVEY.md §8d: 16 query + 80 neighbours read + 80 neighbour-cache write
DS = 0.2
MAX_ITER = 3
MAP_AREA = 112000.0  # bounding area (m^2) of the pre-filled region that yields ~5M map points at 0.2 m
N_SCANS = 120        # scans of the cfg2 workload (fixed: map extent and RNG stream do not depend on --steps)
PARITY_FRAMES = 25   # frames replayed first (GPU and CPU) for the per-frame pose parity
REF_STEPS_CAP = 12   # --impl reference: bounded sample (~0.35 s of CPU work per step)
MIN_TIMED_MS = 500.0  # a timed window shorter than this is noted on stderr (more --steps give a steadier figure)
DUMP_BYTES = 64 << 20  # --dump-outputs: at most this much in all
SEED = 20


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  The reference's ikd-Tree (compiled unmodified into oracle/_ref for the CPU legs)
# printf()s its own thread messages (ikd_Tree.cpp:176,314), also at process teardown: file descriptor 1 is therefore
# pointed at stderr for the whole run and the JSON line is written to the saved real stdout.
_REAL_STDOUT = None


def protect_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


NCU_SHORT = False  # --ncu-short: the same workload, cut to a few steps (every kernel is replayed by the profiler)
TINY = False  # --tiny: test-only shrink of the workload (NOT a bench configuration; used by tests/test_bench_dist.py)


def n_scans_default():
    return 8 if TINY else N_SCANS


def parity_frames_default():
    return 3 if (TINY or NCU_SHORT) else PARITY_FRAMES


SENSOR_HEIGHT = 1.8  # the world origin is the first sensor pose (as in a FAST-LIO run): the ground plane is at z = -1.8 m


def make_workload(seed, n_scans, need_map=True, origin_height=SENSOR_HEIGHT, stream=0):
    """Seeded cfg2 workload: world, map pre-fill (~5M pts), n_scans HDL-64 scans + priors along a 10 m/s trajectory.

    origin_height: height of the world origin above the ground plane.  FAST-LIO's world frame is the first IMU pose, so the
    ground lies ~a sensor height BELOW the origin.  (Round 1 generated the ground at z = 0: every ground plane fit of
    esti_plane — it solves A x = -1, common_lib.h:506-536, singular for a plane through the origin — was then ill-conditioned
    in float32 and the closed loop amplified 1-ulp differences by 1e5 per frame; see DESIGN.md §6a.)

    stream: independent realisation of the SAME route (world, pre-filled map, trajectory): its own range noise and priors.  The
    multi-GPU replicas use stream = rank, so that every GPU does the same amount of work (weak scaling: per-GPU work fixed) on
    an independent session; stream 0 is the single-GPU workload."""
    from better_fastlio2_b200 import synth
    rng = np.random.default_rng(seed)
    dz = -float(origin_height)
    world = synth.city_world(half_extent=60.0 if TINY else 400.0, seed=seed).shifted((0.0, 0.0, dz))
    dirs = synth.lidar_dirs("vlp16" if TINY else "hdl64")
    centre = (0.5 * n_scans, 0.0, 0.0)
    # the pre-filled map covers everything the trajectory will see (sensor range 100 m ahead of / behind the path), so
    # the timed steps run in the steady state of a rolling map; its size is kept near 5M points by the lateral extent
    xh = 0.5 * n_scans + 105.0
    half = 20.0 if TINY else (xh, max(105.0, MAP_AREA / (4.0 * xh)), 1e3)
    mp = synth.sample_surface_map(world, centre, half, DS, rng, zmax=25.0 + dz) if need_map else None
    if stream:
        rng = np.random.default_rng([seed, stream])
    scans, priors, truths = [], [], []
    for k in range(n_scans):
        st = synth.trajectory_state(k, speed=10.0, z=1.8 + dz)
        body = synth.scan_from_pose(world, st, dirs, rng, max_range=100.0, min_range=2.0)
        scans.append(body)
        truths.append(st)
        priors.append(synth.perturb_state(st, rng, 0.05, 0.5))
    return dict(map=mp, scans=scans, priors=priors, truths=truths, P=synth.default_cov(), world=world, dirs=dirs)


def workload_config():
    """The `config` object: identical in both arms (the driver compares them)."""
    return {"workload": "cfg2: HDL-64 120k-ray scans (Q-raw), 0.2 m voxel, ~5M-pt map, max_iteration=3; one independent "
                        "session per GPU (cfg5: the same route and map on every GPU = fixed per-GPU work, own range noise and priors)",
            "seed": SEED, "n_scans": n_scans_default(), "parity_frames": parity_frames_default(),
            "frame_schedule": "cycle 0: frames 0..max(parity_frames, W)-1 from the fresh map (untimed, frames 0..parity_frames-1 "
                              "checked against the CPU replay), then K consecutive timed frames; every further timed row: map "
                              "rebuilt (untimed), W warm-up frames, K frames",
            "pipeline": "replay: two steps in flight",
            "l2_policy": "inputs larger than L2: ~480 MB of map block storage + a new 1.9 MB scan every step",
            "reference_arm": f"same workload and frame schedule; steps capped at {REF_STEPS_CAP} (bounded CPU sample)"}


def build_map(tree, pts, first=100000):
    """Populate a map the way a running node does (laserMapping.cpp:2328-2342 then map_incremental every scan): Build on a
    first cloud, everything else through Add_Points(downsample_on=true) -> at most one point per voxel (the one nearest
    the voxel centre), instead of a verbatim Build of a dense cloud that would leave many multi-point voxels."""
    tree.Build(pts[:first])
    step = 1 << 20
    for i in range(first, len(pts), step):
        tree.Add_Points(pts[i:i + step], True)


class ClockSampler:
    """SM clock / throttle reasons of one GPU during the timed region (B200_PROFILING.md), sampled in-process through
    NVML (nvidia-smi subprocess as the fallback)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0, period=0.02):
        self.rows, self.proc, self.index, self.period = [], None, index, period
        self.nv, self.h, self.stop_flag, self.th = None, None, False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nv = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nv
        names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)]
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                self.rows.append((sm, self.mx, [n for n, b in names if rs & b]))
            except Exception:
                pass
            time.sleep(self.period)

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 7:
                continue
            try:
                self.rows.append((float(f[0]), float(f[1]), [n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")]))
            except ValueError:
                continue

    def wait_first(self, timeout=5.0):
        t0 = time.time()
        while (self.nv or self.proc) and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        return len(self.rows)

    def stop(self, lo=0, hi=None):
        if not (self.nv or self.proc):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        time.sleep(0.05)
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        rows = self.rows[lo:(hi if hi is not None else len(self.rows)) + 1] or self.rows[-3:]
        sm = [r[0] for r in rows]
        mx = [r[1] for r in rows]
        reasons = sorted({x for r in rows for x in r[2]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons, "source": "nvml" if self.nv else "nvidia-smi"}


def cpu_step_runner(work, threads):
    """The reference CPU path (oracle: reference ikd-Tree compiled unmodified + restated h_share_model/ESIKF)."""
    from oracle import pyoracle as po
    from better_fastlio2_b200 import synth
    po.build()
    mp = po.make_map(ds=DS, threads=threads)
    t0 = time.perf_counter()
    build_map(mp, work["map"])
    build_s = time.perf_counter() - t0
    fov = po.FovSegment(cube_len=1000.0, det_range=100.0)
    state = {"pos_lid": np.zeros(3)}

    def step(k):
        body = work["scans"][k]
        boxes = fov.step(state["pos_lid"])
        if len(boxes):
            mp.Delete_Point_Boxes(boxes)
        s, P, sc, st, _ = po.esikf_update(work["priors"][k], work["P"], body, mp, max_iter=MAX_ITER)
        state["pos_lid"] = s[0:3] + synth.quat_to_mat(s[3:7]) @ s[11:14]
        po.map_incremental(s, body, sc, mp, True, DS)
        return s

    return mp, step, build_s


def dist_max(values, device=None, group_ready=None):
    """Max over ranks of a list of floats (NCCL on GPUs, gloo on CPU); identity when not distributed."""
    import torch
    import torch.distributed as dist
    t = torch.tensor(values, dtype=torch.float64, device=device if device is not None else "cpu")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t]


def dist_gather(values, device=None):
    """Every rank's list of floats, as [world][len] (all_gather); [[values]] when not distributed."""
    import torch
    import torch.distributed as dist
    t = torch.tensor(values, dtype=torch.float64, device=device if device is not None else "cpu")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
        dist.all_gather(out, t)
        return [[float(x) for x in o] for o in out]
    return [[float(x) for x in t]]


def aggregate_scans_per_s(world_size, steps, ms_max):
    """Whole-job throughput: every rank processed `steps` scans of its own session (weak scaling) in ms_max."""
    return world_size * steps / (ms_max * 1e-3)


def map_sample(pts, max_rows):
    """The map's points in sorted row order; above max_rows, the points whose coordinate hash falls below a fixed
    threshold (a sample that depends on each point alone, so two nearly equal maps give nearly equal samples)."""
    pts = np.ascontiguousarray(pts, np.float32)
    if len(pts) > max_rows:
        b = pts.view(np.uint32).astype(np.uint64)
        h = (b[:, 0] * 73856093 ^ b[:, 1] * 19349663 ^ b[:, 2] * 83492791) & 0xFFFFFFFF
        pts = pts[h < np.uint64(int(0.95 * max_rows / len(pts) * 2 ** 32))]
    return pts[np.lexsort((pts[:, 2], pts[:, 1], pts[:, 0]))][:max_rows]


def dump_outputs(out_dir, state, P, r, map_points):
    """What the last timed step handed its caller: posterior state (x26) and covariance (23x23), the step's counters
    (update passes, search passes, effective features, converged count, total residual, points added with / without
    downsampling, points deleted, map size; timings left out) and the map it left (float32 xyz rows, sorted)."""
    os.makedirs(out_dir, exist_ok=True)
    u = r.update
    counters = np.array([u.passes, u.search_passes, u.effct_feat_num, u.converged_count, u.total_residual, r.n_to_add,
                         r.n_no_downsample, r.n_deleted, r.map_valid], np.float64)
    arrays = {"state": np.asarray(state, np.float64), "covariance": np.asarray(P, np.float64), "counters": counters}
    room = DUMP_BYTES - sum(a.nbytes for a in arrays.values()) - 4096
    arrays["map_points"] = map_sample(map_points, room // 12)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"dumped {', '.join(f'{k}{list(v.shape)}' for k, v in arrays.items())} to {out_dir}")


def quat_angle(qa, qb):
    """Rotation angle (rad) between two unit quaternions (x,y,z,w): 2*|vec(qa^-1 qb)| (accurate for tiny angles)."""
    ax, ay, az, aw = qa
    bx, by, bz, bw = qb
    vx = aw * bx - ax * bw - ay * bz + az * by
    vy = aw * by - ay * bw - az * bx + ax * bz
    vz = aw * bz - az * bw - ax * by + ay * bx
    return 2.0 * float(np.sqrt(vx * vx + vy * vy + vz * vz))


def pose_parity(post_a, post_b):
    """Per-frame pose difference of two replays of the same frames (north_star: <= 1e-4 m / 1e-4 rad per frame)."""
    n = min(len(post_a), len(post_b))
    dpos = [float(np.linalg.norm(np.asarray(post_a[k][:3]) - np.asarray(post_b[k][:3]))) for k in range(n)]
    drot = [quat_angle(post_a[k][3:7], post_b[k][3:7]) for k in range(n)]
    kmax = int(np.argmax(dpos)) if n else -1
    return {"frames": n, "max_dpos_m": max(dpos) if n else None, "max_drot_rad": max(drot) if n else None,
            "frame_of_max": kmax, "dpos_m": dpos, "tolerance": "1e-4 m / 1e-4 rad per frame (BASELINE north_star)"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores = os.cpu_count() or 1
    NS, F = n_scans_default(), parity_frames_default()
    work = make_workload(SEED, NS)
    mp, step, build_s = cpu_step_runner(work, ncores)
    W, K = args.warmup, args.steps
    w = max(F, W)
    for k in range(w):               # cycle 0 of the repo arm's frame schedule: settle frames (>= W warm-up), then the timed block
        step(k)
    t0 = time.perf_counter()
    for j in range(K):
        step((w + j) % NS)
    dt = time.perf_counter() - t0
    val = K / dt
    # the reference's own thread policy (MP_PROC_NUM = 3, CMakeLists.txt:11-24) on a few further frames, beside the all-core figure
    mp.set_threads(3)
    t0 = time.perf_counter()
    S3 = min(4, K)
    for j in range(S3):
        step((w + K + j) % NS)
    v3 = S3 / (time.perf_counter() - t0)
    npts = float(np.mean([len(s) for s in work["scans"]]))
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "scans/s", "n_gpus": args.gpus, "steps": K,
           "warmup": W, "ms_per_step": 1e3 * dt / K, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32 search/plane + f64 Jacobian/ESIKF", "data": "synthetic",
           "config": workload_config(),
           "workload_stats": {"scan_points_mean": npts, "map_points_in": int(len(work["map"])), "map_valid": int(mp.validnum())},
           "cpu_baseline": {"value": val, "unit": "scans/s", "cores": ncores,
                            "kind": "reference" if mp.kind == "reference" else "port",
                            "sample": f"{K} timed steps (frames {w}..{w + K - 1}) after {w} settle frames; ikd-Tree = reference source "
                                      f"compiled unmodified (Build {build_s:.1f}s untimed), search on all {ncores} host threads, "
                                      "Add_Points serial; h_share_model/ESIKF = restated port",
                            "value_mp_proc_num_3": v3},
           "e2e": {"value": val, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def run_b200(args):
    import torch
    import torch.distributed as dist
    from better_fastlio2_b200 import capi
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if capi.device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    devname = f"cuda:{local}"
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W, K = args.warmup, args.steps
    PROF = 10 if not (TINY or NCU_SHORT) else 2  # profiled steps (per-kernel CUDA-event timing) after the timed regions
    NS, F = n_scans_default(), parity_frames_default()
    t_gen = time.perf_counter()
    work = make_workload(SEED, NS, stream=rank)  # cfg5: one independent session per GPU (same route, own noise and priors)
    log(f"[rank {rank}] workload: map {len(work['map'])} pts, {NS} scans, gen {time.perf_counter() - t_gen:.1f}s")
    tree = capi.KDTree(voxel_size=DS, max_points=16 << 20, max_blocks=2 << 20, device=local)
    build_map(tree, work["map"])
    nmax = max(len(s) for s in work["scans"])
    ses = capi.Session(tree, max_scan_points=max(131072, nmax), max_iterations=MAX_ITER, filter_size_map_min=DS)
    fov = capi.make_fov(cube_len=1000.0, det_range=100.0)
    stream = torch.cuda.ExternalStream(ses.stream_ptr(), device=torch.device("cuda", local))
    # device-resident copies (for `value`) and pinned host copies (for `e2e`)
    dev, pin = [], []
    for s in work["scans"]:
        b4 = np.zeros((len(s), 4), np.float32)
        b4[:, :3] = s
        dev.append(torch.from_numpy(b4).to(devname))
        pin.append(torch.from_numpy(b4).pin_memory())
    torch.cuda.synchronize()
    P0 = work["P"]
    nk_all = [len(s) for s in work["scans"]]
    dptr_all = [d.data_ptr() for d in dev]
    pptr_all = [p.data_ptr() for p in pin]
    set_dev, step_ptr = ses.scan_set_device, ses.scan_step_ptr

    def barrier():
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- frame schedule.  A CYCLE starts from the freshly built map: `w` untimed frames 0..w-1 (cycle 0:
    # w = max(F, W), the posteriors of frames 0..F-1 are the ones checked against the CPU replay — the `parity` key; later
    # cycles: w = W warm-up steps), then one block of exactly K consecutive frames.  The map is rebuilt (untimed) between
    # cycles so that every timed block sees the same, well-defined map state: replaying a scan list over and over into ONE
    # map would keep appending its verbatim (PointNoNeedDownsample) points and grow overflow chains no real trajectory
    # produces.  Nothing in the schedule depends on a measured time, so the same arguments replay the same frames.
    fov_box = [fov]

    def block(w):
        return [(w + j) % NS for j in range(K)]

    def begin_cycle(first):
        w = max(F, W) if first else max(W, 0)
        if not first:
            build_map(tree, work["map"])
            fov_box[0] = capi.make_fov(cube_len=1000.0, det_range=100.0)
        out = []
        for k in range(w):
            r, st = step_dev(k)
            out.append((r, st))
        return w, out

    def step_dev(k):
        set_dev(dptr_all[k], nk_all[k])
        st = work["priors"][k].copy()
        P = P0.copy()
        return step_ptr(fov_box[0], None, 0, 0, st, P), st

    clocks = ClockSampler(local)
    clocks.start()
    clocks.wait_first()
    barrier()
    w0, settle = begin_cycle(True)
    post = [st for _, st in settle[:F]]
    valid_after = settle[F - 1][0].map_valid if settle else 0

    # ---------------- timed region 1: inputs resident in HBM (value).  One block = EXACTLY K steps between a barrier +
    # synchronize on both sides, timed with CUDA events on the library stream (max over ranks).
    def timed_block(idx, pipelined=True):
        # the harness keeps its own work out of the timed loop (a C++ caller has none): states/covariances are staged
        # beforehand, results are inspected afterwards
        sts = [work["priors"][k].copy() for k in idx]
        Ps = [P0.copy() for _ in idx]
        res = [None] * K
        f = fov_box[0]
        begin, finish = ses.scan_step_begin, ses.scan_step_finish
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        if pipelined:
            # two steps in flight: scan j+1 is enqueued (its prior is known: replay) before scan j's posterior is collected,
            # so the GPU never waits for the host between scans
            set_dev(dptr_all[idx[0]], nk_all[idx[0]])
            begin(f, sts[0], Ps[0], True)
            for j in range(K):
                if j + 1 < K:
                    set_dev(dptr_all[idx[j + 1]], nk_all[idx[j + 1]])
                    begin(f, sts[j + 1], Ps[j + 1], True)
                res[j] = finish(f, sts[j], Ps[j])
        else:
            for j in range(K):
                set_dev(dptr_all[idx[j]], nk_all[idx[j]])
                res[j] = step_ptr(f, None, 0, 0, sts[j], Ps[j])
        e1.record(stream)
        barrier()
        perr = max(float(np.linalg.norm(sts[j][:3] - work["truths"][idx[j]][:3])) for j in range(K))
        return e0.elapsed_time(e1), sum(r.kernel_launches for r in res), sum(nk_all[k] for k in idx), perr, (sts[-1], Ps[-1], res[-1])

    # ---------------- timed region 2: host buffers through the C ABI (e2e).  Streaming use of the public API: every
    # step's scan is copied from pinned host memory inside the region (flb_scan_prefetch, overlapping the previous
    # step's kernels) and every step's posterior state / covariance / counters are read back to the host.
    def e2e_block(idx, pipelined=True):
        sts2 = [work["priors"][k].copy() for k in idx]
        Ps2 = [P0.copy() for _ in idx]
        pptr = [pptr_all[k] for k in idx] + [0, 0]
        pn = [nk_all[k] for k in idx] + [0, 0]
        res2 = [None] * K
        lat = np.empty(K)
        f = fov_box[0]
        barrier()
        t0 = time.perf_counter()
        ses.scan_prefetch_ptr(pptr[0], pn[0], 16)
        tp = t0
        if pipelined:
            ses.scan_step_begin(f, sts2[0], Ps2[0], True)
            if K > 1:
                ses.scan_prefetch_ptr(pptr[1], pn[1], 16)
            for j in range(K):
                if j + 1 < K:
                    ses.scan_step_begin(f, sts2[j + 1], Ps2[j + 1], True)     # adopts the prefetched scan j+1
                res2[j] = ses.scan_step_finish(f, sts2[j], Ps2[j])            # scan j done: its buffer is free again
                if j + 2 < K:
                    ses.scan_prefetch_ptr(pptr[j + 2], pn[j + 2], 16)
                tn = time.perf_counter()
                lat[j] = tn - tp
                tp = tn
        else:
            for j in range(K):
                ses.scan_step_begin(f, sts2[j], Ps2[j], True)
                if j + 1 < K:
                    ses.scan_prefetch_ptr(pptr[j + 1], pn[j + 1], 16)
                res2[j] = ses.scan_step_finish(f, sts2[j], Ps2[j])
                tn = time.perf_counter()
                lat[j] = tn - tp    # posterior-to-posterior period of the streaming loop (host clock)
                tp = tn
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        return dt * 1e3, lat, sum(r.update.passes for r in res2), sum(nk_all[k] for k in idx)

    row_lo = clocks.mark()
    own_ms, launches, npts, perr, last = timed_block(block(w0))
    row_hi = clocks.mark()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last, tree.flatten())
    ms = dist_max([own_ms], device=devname)[0]
    if ms < MIN_TIMED_MS and not (TINY or NCU_SHORT):
        log(f"note: the {K} timed steps took {ms:.1f} ms of device time; more --steps give a steadier figure")
    w, _ = begin_cycle(False)
    own_e2e_ms, lat, passes, _ = e2e_block(block(w))
    e2e_ms = dist_max([own_e2e_ms], device=devname)[0]
    # the strictly alternating begin / finish figures (a live filter, whose next prior needs this posterior)
    w, _ = begin_cycle(False)
    seq_ms = dist_max([timed_block(block(w), pipelined=False)[0]], device=devname)[0]
    w, _ = begin_cycle(False)
    seq_e2e_ms, seq_lat, _, _ = e2e_block(block(w), pipelined=False)
    seq_e2e_ms = dist_max([seq_e2e_ms], device=devname)[0]
    clk = clocks.stop(row_lo, row_hi)
    # per-rank view of the same measurement: own block time, own GPU's clocks, own e2e
    mine = [own_ms, own_e2e_ms, float(clk["sm_mhz"] or 0.0), float(clk["sm_max_mhz"] or 0.0), float(len(clk["reasons"]))]
    per_rank = dist_gather(mine, device=devname)
    fov = fov_box[0]

    # ---------------- profiled replay: per-kernel-class CUDA events on the library stream (event timing needs the
    # direct-launch path — no CUDA graph, no side-stream overlap — so it is kept out of the two headline loops)
    tree.profile_enable(True)
    npts_prof = 0
    w, _ = begin_cycle(False)
    for k in range(w, w + PROF):
        step_dev(k % NS)
        npts_prof += nk_all[k % NS]
    prof = tree.profile_read(reset=True)
    tree.profile_enable(False)
    solo = world_size == 1 and not args.no_cpu_baseline
    frontend = frontend_rows(work, ses, fov, torch, local, F, rank, cpu=solo) if not (TINY or NCU_SHORT) else None
    stats = tree.stats()
    ses.close()
    tree.close()
    frontier = frontier_rows(work, torch, local) if (rank == 0 and not (TINY or NCU_SHORT)) else None
    if rank == 0:
        peaks = {}
        pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk_path):
            peaks = json.load(open(pk_path))
        peak = float(peaks.get("hbm_gbs", 6650.0))
        knn = prof["knn"]
        n_mean = npts / K
        # k-NN regions of non-search passes are empty launches (device-side early exit): only search passes count
        searches = max(sum(prof["knn_phase"]) / max(npts_prof / PROF, 1), 1e-9)   # search passes actually run
        knn_ms = knn["ms"] / searches
        achieved = ALG_BYTES_PER_QUERY_SEARCH * (npts_prof / PROF) / (knn_ms * 1e-3) / 1e9 if knn_ms > 0 else 0.0
        value = aggregate_scans_per_s(world_size, K, ms)
        out = {
            "metric": METRIC, "value": value, "unit": "scans/s", "n_gpus": world_size, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 search/plane + f64 Jacobian/ESIKF", "data": "synthetic",
            "config": workload_config(),
            "workload_stats": {"scan_points_mean": n_mean, "map_valid": int(stats["valid_points"]),
                               "map_block_storage_mb": stats["blocks_in_use"] * 1024 / 1e6, "pose_err_vs_truth_max_m": perr},
            "timing": {"what": f"one block of exactly {K} steps (frames {w0}..{w0 + K - 1} mod {NS}) between barrier+synchronize, "
                               "CUDA events on the library stream, max over ranks",
                       "pipeline": "two steps in flight (flb_scan_step_begin of scan j+1 before flb_scan_step_finish of scan j: replay, the "
                                   "priors are known); `sequential` = strictly alternating begin / finish",
                       "sequential": {"value": aggregate_scans_per_s(world_size, K, seq_ms), "e2e": aggregate_scans_per_s(world_size, K, seq_e2e_ms),
                                      "latency_ms_p50": float(np.percentile(seq_lat, 50) * 1e3),
                                      "latency_ms_p99": float(np.percentile(seq_lat, 99) * 1e3)},
                       "block_ms": ms, "e2e_block_ms": e2e_ms},
            "per_rank": [{"rank": i, "block_ms": r[0], "e2e_block_ms": r[1], "sm_mhz": r[2], "sm_max_mhz": r[3],
                          "throttle_reasons": int(r[4])} for i, r in enumerate(per_rank)],
            "slowest_rank": int(np.argmax([r[0] for r in per_rank])),
            "sum_of_rank_rates": float(sum(K / (r[0] * 1e-3) for r in per_rank)),   # (each rank's own block; NOT the headline)
            "gpu_launches": launches,
            "latency_ms": {"p50": float(np.percentile(lat, 50) * 1e3), "p99": float(np.percentile(lat, 99) * 1e3),
                           "max": float(lat.max() * 1e3), "samples": int(len(lat)),
                           "what": "per-scan period of the e2e loop (host buffers, host clock)"},
            "device_bytes": int(stats.get("device_bytes", 0)),
            "e2e": {"value": aggregate_scans_per_s(world_size, K, e2e_ms), "unit": "scans/s",
                    "h2d_bytes_per_step": int(16 * n_mean), "d2h_bytes_per_step": int(passes / K * 93 * 8 + 2 * 128 + 8)},
            "roofline": {"bound": "hbm", "kernel": "k_knn_stencil<5> + k_knn<5> (one 5-NN search pass)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": knn_traffic(),
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6.65 TB/s",
                         "alg_bytes_per_launch": ALG_BYTES_PER_QUERY_SEARCH * (npts_prof / PROF), "avg_launch_ms": knn_ms,
                         "launches_timed": searches,
                         "how": f"CUDA events on the library stream around every k-NN pass (k_knn_stencil + k_knn) over a "
                                f"profiled replay of {PROF} further steps of the same workload, direct-launch path"},
            "kernel_ms_per_step": {k: prof[k]["ms"] / PROF for k in capi.K_CLASSES},
            "knn_phase_fraction": [x / max(sum(prof["knn_phase"]), 1) for x in prof["knn_phase"]],
            "knn_per_query": {"stencil_voxels": prof["knn_head_candidates"] / max(sum(prof["knn_phase"]), 1),
                              "chain_nodes": prof["knn_chain_nodes"] / max(sum(prof["knn_phase"]), 1),
                              "chain_nodes_max": prof["knn_chain_max"]},
            "map_stats": {k: stats[k] for k in ("blocks_in_use", "overflow_in_use", "coarse_cells", "hash_tombstones")},
            "clocks": clk,
        }
        if frontend:
            out["frontend"] = frontend
        if frontier:
            out["frontier"] = frontier
        if solo:
            cb, cpu_post, cpu_valid = cpu_baseline(work, F)
            out["cpu_baseline"] = cb
            par = pose_parity(post, cpu_post)
            par["what"] = ("GPU posterior vs the CPU replay (reference ikd-Tree compiled unmodified + restated h_share_model/ESIKF, "
                           "unpinned) of the same frames 0..frames-1 from the same initial map")
            par["map_size_diff"] = int(abs(valid_after - cpu_valid))
            out["parity"] = par
        emit(out)
    if world_size > 1:
        dist.destroy_process_group()


def knn_traffic():
    """dram bytes per k-NN launch from this round's `ncu --set full` capture (tools/gpu_round.sh writes
    profiles/knn_traffic.json with the md5 of csrc/knn_kernels.cuh it was taken on); null when the kernel changed since."""
    import hashlib
    tr_path = os.path.join(ROOT, "profiles", "knn_traffic.json")
    try:
        rec = json.load(open(tr_path))
        src = open(os.path.join(ROOT, "better_fastlio2_b200", "csrc", "knn_kernels.cuh"), "rb").read()
        if rec.get("knn_kernels_md5") != hashlib.md5(src).hexdigest():
            return None
        return rec.get("dram_bytes_per_launch")
    except Exception:
        return None


def frontier_rows(work, torch, local, S=40):
    """Exploration regime (NOT the headline): a node starting up (laserMapping.cpp:2328-2342: Build on the first scan) whose
    map only ever holds what the previous scans inserted through map_incremental, so every scan has returns with no map
    behind them; the filter is CHAINED (prior = previous posterior moved by the true relative motion) and additionally
    perturbed by 20 cm / 2 deg.  Device-resident inputs, CUDA events over the S steps."""
    from better_fastlio2_b200 import capi, synth
    rng = np.random.default_rng(777)
    S = min(S, len(work["scans"]) - 1)
    tree = capi.KDTree(voxel_size=DS, max_points=16 << 20, max_blocks=2 << 20, device=local)
    tree.Build(synth.body_to_world_np(work["truths"][0], work["scans"][0]))
    nmax = max(len(s) for s in work["scans"])
    ses = capi.Session(tree, max_scan_points=max(131072, nmax), max_iterations=MAX_ITER, filter_size_map_min=DS)
    fov = capi.make_fov(cube_len=1000.0, det_range=100.0)
    stream = torch.cuda.ExternalStream(ses.stream_ptr(), device=torch.device("cuda", local))
    dev = []
    for s in work["scans"][:S + 1]:
        b4 = np.zeros((len(s), 4), np.float32)
        b4[:, :3] = s
        dev.append(torch.from_numpy(b4).to(f"cuda:{local}"))
    torch.cuda.synchronize()
    post = work["truths"][0].copy()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    errs, lat, launches = [], [], 0
    for k in range(1, S + 1):
        if k == 2:
            e0.record(stream)     # (scan 1 is the warm-up: it pays the session's graph capture)
        pri = post.copy()
        pri[0:3] += work["truths"][k][0:3] - work["truths"][k - 1][0:3]
        pri[3:7] = work["truths"][k][3:7]
        pri = synth.perturb_state(pri, rng, 0.2 / np.sqrt(3.0), 2.0 / np.sqrt(3.0))   # |error| ~ 20 cm / 2 deg
        P = work["P"].copy()
        ses.scan_set_device(dev[k].data_ptr(), len(work["scans"][k]))
        t0 = time.perf_counter()
        r = ses.scan_step_ptr(fov, None, 0, 0, pri, P)
        lat.append(time.perf_counter() - t0)
        launches += r.kernel_launches
        post = pri
        errs.append(float(np.linalg.norm(post[:3] - work["truths"][k][:3])))
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    st = tree.stats()
    ses.close()
    tree.close()
    S = S - 1
    lat = lat[1:]
    return {"what": "exploration regime: map = first scan + what map_incremental inserted, chained filter, prior off by ~20 cm / 2 deg; "
                    "device-resident scans, CUDA events over all steps after one warm-up scan",
            "steps": S, "scans_per_s": S / (ms * 1e-3), "ms_per_step": ms / S, "step_ms_p50": float(np.median(lat) * 1e3),
            "step_ms_max": float(max(lat) * 1e3),
            "pose_err_vs_truth_max_m": max(errs), "pose_err_vs_truth_last_m": errs[-1], "map_valid_end": int(st["valid_points"]),
            "gpu_launches": launches}


def frontend_rows(work, ses, fov, torch, local, k0, rank, S=20, leaf=0.5, cpu=True):
    """SURVEY.md §8f rows measured beside the headline (NOT part of `value`/`e2e`): the raw 120k-point scan goes
    host -> UndistortPcl backward pass -> pcl::VoxelGrid(leaf) -> update -> map_incremental ("Q-ds" query mode: the queries
    are the filtered scan, as laserMapping.cpp:2322 does), all through the C ABI from pinned host buffers; the CPU figure
    is the oracle's restatement of the same two front-end steps on one core (PCL / the reference run them serially)."""
    from better_fastlio2_b200 import capi, synth
    rng = np.random.default_rng(99 + rank)
    nmax = max(len(s) for s in work["scans"])
    fe = capi.FrontEnd(ses, max_raw_points=max(131072, nmax))
    ks = [(k0 + j) % len(work["scans"]) for j in range(S)]
    raw, poses, ends = [], [], []
    for k in ks:
        xyz, inten, cur = synth.raw_scan_with_times(work["scans"][k], rng, shuffle=False)
        raw.append(torch.from_numpy(capi.pack_pointtype(xyz, inten, cur)).pin_memory())
        # a sensor (almost) at rest during the sweep: the synthetic scans carry no motion distortion, so the compensation
        # must stay ~identity while still running its full arithmetic (non-zero gyro -> Rodrigues path)
        st = work["priors"][k]
        R = synth.quat_to_mat(st[3:7]).reshape(-1)
        pz = [np.concatenate([[0.005 * j], [1e-4, 0, 0], [1e-5, 2e-5, -1e-5], [1e-4, 0, 0], st[0:3], R]) for j in range(21)]
        pz[0][0] = 0.0
        poses.append(np.array(pz))
        ends.append(st.copy())
    P0 = work["P"]

    def one(i, with_step=True):
        n = fe.process_ptr(raw[i].data_ptr(), raw[i].shape[0], poses[i], ends[i], leaf)
        if with_step:
            st, P = work["priors"][ks[i]].copy(), P0.copy()
            ses.scan_step_ptr(fov, None, 0, 0, st, P)
        return n

    one(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    nd = [one(i, with_step=False) for i in range(S)]
    torch.cuda.synchronize()
    t_front = (time.perf_counter() - t0) / S
    t0 = time.perf_counter()
    for i in range(S):
        one(i)
    torch.cuda.synchronize()
    t_all = (time.perf_counter() - t0) / S
    # stage breakdown (wall clock with a synchronisation after every stage: an upper bound per stage, not additive)
    stage = {"upload_ms": 0.0, "undistort_ms": 0.0, "voxel_filter_ms": 0.0}
    for i in range(min(S, 8)):
        t0 = time.perf_counter()
        fe.upload_ptr(raw[i].data_ptr(), raw[i].shape[0])
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        fe.undistort(poses[i], ends[i])
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        fe.voxel_filter(leaf)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        stage["upload_ms"] += 1e3 * (t1 - t0) / min(S, 8)
        stage["undistort_ms"] += 1e3 * (t2 - t1) / min(S, 8)
        stage["voxel_filter_ms"] += 1e3 * (t3 - t2) / min(S, 8)
    out = {"what": "raw scan (host, 48-B PointType) -> undistort -> VoxelGrid -> update -> map_incremental; wall clock, host buffers",
           "stages_synced": stage,
           "leaf": leaf, "raw_points_mean": float(np.mean([r.shape[0] for r in raw])), "down_points_mean": float(np.mean(nd)),
           "front_ms_per_scan": 1e3 * t_front, "scans_per_s_raw_to_posterior": 1.0 / t_all, "samples": S,
           "h2d_bytes_per_scan": int(48 * np.mean([r.shape[0] for r in raw]))}
    if rank == 0 and cpu:   # part of the cpu_baseline leg (rank 0, N = 1 only): the oracle timed on one host core
        try:
            from oracle import pyoracle as po
            t0 = time.perf_counter()
            for i in range(3):
                a = raw[i].numpy()
                ox, op = po.undistort(a[:, 0:3].copy(), a[:, 9].copy(), poses[i], ends[i])
                po.voxel_grid(np.column_stack([ox, a[op, 8]]), leaf, order="pcl")
            out["cpu_front_ms_per_scan"] = 1e3 * (time.perf_counter() - t0) / 3
            out["cpu_kind"] = "port (oracle restatement of UndistortPcl backward pass + PCL 1.10 VoxelGrid), 1 core"
        except Exception as e:   # the oracle is test infrastructure: its absence must not break the bench line
            out["cpu_front_ms_per_scan"] = None
            out["cpu_kind"] = f"unavailable: {e}"
    fe.close()
    return out


def cpu_baseline(work, F):
    """Bounded sample of the same workload on the host cores with the reference's own thread policy (MP_PROC_NUM = 3,
    CMakeLists.txt:11-24): frames 0..F-1 in order from the same initial map (frame 0 = warm-up).  Returns the baseline
    record, the posteriors of the replayed frames (for the parity key) and the reference map's final size."""
    threads = 3
    F = max(2, min(F, len(work["scans"])))
    mp, step, build_s = cpu_step_runner(work, threads)
    post = [step(0)]
    t0 = time.perf_counter()
    for k in range(1, F):
        post.append(step(k))
    dt = time.perf_counter() - t0
    S = F - 1
    rec = {"value": S / dt, "unit": "scans/s", "cores": threads, "kind": "reference" if mp.kind == "reference" else "port",
           "sample": f"{S} scans of the same workload after 1 warm-up; ikd-Tree = reference source compiled unmodified "
                     f"(5M-pt Build {build_s:.1f}s untimed), search threads = 3 (MP_PROC_NUM), Add_Points serial; "
                     "h_share_model/ESIKF = restated port",
           "ms_per_scan": 1e3 * dt / S}
    return rec, post, int(mp.validnum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4"])
    ap.add_argument("--scans", type=int, default=0, help="cfg3/cfg4: number of consecutive scans (0 = the config's default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ncu-short", action="store_true", help="profiling runs under ncu: 3 settle frames, one timed block, no extra rows")
    ap.add_argument("--tiny", action="store_true", help="test-only: shrink the workload (not a bench configuration)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (state, covariance, counters, map)")
    args = ap.parse_args()
    global TINY, NCU_SHORT
    TINY = args.tiny
    NCU_SHORT = args.ncu_short
    protect_stdout()
    if args.warmup < 3 and args.impl == "b200":
        log("note: timing rules ask for >= 3 warm-up steps")
    if args.config != "cfg2":
        import bench_configs
        return bench_configs.run(args, sys.modules[__name__])
    if args.impl == "reference":
        args.steps = min(args.steps, REF_STEPS_CAP)  # bounded sample
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
