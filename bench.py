#!/usr/bin/env python
"""bench.py -- ICP registrations/s, 131072-point scan vs 524288-point rolling map, 30 iterations
(BASELINE.json configs[1]) on N B200s, one independent track per GPU.

A "step" = one scan-to-local-map registration (LaserTrack::localScanToSubMap -> icp_.compute,
reference laser_slam/src/laser_track.cpp:466-519) of the next scan of a synthetic HDL-64-shaped sequence.
  value : registrations/s with every scan already resident in HBM (ls_icp_register_submap only)
  e2e   : same metric through the public C-ABI with HOST buffers: every step uploads the new scan
          from pinned host memory (ls_map_push_scan) and reads the 4x4 result + stats back.
  --impl reference : the reference's CPU algorithm (oracle port: kd-tree 1-NN, nth_element trim,
          point-to-plane) on the host cores -- the reference's own libraries are absent (SURVEY.md §8c).
  --dump-outputs DIR : after the timed steps, write what the resident arm's last timed step returned to its
          caller, one DIR/<name>.npy per array (see dump_outputs); the inputs depend only on the arguments, so two
          builds run with the same arguments can be compared output for output.
Prints ONE JSON line on rank 0.  Writes nothing into the source tree.
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
sys.dont_write_bytecode = True   # the tree may be read-only; no __pycache__ next to the sources

# BASELINE.json configs[1] (default) and configs[4] (--config 5): scan size, scans per map, ICP iterations, sensor
WORKLOADS = {
    2: dict(n_scan=131072, k_map=4, iters=30, sensor=0, pool=24, tracks=74,
            name="configs[1]: scan-to-local-map ICP, 131072-pt scan vs 524288-pt rolling map (4 scans), 30 iterations",
            metric="ICP registrations/s (131072-pt scan vs 524288-pt map, 30 iterations)"),
    5: dict(n_scan=262144, k_map=8, iters=50, sensor=1, pool=14, tracks=8,
            name="configs[4]: dense-sensor stress, 262144-pt scan (VLS-128-like) vs 2097152-pt map (8 scans), 50 iterations",
            metric="ICP registrations/s (262144-pt scan vs 2097152-pt map, 50 iterations)"),
}
N_SCAN, K_MAP, ITERS, POOL, SENSOR = 131072, 4, 30, 24, 0   # set by select_workload()
ALG_BYTES_ICP = ALG_BYTES_REG = 0


def select_workload(cfg):
    """Algorithmic bytes (SURVEY.md §8d): 64 B per query per iteration + 68 B per map point for ingest/index."""
    global N_SCAN, K_MAP, ITERS, POOL, SENSOR, ALG_BYTES_ICP, ALG_BYTES_REG
    w = WORKLOADS[cfg]
    N_SCAN, K_MAP, ITERS, POOL, SENSOR = w["n_scan"], w["k_map"], w["iters"], w["pool"], w["sensor"]
    ALG_BYTES_ICP = 64 * N_SCAN * ITERS
    ALG_BYTES_REG = 68 * (K_MAP * N_SCAN) + ALG_BYTES_ICP
    return w


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region.  NVML in-process (the library nvidia-smi itself
    reads; no process is spawned next to the measurement); `nvidia-smi --query-gpu` only if NVML cannot be loaded."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BAD = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.stop_flag, self.source = gpu, [], False, "nvml"
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            phys = gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                tok = vis.split(",")[gpu].strip()
                phys = int(tok) if tok.isdigit() else None
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys) if phys is not None else pynvml.nvmlDeviceGetHandleByUUID(tok)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h, self.source = None, "nvidia-smi"

    def run(self):
        while not self.stop_flag:
            try:
                if self.h is not None:
                    sm = float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                    try:
                        mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        mask = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    self.samples.append((sm, self.max_sm, [n for n, bit in self.BAD if mask & bit]))
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    f = [x.strip() for x in out.split(",")]
                    if len(f) >= 8:
                        self.samples.append((float(f[1]), float(f[2]),
                                             [n for (n, _), v in zip(self.BAD, f[4:8]) if v.lower().startswith("active")]))
            except Exception:
                pass
            time.sleep(0.05 if self.h is not None else 0.25)

    def summary(self):
        self.stop_flag = True
        sm = [s[0] for s in self.samples]
        mx = [s[1] for s in self.samples]
        reasons = sorted({r for s in self.samples for r in s[2]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples), "source": self.source}


def make_pool(seq):
    from laser_slam_b200 import synth
    truth, odom = synth.trajectory(seq, POOL, y_start=-20.0)
    scans = [synth.scan(truth[k], seq, k, sensor=SENSOR) for k in range(POOL)]
    return truth, odom, scans


def make_pools(seqs):
    """One pool per sequence, generated on a few host threads (the generator is C++ behind ctypes: no GIL)."""
    from concurrent.futures import ThreadPoolExecutor
    from laser_slam_b200 import synth
    synth.build()
    with ThreadPoolExecutor(max_workers=min(16, usable_threads())) as ex:
        return list(ex.map(make_pool, seqs))


def walk(step):
    """Ping-pong index walk over the pool so consecutive steps are consecutive scans (a continuous drive)."""
    period = 2 * (POOL - 1)
    j = step % period
    return j if j < POOL else period - j


def submap_parts(truth, idx_hist):
    """Parts of the reference = the 4 scans before the newest, in the frame of the most recent of them."""
    ref = idx_hist[-2]
    ks = idx_hist[-2:-2 - K_MAP:-1]
    Ts = [np.eye(4, dtype=np.float32) if k == ref else (np.linalg.inv(truth[ref]) @ truth[k]).astype(np.float32) for k in ks]
    return ref, ks, Ts


def usable_threads():
    """Host threads the CPU arm may use: affinity mask, capped by the cgroup CPU quota if there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def best_thread_count(oracle, reading, refp, refn, T0):
    """The kd-tree query loop does not scale to every core count (memory bound; oversubscription under a
    quota): calibrate with 6 ICP iterations of the real workload and keep the fastest count -- the
    strongest CPU baseline this host can give."""
    nmax = usable_threads()
    cands = sorted({c for c in (1, 2, 4, 8, 16, 32, 64, nmax) if c <= nmax})
    t1 = {}
    for its in (2, 8):   # difference of two runs isolates the per-iteration (query) cost from the tree build
        for c in cands:
            po = oracle.default_params(max_iterations=its, use_differential=0, num_threads=c)
            t0 = time.perf_counter()
            oracle.icp(reading, refp, refn, T0, po)
            t1[(its, c)] = time.perf_counter() - t0
    return min(cands, key=lambda c: t1[(8, c)] - t1[(2, c)])


def run_reference(args, rank, wl):
    """The reference arm: the CPU algorithm on the host cores (oracle port; kind == "port")."""
    if rank != 0:
        return
    import oracle
    truth, odom, scans = make_pool(0)
    hist = [walk(s) for s in range(K_MAP + 1)]
    ref0, ks0, Ts0 = submap_parts(truth, hist)
    parts0 = [scans[k] if k == ref0 else oracle.transform_cloud(T, *scans[k]) for k, T in zip(ks0, Ts0)]
    threads = best_thread_count(oracle, scans[hist[-1]][0], np.concatenate([p[0] for p in parts0]),
                                np.concatenate([p[1] for p in parts0]),
                                (np.linalg.inv(truth[ref0]) @ odom[hist[-1]]).astype(np.float32))
    po = oracle.default_params(max_iterations=ITERS, use_differential=0, num_threads=threads)

    def step(s):
        idx = walk(s + K_MAP + 1)
        hist.append(idx)
        ref, ks, Ts = submap_parts(truth, hist)
        parts = [scans[k] if k == ref else oracle.transform_cloud(T, *scans[k]) for k, T in zip(ks, Ts)]
        refp = np.concatenate([p[0] for p in parts])
        refn = np.concatenate([p[1] for p in parts])
        T0 = (np.linalg.inv(truth[ref]) @ odom[idx]).astype(np.float32) if abs(idx - ref) == 1 else np.eye(4, dtype=np.float32)
        return oracle.icp(scans[idx][0], refp, refn, T0, po)

    for s in range(args.warmup):
        step(s)
    t0 = time.perf_counter()
    for s in range(args.steps):
        step(args.warmup + s)
    dt = time.perf_counter() - t0
    val = args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": wl["metric"],
        "value": val, "unit": "registrations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "pool_scans": POOL},
        "cpu_baseline": {"value": val, "unit": "registrations/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} full registrations (sub-map assembly + kd-tree build + 30 ICP iterations), "
                                   f"query loop OpenMP over {threads} threads (fastest of the counts tried, "
                                   f"{usable_threads()} usable)"},
        "e2e": {"value": val, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_baseline_sample():
    import oracle
    truth, odom, scans = make_pool(0)
    hist = list(range(K_MAP + 1))
    ref, ks, Ts = submap_parts(truth, hist)
    parts = [scans[k] if k == ref else oracle.transform_cloud(T, *scans[k]) for k, T in zip(ks, Ts)]
    refp = np.concatenate([p[0] for p in parts])
    refn = np.concatenate([p[1] for p in parts])
    T0 = (np.linalg.inv(truth[ref]) @ odom[K_MAP]).astype(np.float32)
    threads = best_thread_count(oracle, scans[K_MAP][0], refp, refn, T0)
    out = {}
    for th, reps in ((threads, 4), (1, 1)) if threads > 1 else ((1, 3),):
        po = oracle.default_params(max_iterations=ITERS, use_differential=0, num_threads=th)
        t0 = time.perf_counter()
        for _ in range(reps):
            oracle.icp(scans[K_MAP][0], refp, refn, T0, po)
        out[th] = reps / (time.perf_counter() - t0)
    return {"value": out[threads], "unit": "registrations/s", "cores": threads, "kind": "port",
            "sample": f"oracle port (kd-tree 1-NN + nth_element trim + point-to-plane), 4 full registrations of this workload with the "
                      f"query loop on {threads} OpenMP threads (fastest count, {usable_threads()} usable); "
                      f"single-thread (libpointmatcher default): {out[1]:.3f} registrations/s"}


# IcpStats fields that say how a registration ended.  The timings (device_ms, build_ms, icp_ms) and the spatial-hash
# diagnostics (grid_*) describe how it was computed, not what, so two correct builds may differ in them.
DUMP_STATS = ("iterations", "converged", "max_iter_reached", "last_kept", "last_limit", "used_ratio")


def dump_outputs(out_dir, touts, stats):
    """One registration per track, tracks in order: transforms.npy (B,4,4) float32, the row-major T_ref<-reading each
    registration returned, and one <field>.npy (B,) float64 per DUMP_STATS field of its IcpStats."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "transforms.npy"), np.ascontiguousarray(touts.reshape(-1, 4, 4).transpose(0, 2, 1)))
    for f in DUMP_STATS:
        np.save(os.path.join(out_dir, f"{f}.npy"), np.array([getattr(st, f) for st in stats], np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--tracks", type=int, default=0, help="independent sequences (tracks) hosted per GPU, batched per "
                    "launch (default: 74 for config 2 = 4 of the 296 co-resident CTAs each, 8 for config 5)")
    ap.add_argument("--contexts", type=int, default=1,
                    help="device contexts the tracks of a GPU are split over, each with 1/contexts of the co-resident CTAs "
                         "(experiment: measured on B200, cooperative launches of different contexts do NOT overlap -- 2 contexts "
                         "run at 0.66x -- so the default is 1)")
    ap.add_argument("--config", type=int, default=2, choices=(2, 3, 4, 5),
                    help="BASELINE.json workload: 2 scan-to-map ICP (default, the headline metric), 3 batched trajectories "
                         "feeding the shared estimator, 4 pose-graph solve, 5 dense-sensor stress")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the transforms and ICP stats of the last timed step as DIR/<name>.npy (configs 2 and 5)")
    args = ap.parse_args()
    if args.dump_outputs and (args.config in (3, 4) or args.impl == "reference"):
        ap.error("--dump-outputs records the GPU scan-to-map registrations: --config 2 or 5, --impl ours")
    if args.config == 4:
        import bench_posegraph
        return bench_posegraph.main(args)
    if args.config == 3:
        import bench_trajectory
        return bench_trajectory.main(args)
    wl = select_workload(args.config)
    if args.tracks <= 0:
        args.tracks = wl["tracks"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, wl)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import laser_slam_b200 as ls
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.tracks
    G = max(1, min(args.contexts, B))
    ctxs = [ls.Context(local) for _ in range(G)]
    ctx = ctxs[0]
    if G > 1:
        full = ctx.set_icp_cta_budget(0)
        for c in ctxs:
            c.set_icp_cta_budget(full // G)
    group_of = [t * G // B for t in range(B)]                 # contiguous groups of tracks
    members = [[t for t in range(B) if group_of[t] == g] for g in range(G)]
    # B independent sequences (tracks) per GPU -- the reference's n_laser_slam_workers LaserTracks hosted on one device
    seq_base = int(os.environ.get('LS_BENCH_SEQ_BASE', '0'))   # diagnostic: run another rank's tracks on this one
    # every rank drives the SAME B synthetic sequences: per-GPU work is then identical by construction (the cost of a
    # registration varies by +-25 % with where along the street the vehicle is), which is what weak scaling assumes
    tracks = make_pools([seq_base + t for t in range(B)])
    prm = ls.default_params(max_iterations=ITERS, use_differential=0)
    feats = [[torch.from_numpy(s[0]).pin_memory() for s in tr[2]] for tr in tracks]   # pinned host staging
    nrms = [[torch.from_numpy(s[1]).pin_memory() for s in tr[2]] for tr in tracks]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from laser_slam_b200 import dist as lsd
    exchange = lsd.Exchange(rank, world, device=None if os.environ.get('LS_BENCH_NO_COMM') else local)   # ls_comm_* (one ncclAllGather of 32 B/rank) when world > 1

    xmode = os.environ.get("LS_BENCH_EXCHANGE", "split")   # split | blocking | none (diagnostic)

    def share_pose_delta(T):
        """One 32-byte {delta[6], status, key} record per rank per step (SURVEY.md §8e).  Split-phase: the records
        of step s are collected when step s+1 posts its own (the estimator consumes factors asynchronously)."""
        if world > 1 and xmode != "none":
            rec = lsd.pose_record(T, status=0, key=rank)
            if xmode == "blocking":
                exchange.allgather(rec)
            else:
                exchange.collect()
                exchange.post(rec)

    n_total = args.warmup + args.steps

    def stage_track(t, n_steps):
        """Per-step arguments of track t (sub-map scans, their float32 transforms, initial guess): what
        LaserTrack::localScanToSubMap hands to the ICP.  Staged before the clock starts."""
        truth, odom, _ = tracks[t]
        h = [walk(s) for s in range(K_MAP + 1)]
        out = []
        for s in range(n_steps):
            idx = walk(s + K_MAP + 1)
            h.append(idx)
            ref, ks, Ts = submap_parts(truth, h)
            T0 = (np.linalg.inv(truth[ref]) @ odom[idx]).astype(np.float32) if abs(idx - ref) == 1 else np.eye(4, dtype=np.float32)
            out.append((idx, ref, ks, Ts, T0))
        return out

    staged = [stage_track(t, n_total + 1) for t in range(B)]   # one step of look-ahead for the pipelined uploads

    # ------------------------------------------------------------------ resident arm (value)
    # Every group of tracks lives in its own context (own ring, own workspaces).  A step registers the next scan of every
    # track: group g's launch is begun, then the previous launch of the NEXT group is collected and begun again, ... so that
    # while one group iterates, the other's sub-maps are assembled and indexed.
    mps = [ctxs[g].create_map(len(members[g]) * POOL + 2, N_SCAN) for g in range(G)]
    sid = [None] * B
    for t in range(B):
        sid[t] = [mps[group_of[t]].push_scan_raw(feats[t][k].data_ptr(), nrms[t][k].data_ptr(), 3, N_SCAN) for k in range(POOL)]
    prepared = [[] for _ in range(G)]
    for s in range(n_total):
        for g in range(G):
            probs = [(sid[t][staged[t][s][0]], [sid[t][k] for k in staged[t][s][2]], staged[t][s][3], staged[t][s][4]) for t in members[g]]
            prepared[g].append(mps[g].prepare_begin_batch(probs, prm))
    dev_ms, icp_ms = [], []
    last_touts = [None] * G
    last_stats = [None] * G

    def finish(g, s, record):
        rc, statuses, touts, stats = prepared[g][s][1]()
        if rc != 0 or statuses.any():
            raise RuntimeError(f"registration failed rc={rc} {list(statuses)}")
        last_touts[g] = touts.copy()
        last_stats[g] = stats   # every prepared step owns its stats array: a reference is enough
        if world > 1 and g == 0:
            share_pose_delta(ls.from_colmajor(touts[0]))
        if record:
            dev_ms.append(max(st.device_ms for st in stats))
            icp_ms.append(stats[0].icp_ms)
            if os.environ.get("LS_BENCH_TRACE"):
                print(f"[trace] step {s} group {g}: icp {stats[0].icp_ms:.2f} ms; per track last_limit " +
                      " ".join(f"{st.last_limit:.4f}" for st in stats) + " kept " + " ".join(str(st.last_kept) for st in stats),
                      file=sys.stderr, flush=True)

    def run_resident(s0, n, record):
        inflight = [None] * G
        for s in range(s0, s0 + n):
            for g in range(G):
                if inflight[g] is not None:
                    finish(g, inflight[g], record)
                prepared[g][s][0]()          # stage + launch, returns at once
                inflight[g] = s
        for g in range(G):
            if inflight[g] is not None:
                finish(g, inflight[g], record)

    run_resident(0, args.warmup, False)
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = sum(c.launch_count for c in ctxs)
    barrier()
    t0 = time.perf_counter()
    run_resident(args.warmup, args.steps, True)
    exchange.collect()   # the last step's records, inside the timed region
    barrier()
    t_res = time.perf_counter() - t0
    launches = sum(c.launch_count for c in ctxs) - launches0
    idx, ref = staged[0][n_total - 1][0], staged[0][n_total - 1][1]
    truth_rel = np.linalg.inv(tracks[0][0][ref]) @ tracks[0][0][idx]
    pose_err = float(np.abs(ls.from_colmajor(last_touts[0][0])[:3, 3] - truth_rel[:3, 3]).max())

    # parity of what was just timed, outside the clock: one problem of the last batched step against the oracle
    parity = None
    if rank == 0:
        import oracle
        tchk = (n_total - 1) % B
        idx_c, ref_c, ks_c, Ts_c, T0_c = staged[tchk][n_total - 1]
        sc = tracks[tchk][2]
        parts_c = [sc[k] if k == ref_c else oracle.transform_cloud(T, *sc[k]) for k, T in zip(ks_c, Ts_c)]
        r = oracle.icp(sc[idx_c][0], np.concatenate([p_[0] for p_ in parts_c]), np.concatenate([p_[1] for p_ in parts_c]), T0_c,
                       oracle.default_params(max_iterations=ITERS, use_differential=0, num_threads=usable_threads()))
        got = ls.from_colmajor(last_touts[group_of[tchk]][members[group_of[tchk]].index(tchk)])
        parity = {"problem": f"track {tchk}, last timed step ({len(members[group_of[tchk]])} registrations in that launch)",
                  "final_transform_bit_equal_to_oracle": bool(np.array_equal(got, r["T"])),
                  "max_abs_diff": float(np.abs(got - r["T"]).max())}
        if not parity["final_transform_bit_equal_to_oracle"]:
            raise RuntimeError(f"bench: the timed batched launch disagrees with the oracle: {parity}")

    # single-stream latency (one track, one registration per launch), a few steps
    lat = []
    for s in range(min(20, n_total)):
        g = mps[0].register(sid[0][staged[0][s][0]], [sid[0][k] for k in staged[0][s][2]], staged[0][s][3], staged[0][s][4], prm)
        lat.append(g["stats"].device_ms)
    single_ms = float(np.median(lat))

    # ------------------------------------------------------------------ end-to-end arm (host buffers)
    # every step uploads the new scan of every track from pinned host memory, then registers the batch
    mp2 = [ctxs[g].create_map(len(members[g]) * (2 * K_MAP + 8), N_SCAN) for g in range(G)]   # rings: every track keeps its last K_MAP+1 scans resident with slack
    sid2 = [dict() for _ in range(B)]
    for t in range(B):
        for s in range(K_MAP + 1):
            k = walk(s)
            sid2[t][k] = mp2[group_of[t]].push_scan_raw(feats[t][k].data_ptr(), nrms[t][k].data_ptr(), 3, N_SCAN)

    # Uploads are double-buffered: while step s is registered, the scans of step s+1 go up on the map's own stream
    # (ls_map_push_scan_async; the sensor delivers the next scan while the current one is being registered).  Every
    # timed step still issues one full set of uploads and reads its results back.
    def upload(g, s):
        for t in members[g]:
            idx = staged[t][s][0]
            sid2[t][idx] = mp2[g].push_scan_raw_async(feats[t][idx].data_ptr(), nrms[t][idx].data_ptr(), 3, N_SCAN)   # H2D, pinned

    def begin_e2e(g, s):
        probs = []
        for t in members[g]:
            idx, ref, ks, Ts, T0 = staged[t][s]
            probs.append((sid2[t][idx], [sid2[t][k] for k in ks], Ts, T0))
        end = mp2[g].begin_batch(probs, prm)   # stage + launch step s of this group, returns at once
        upload(g, s + 1)   # new ids land in ring slots last used >= K_MAP+1 steps ago (the library refuses anything else)
        return end

    def run_e2e(s0, n):
        inflight = [None] * G
        for s in range(s0, s0 + n):
            for g in range(G):
                if inflight[g] is not None:
                    out = inflight[g]()                                                              # wait; D2H of T + stats
                    if world > 1 and g == 0:
                        share_pose_delta(out[0]["T"])
                inflight[g] = begin_e2e(g, s)
        for g in range(G):
            if inflight[g] is not None:
                out = inflight[g]()
                if world > 1 and g == 0:
                    share_pose_delta(out[0]["T"])

    for g in range(G):
        upload(g, 0)
    run_e2e(0, args.warmup)
    barrier()
    t0 = time.perf_counter()
    run_e2e(args.warmup, args.steps)
    exchange.collect()
    barrier()
    t_e2e = time.perf_counter() - t0
    clocks = sampler.summary()

    # ------------------------------------------------------------------ the same through the C++ host layer
    # laser_slam::IncrementalEstimator::processPosesAndLaserScans (libls_host.so): what laser_slam_ros would call.  Host
    # clouds arrive as DataPoints (pageable std::vector storage, copied into the track as the reference does), every
    # track's scan is uploaded by LaserTrack::residentScan and the B registrations of a step run as one batched launch.
    host_arm = None
    if not os.environ.get("LS_BENCH_NO_HOST_ARM"):
        import tempfile
        from laser_slam_b200 import host as lsh
        with tempfile.NamedTemporaryFile("w", suffix=".yaml", delete=False) as f:
            f.write("matcher:\n  KDTreeMatcher:\n    knn: 1\noutlierFilters:\n  - TrimmedDistOutlierFilter:\n      ratio: 0.75\n"
                    "errorMinimizer:\n  PointToPlaneErrorMinimizer\ntransformationCheckers:\n  - CounterTransformationChecker:\n"
                    f"      maxIterationCount: {ITERS}\n")
            yaml_path = f.name
        est = lsh.Estimator(n_workers=B, nscan_in_sub_map=K_MAP, use_icp_factors=True, use_odom_factors=True, robust_icp=True,
                            device=local, icp_yaml_path=yaml_path)

        def pose7(T):
            q = np.empty(4)
            R = T[:3, :3]
            q[0] = 0.5 * np.sqrt(max(1e-12, 1.0 + np.trace(R)))
            q[1:] = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]]) / (4.0 * q[0])
            return np.concatenate([q / np.linalg.norm(q), T[:3, 3]])

        def host_args(s):
            idxs = [walk(s) for _ in range(B)]
            return (list(range(B)), [s * 100_000_000] * B, [feats[t][idxs[t]].data_ptr() for t in range(B)],
                    [nrms[t][idxs[t]].data_ptr() for t in range(B)], [N_SCAN] * B), [pose7(tracks[t][1][idxs[t]]) for t in range(B)]

        # the same scans as the C-ABI arm's timed steps: its step s registers scan walk(s + K_MAP + 1)
        n_host = args.steps
        w_host = args.warmup + K_MAP + 1
        hargs = [host_args(s) for s in range(w_host + n_host + 1)]   # marshalled before the clock, like the C-ABI arm's

        def run_host(s0, n):
            """Step s: begin (stage + launch), prefetch step s+1's scans while it runs, end."""
            out = None
            for s in range(s0, s0 + n):
                (wk, tm, fp, npp, ns), poses = hargs[s]
                est.begin_batch(wk, tm, poses, fp, npp, ns, views=True)
                (wk2, tm2, fp2, np2, ns2), _ = hargs[s + 1]
                est.prefetch(wk2, tm2, fp2, np2, ns2, views=True)
                out = est.end_batch(with_estimator=False)
            return out

        run_host(0, w_host)
        barrier()
        t0 = time.perf_counter()
        icp7, hstats = run_host(w_host, n_host)
        barrier()
        t_host = time.perf_counter() - t0
        t_host, = lsd.max_over_ranks([t_host], device=local)
        host_arm = {"value": world * B * n_host / t_host, "unit": "registrations/s", "steps": n_host,
                    "api": "laser_slam::IncrementalEstimator::processPosesAndLaserScans over libls_host.so: DataPoints in "
                           "(views of the same pinned host buffers the C-ABI arm reads, no copy), RelativePose out; "
                           "beginPosesAndLaserScans / prefetchLaserScans(next step) / endPosesAndLaserScans, so the next "
                           "step's uploads overlap this step's launch, as in the C-ABI arm",
                    "iterations": int(hstats[0].iterations)}
        est.close()
        os.unlink(yaml_path)

    # ------------------------------------------------------------------ reduce over ranks (max time)
    t_res, t_e2e = lsd.max_over_ranks([t_res, t_e2e], device=local)
    exchange.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = load_peaks()
    t_icp = float(np.mean(icp_ms)) * 1e-3
    t_dev = float(np.mean(dev_ms)) * 1e-3
    # ncu DRAM bytes of one launch of the same shape (8 registrations per launch has its own capture: eight maps do
    # not fit L2 together, one does)
    traffic, traffic_note = None, None
    import glob
    import re
    caps = {}
    for prof in glob.glob(os.path.join(ROOT, "profiles", f"r2_icp_kernel_cfg{args.config}_batch*_summary.json")):
        m = re.search(r"_batch(\d+)_summary", prof)
        if m:
            caps[int(m.group(1))] = prof
    if caps:
        regs = min(caps, key=lambda r: (abs(r - B // G), -r))   # the capture closest in shape to what was timed
        try:
            per_launch = float(json.load(open(caps[regs])).get("dram_bytes_per_launch"))
            fname = os.path.basename(caps[regs])
            if regs == B // G:
                traffic = per_launch
                traffic_note = f"ncu dram__bytes_read+write of one launch with {regs} registration(s) (profiles/{fname})"
            else:
                traffic = per_launch * (B // G) / regs
                traffic_note = (f"no ncu capture with {B // G} registrations per launch: scaled per registration from the capture with "
                                f"{regs} per launch (profiles/{fname}: {per_launch / 1e9:.2f} GB for {regs}); the working sets "
                                "of > 3 registrations already exceed L2, so DRAM bytes per registration are flat from there on")
        except Exception:
            traffic, traffic_note = None, None
    Bg = B / G   # registrations per launch
    t_step = t_res / args.steps
    # G launches (one per context, B/G registrations and 1/G of the co-resident CTAs each) run side by side, so the device-level
    # figure is the algorithmic bytes of ALL launches of a step over the step's duration; the per-launch figure (bytes of one
    # launch over its own CUDA-event duration, during which it holds 1/G of the SM slots) is given next to it.
    roof = {"bound": "hbm", "kernel": f"ls::icp_kernel (persistent: NN query + trimmed select + normal equations, {ITERS} iterations, "
                                      f"{Bg:.0f} registrations per launch, {G} launches side by side)",
            "achieved": B * ALG_BYTES_ICP / t_step / 1e9, "peak": peak, "unit": "GB/s",
            "frac": B * ALG_BYTES_ICP / t_step / 1e9 / peak,
            "traffic": traffic, "traffic_note": traffic_note,
            "peak_source": peak_src, "algorithmic_bytes_per_step": B * ALG_BYTES_ICP, "step_ms": t_step * 1e3,
            "per_launch": {"registrations": Bg, "algorithmic_bytes": Bg * ALG_BYTES_ICP, "kernel_ms": t_icp * 1e3,
                           "achieved": Bg * ALG_BYTES_ICP / t_icp / 1e9, "sm_share": 1.0 / G,
                           "frac_of_peak": Bg * ALG_BYTES_ICP / t_icp / 1e9 / peak},
            "kernel_ms": t_icp * 1e3,
            "registration": {"algorithmic_bytes": ALG_BYTES_REG, "device_ms_per_batch": t_dev * 1e3,
                             "achieved": B * ALG_BYTES_REG / t_step / 1e9, "frac": B * ALG_BYTES_REG / t_step / 1e9 / peak}}
    cpu = cpu_baseline_sample() if args.gpus == 1 and not os.environ.get('LS_BENCH_NO_CPU') else None
    out = {
        "metric": wl["metric"],
        "value": world * B * args.steps / t_res, "unit": "registrations/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_res / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"],
                   "tracks_per_gpu": B, "registrations_per_step": world * B,
                   "contexts_per_gpu": G,
                   "concurrency": f"{B} independent sequences (tracks) per GPU (the same {B} synthetic sequences on every rank, so "
                                  f"per-GPU work is identical) in {G} groups, one device context each; one step registers the "
                                  f"next scan of every track, one cooperative launch per group (ls_icp_register_submap_batch_begin/"
                                  f"_end), the groups' launches overlapping",
                   "single_stream_ms_per_registration": single_ms,
                   "l2": f"inputs larger than L2: {B * POOL} resident scans/rank cycled ({B * POOL * N_SCAN * 32 / 1e6:.0f} MB) "
                         f"+ {B} x ~170 MB workspaces",
                   "collective": "none on the data path; one 32 B/rank NCCL all-gather of pose records per step when n_gpus > 1",
                   "final_pose_err_vs_truth_m": pose_err, "parity_check": parity},
        "e2e": {"value": world * B * args.steps / t_e2e, "unit": "registrations/s",
                "h2d_bytes_per_step": B * (N_SCAN * 16 + N_SCAN * 12 + 16 * 4 * (K_MAP + 1) + 8 * (K_MAP + 1)),
                "d2h_bytes_per_step": B * (216 + 212),   # per registration: result block of the ICP scratch + grid header
                "pipeline": "the scans of step s+1 are uploaded (ls_map_push_scan_async, own stream) while step s is "
                            "registered; every timed step issues one full set of uploads and reads its results back",
                "host_layer": host_arm},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
    }
    if cpu:
        out["cpu_baseline"] = cpu
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.concatenate(last_touts), [st for g in range(G) for st in last_stats[g]])
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
