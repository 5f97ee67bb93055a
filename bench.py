#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native association engine.

Metric (BASELINE.json): pair-associations/s of BatchVisualSORT on 256 scenes x 512 tracks x 512 detections x 512-dim
features (cfg5), one `predict` per step.  pair-associations = sum over scenes of N_s * M_s per frame.

  value : device-timed throughput, inputs already resident in HBM (sb200_predict_batch_device)
  e2e   : the same metric through the host-pointer C-ABI call (sb200_predict_batch): pinned host inputs, H2D inside
          the timed region, result ids / voting types / epochs / lengths copied back
  roofline      : the visual cost-matrix kernel (dominant cost kernel), timed live with CUDA events on its stream
  cpu_baseline  : the CPU oracle (port of the reference's algorithm, all host cores) on a bounded sample

`--impl reference` times the reference's algorithm (the oracle port; the Rust reference cannot be built in this
image) on the host cores for the same config and prints the same JSON line with "impl": "reference".

Launch: python bench.py --gpus N --steps K --warmup W   (N > 1 under torch.distributed.run, one rank per GPU;
scenes are sharded by rank -- weak scaling, per-GPU work fixed -- and the assigned track ids are gathered with NCCL).

`--dump-outputs DIR` writes what the timed path returned for the last timed frame as DIR/<name>.npy (rank 0's shard):
ids, epochs, lengths, voting_types of the device-pointer path and predicted_boxes, observed_boxes of the host-pointer
path (with --impl reference: the oracle's ids, epochs, lengths, voting_types).  The frames are seeded, so two builds run
with the same arguments can be compared array for array.
"""
from __future__ import annotations

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

METRIC = "pair_associations_per_sec"
UNIT = "pair-associations/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg5")
    ap.add_argument("--scenes", type=int, default=0, help="override the scene count (debug)")
    ap.add_argument("--cpu-sample-scenes", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--visual-threshold", default=None,
                    help="override the visual metric's threshold: a float, or 'max' = the reference's default Euclidean(f32::MAX)")
    ap.add_argument("--feat-noise", type=float, default=None, help="override the workload's feature noise (sensitivity sweeps)")
    ap.add_argument("--no-scatter", action="store_true", help="N > 1: skip the ingest-rank scatter arm (sb200_shard_*)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays):
    """Writes the per-detection arrays of one frame as out_dir/<name>.npy: float64 where float32 could not hold every
    value (ids, epochs, lengths), float32 otherwise.  When they would exceed DUMP_LIMIT_BYTES, a fixed, seeded sample of
    the detections is written instead -- the same rows of every array, their indices in rows.npy."""
    def as_float(a):
        a = np.asarray(a)
        return a.astype(np.float64 if a.dtype.kind in "iu" and a.dtype.itemsize >= 4 else np.float32)

    arrays = {k: as_float(a) for k, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, (DUMP_LIMIT_BYTES - 4096) // (row_bytes + 8), replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def config_dict(name, cfg, extra=None):
    d = {
        "workload": f"{name}: {cfg.name}",
        "scenes_per_gpu": cfg.n_scenes,
        "tracks_per_scene": cfg.n_objects,
        "detections_per_scene": f"~{int(cfg.n_objects * 0.95)} (5% dropped, 5% fresh identities per frame)",
        "feature_dim": cfg.feature_dim,
        "visual_max_observations": 3,
        "oriented_boxes": cfg.oriented,
        "l2": "per-step inputs exceed L2 (features %.0f MB/step)" % (cfg.n_scenes * cfg.n_objects * max(cfg.feature_dim, 6) * 4 / 1e6),
        "parallelism": "scene-sharded, one process per GPU",
        "units": "pair-associations = sum over scenes of M detections x N stored tracks that can still match "
                 "(expired tracks awaiting collection are not counted)",
    }
    if extra:
        d.update(extra)
    return d


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons while the timed region runs.  Sampled in-process through NVML (a query costs
    microseconds and holds no driver lock the compute path needs); falls back to forking nvidia-smi at 2 Hz when the
    NVML binding is missing.  Round 1 forked nvidia-smi at 10 Hz from every rank, which slowed the host-bound loop down."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.source = "nvml"
        self.times = []          # perf_counter of every sample
        self.call_ms = []        # host cost of every query
        self.window = [None, None]
        self._halt = threading.Event()
        self._h = None
        try:
            import pynvml

            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES remaps ordinals: resolve through the PCI bus id of the torch device
            import torch

            prop = torch.cuda.get_device_properties(index)
            bdf = "%08x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByPciBusId(bdf.encode())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None
            self.source = "nvidia-smi"

    def _sample_nvml(self):
        nv = self._nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        try:
            r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
        except Exception:
            r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
        for bit, nm in self.REASONS.items():
            if r & bit:
                self.reasons.add(nm)

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip().split(",")
        self.samples.append(float(out[0]))
        self.max_mhz = float(out[1])
        for nm, v in zip(names, out[2:]):
            if "Active" in v and "Not" not in v:
                self.reasons.add(nm)

    def run(self):
        while not self._halt.is_set():
            t0 = time.perf_counter()
            try:
                n0 = len(self.samples)
                if self._h is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
                if len(self.samples) > n0:
                    self.times.append(t0)
                    self.call_ms.append(1e3 * (time.perf_counter() - t0))
            except Exception:
                pass
            self._halt.wait(0.005 if self._h is not None else 0.5)

    def mark_begin(self):
        self.window[0] = time.perf_counter()

    def mark_end(self):
        self.window[1] = time.perf_counter()

    def stop(self):
        """Median SM clock over the samples taken under load: the warm-up steps (same kernels, same clocks) and the
        timed region; `samples_in_timed_region` says how many fell between the two marks."""
        self._halt.set()
        self.join(timeout=5)
        med = float(np.median(self.samples)) if self.samples else None
        inside = 0
        if self.window[0] is not None and self.window[1] is not None:
            inside = sum(1 for t in self.times if self.window[0] <= t <= self.window[1])
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples),
                "samples_in_timed_region": inside, "source": self.source,
                "query_ms_max": max(self.call_ms) if self.call_ms else None}


def usable_cores():
    """Host threads the CPU legs may really use: min(cpu_count, scheduler affinity, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:   # cgroup v2: "max 100000" or "<quota> <period>"; cgroup v1: cpu.cfs_quota_us / cpu.cfs_period_us (-1 == none)
        if os.path.exists("/sys/fs/cgroup/cpu.max"):
            q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
            if q != "max":
                n = min(n, max(1, int(float(q) / float(p))))
        else:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and p > 0:
                n = min(n, max(1, q // p))
    except Exception:
        pass
    return max(1, n)


def bind_near_gpu(local):
    """Pins this process to the CPUs of the GPU's NUMA node before the pinned host buffers are allocated (first touch
    puts them on that node), so the H2D copies of the e2e arm do not cross the socket interconnect.  Returns a short
    description and the previous affinity (restored before the CPU baseline, which wants every core)."""
    try:
        import torch

        prop = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return "numa node unknown", None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        old = os.sched_getaffinity(0)
        cpus &= old
        if not cpus:
            return f"numa node {node}: no usable cpu", None
        os.sched_setaffinity(0, cpus)
        return f"numa node {node} of GPU {bdf} ({len(cpus)} cpus)", old
    except Exception as e:   # no sysfs / restricted container: run unpinned
        return f"unpinned ({type(e).__name__})", None


def make_frames(name, n_frames, scene_base, n_scenes_override=0, feat_noise=None):
    import dataclasses

    from similari_b200.workload import CONFIGS, Workload

    cfg = CONFIGS[name]
    if n_scenes_override:
        cfg = dataclasses.replace(cfg, n_scenes=n_scenes_override)
    if feat_noise is not None:
        cfg = dataclasses.replace(cfg, feat_noise=feat_noise)
    cfg = dataclasses.replace(cfg, seed=cfg.seed + 7919 * scene_base)
    wl = Workload(cfg, scene_base=scene_base)
    return cfg, [wl.next_frame() for _ in range(n_frames)]


def option_overrides(args):
    """Tracker option overrides of the command line (same for the GPU arm and the CPU arms)."""
    over = {}
    if args.visual_threshold is not None:
        over["visual_threshold"] = 3.402823466e38 if args.visual_threshold == "max" else float(args.visual_threshold)
    return over


def cpu_port_run(name, frames, warm, steps, threads, over=None):
    """Times the oracle tracker (reference algorithm, reference execution order, `threads` host threads).  Returns the
    pair-associations and seconds of the timed frames and the result of the last frame."""
    import oracle as orc
    from similari_b200.workload import tracker_options_for

    opts = tracker_options_for(name, orc.make_options, **(over or {}))
    t = orc.Tracker(opts, threads=threads)
    units, secs, last = 0, 0.0, None

    def live_tracks(scene):
        # N of the metric = stored tracks that can still match (the reference keeps expired tracks in its store until
        # its next auto-waste tick and rejects them pair by pair in `compatible`; they are not counted as work)
        stored = len(t.scene_tracks(scene, cap=1 << 14)["ids"])
        idle = t.idle_tracks(scene, cap=1 << 14)["epochs"].astype(np.int64)
        return stored - int((idle + int(opts.max_idle_epochs) < int(t.current_epoch(scene))).sum())

    for i, f in enumerate(frames[: warm + steps]):
        m = np.diff(f["det_offsets"]).astype(np.int64)
        n_before = np.array([live_tracks(int(s)) for s in f["scene_ids"]], dtype=np.int64) if i >= warm else None
        t0 = time.perf_counter()
        last = t.predict_batch(f["scene_ids"], f["det_offsets"], f["boxes"], features=f["features"], want_boxes=False)
        dt = time.perf_counter() - t0
        if i >= warm:
            units += int((m * n_before).sum())
            secs += dt
    return units, secs, last


def run_reference(args):
    """The reference arm: the reference's algorithm (the C++ oracle port -- no Rust toolchain in this image) on the host
    cores, SAME config, SAME step count as the GPU arm by default (all scenes; the oracle does a 256-scene cfg5 frame in
    ~2 s on 16 threads); --cpu-sample-scenes bounds it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle as orc

    orc.build()
    cores = usable_cores()
    from similari_b200.workload import CONFIGS

    full = CONFIGS[args.config].n_scenes
    sample_scenes = min(args.cpu_sample_scenes or full, full)
    warm = max(3, args.warmup)
    steps = args.steps
    cfg, frames = make_frames(args.config, warm + steps, 0, sample_scenes, feat_noise=args.feat_noise)
    units, secs, last = cpu_port_run(args.config, frames, warm, steps, cores, option_overrides(args))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: last[k] for k in ("ids", "epochs", "lengths", "voting_types")})
    value = units / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * secs / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.config, cfg, {"note": "the whole workload" if sample_scenes == full else
                                                 "bounded sample of the full workload: same per-scene shape"}),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample_scenes} of {full} scenes, {steps} timed frame(s) "
                                   f"after {warm} warm-up frames, {cores} threads (scene-parallel)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def newest_traffic():
    """DRAM bytes per launch of the dominant kernel from the newest ncu --set full capture under profiles/."""
    import glob

    best = None
    for fn in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_dominant_kernel_traffic*.json"))):
        try:
            best = (fn, json.load(open(fn)))
        except Exception:
            pass
    return best


def run_scatter_arm(eng, torch, dist, new_tracker, frames, dboxes, dfeats, W, K, D, visual, max_total, rank, world, local,
                    ids_ref_last):
    """N > 1: the request enters on ONE rank.  Rank 0 holds the detections of all shards; every step it scatters them to the
    ranks that own the scenes (sb200_shard_scatter: ncclSend/ncclRecv grouped, on a side stream, one frame ahead of the
    kernels) and gathers the assigned track records back (sb200_shard_gather) -- the exchange step of the sharded path
    inside the library.  Same frames as the local-ingest arm, so every rank's ids must equal that arm's."""
    dev = torch.device("cuda", local)
    uid = [eng.Comm.unique_id() if rank == 0 else None, eng.Comm.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    c_sc = eng.Comm(rank, world, uid[0], local)     # scatter traffic (side stream)
    c_ga = eng.Comm(rank, world, uid[1], local)     # gather traffic (compute stream)
    # untimed set-up: rank 0 collects the timed frames of every shard (what an ingest node would have received)
    totals = torch.zeros(world, K, dtype=torch.int64, device=dev)
    mine_tot = torch.tensor([len(frames[W + j]["boxes"]) for j in range(K)], dtype=torch.int64, device=dev)
    tl = [torch.zeros(K, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(tl, mine_tot)
    totals = torch.stack(tl).cpu().numpy()          # [world][K]
    all_boxes, all_feats, ranges = [], [], []
    for j in range(K):
        pad_b = torch.zeros(max_total, 6, dtype=torch.float32, device=dev)
        pad_b[: len(frames[W + j]["boxes"])] = dboxes[W + j]
        gb = [torch.empty_like(pad_b) for _ in range(world)] if rank == 0 else None
        dist.gather(pad_b, gb, dst=0)
        gf = None
        if visual:
            pad_f = torch.zeros(max_total, D, dtype=torch.float32, device=dev)
            pad_f[: len(frames[W + j]["boxes"])] = dfeats[W + j]
            gf = [torch.empty_like(pad_f) for _ in range(world)] if rank == 0 else None
            dist.gather(pad_f, gf, dst=0)
            del pad_f
        rng = np.concatenate([[0], np.cumsum(totals[:, j])]).astype(np.int32)
        ranges.append(rng)
        if rank == 0:
            all_boxes.append(torch.cat([gb[r][: totals[r, j]] for r in range(world)]).contiguous())
            all_feats.append(torch.cat([gf[r][: totals[r, j]] for r in range(world)]).contiguous() if visual else None)
        del gb, gf
    torch.cuda.synchronize()
    t = new_tracker()
    d_out = {"ids": torch.zeros(max_total, dtype=torch.int64, device=dev), "epochs": torch.zeros(max_total, dtype=torch.int32, device=dev),
             "lengths": torch.zeros(max_total, dtype=torch.int32, device=dev), "voting_types": torch.zeros(max_total, dtype=torch.uint8, device=dev)}
    all_out = None
    if rank == 0:
        n_all = int(max(r[-1] for r in ranges))
        all_out = {"ids": torch.zeros(n_all, dtype=torch.int64, device=dev), "epochs": torch.zeros(n_all, dtype=torch.int32, device=dev),
                   "lengths": torch.zeros(n_all, dtype=torch.int32, device=dev), "voting_types": torch.zeros(n_all, dtype=torch.uint8, device=dev)}
    rb = [torch.zeros(max_total, 6, dtype=torch.float32, device=dev) for _ in range(2)]
    rf = [torch.zeros(max_total, D, dtype=torch.float32, device=dev) if visual else None for _ in range(2)]
    main = torch.cuda.current_stream()
    side = torch.cuda.Stream(device=dev)
    landed = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [None, None]

    def addr(d):
        return {k: v.data_ptr() for k, v in d.items()} if d is not None else None

    def scatter(j):
        b = j & 1
        with torch.cuda.stream(side):
            if consumed[b] is not None:
                side.wait_event(consumed[b])
            c_sc.scatter(0, ranges[j], D, all_boxes[j].data_ptr() if rank == 0 else 0,
                         all_feats[j].data_ptr() if (rank == 0 and visual) else 0, rb[b].data_ptr(),
                         rf[b].data_ptr() if visual else 0, side.cuda_stream)
            landed[b].record(side)

    for i in range(W):   # warm-up on the local copies (identical data)
        f = frames[i]
        t.predict_batch_device(f["scene_ids"], f["det_offsets"], dboxes[i].data_ptr(), dfeats[i].data_ptr() if visual else 0,
                               d_ids=d_out["ids"].data_ptr(), d_epochs=d_out["epochs"].data_ptr(),
                               d_lengths=d_out["lengths"].data_ptr(), d_voting_types=d_out["voting_types"].data_ptr())
    t.sync()
    # NCCL sets up its peer-to-peer channels on a communicator's first operation (tens of milliseconds): one untimed
    # scatter and gather first
    scatter(0)
    main.wait_event(landed[0])
    c_ga.gather(0, ranges[0], addr(d_out), addr(all_out), main.cuda_stream)
    torch.cuda.synchronize()
    # scatter alone (K back-to-back scatters, nothing else running): what the exchange costs
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(side)
    for j in range(K):
        scatter(j)
    e1.record(side)
    dist.barrier()
    torch.cuda.synchronize()
    scatter_only_ms = e0.elapsed_time(e1) / K
    consumed[0] = consumed[1] = None
    # timed: scatter of frame j+1 overlaps the kernels of frame j
    dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    scatter(0)
    for j in range(K):
        b = j & 1
        if j + 1 < K:
            scatter(j + 1)
        f = frames[W + j]
        main.wait_event(landed[b])
        t.predict_batch_device(f["scene_ids"], f["det_offsets"], rb[b].data_ptr(), rf[b].data_ptr() if visual else 0,
                               d_ids=d_out["ids"].data_ptr(), d_epochs=d_out["epochs"].data_ptr(),
                               d_lengths=d_out["lengths"].data_ptr(), d_voting_types=d_out["voting_types"].data_ptr())
        ev = torch.cuda.Event()
        ev.record(main)
        consumed[b] = ev
        c_ga.gather(0, ranges[j], addr(d_out), addr(all_out), main.cuda_stream)
    ev1.record()
    dist.barrier()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    t.sync()
    n_last = len(frames[W + K - 1]["boxes"])
    ok = bool(np.array_equal(d_out["ids"][:n_last].cpu().numpy().astype(np.uint64), ids_ref_last))
    if rank == 0:
        r0 = ranges[K - 1]
        ok = ok and bool(np.array_equal(all_out["ids"][r0[0]:r0[1]].cpu().numpy().astype(np.uint64), ids_ref_last))
    t.close()
    c_sc.close()
    c_ga.close()
    tm = torch.tensor([ms, scatter_only_ms, 0.0 if ok else 1.0], dtype=torch.float64, device=dev)
    dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    bytes_root = float(np.mean([(r[-1] - r[1]) * (24 + (D * 4 if visual else 0)) for r in ranges]))
    return {"ms_per_step": float(tm[0]) / K, "scatter_only_ms_per_step": float(tm[1]),
            "bytes_sent_by_the_ingest_rank_per_step": bytes_root, "ids_identical_to_local_ingest": float(tm[2]) == 0.0,
            "ingest_rank_egress_gbs": bytes_root / (float(tm[1]) * 1e-3) / 1e9 if float(tm[1]) > 0 else None,
            "how": "rank 0 holds every shard's detections; per step sb200_shard_scatter (ncclSend/Recv in one group, side "
                   "stream, one frame ahead) + sb200_predict_batch_device + sb200_shard_gather of ids / epochs / lengths / "
                   "voting types to rank 0"}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} != WORLD_SIZE {world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    affinity_note, old_affinity = ("disabled", None) if os.environ.get("SB200_BENCH_NUMA") == "0" else bind_near_gpu(local)

    import similari_b200.engine as eng
    from similari_b200._lib import default_options, pinned_empty
    from similari_b200.workload import CONFIGS, tracker_options_for

    name = args.config
    W, K = max(args.warmup, 3), args.steps
    base_cfg = CONFIGS[name]
    n_sc = args.scenes or base_cfg.n_scenes
    over = option_overrides(args)
    # one extra frame: the e2e loop prefetches frame i+1 while frame i computes, so K timed steps issue K copies
    cfg, frames = make_frames(name, W + K + 1, scene_base=rank * n_sc, n_scenes_override=args.scenes,
                              feat_noise=args.feat_noise)
    D = cfg.feature_dim
    visual = D > 0

    # capacity hint: with frames in flight the store is sized for upper bounds (every queued detection may become a track).
    # A threshold that cuts nothing (--visual-threshold max / 10.0) also creates ~1.6 x the tracks of the headline metric;
    # with 4 x it sat at the edge of a store regrow (8 GB of feature arena reallocated inside the timed region when the
    # ring happened to be full), so those runs get 8 x.
    tracks_hint = (8 if args.visual_threshold is not None else 4) * cfg.n_objects

    def new_tracker():
        t = eng.Tracker(tracker_options_for(name, default_options, device=local, max_scenes_hint=cfg.n_scenes,
                                            max_tracks_per_scene_hint=tracks_hint,
                                            max_dets_per_scene_hint=cfg.n_objects, **over))
        t.set_stream(torch.cuda.current_stream().cuda_stream)
        return t

    def timed_region_begin():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- e2e: host pointers (pinned), H2D + D2H timed
    # The call a user of the reference makes: BatchVisualSort.predict(batch) -> per-detection SortTrack records.
    # sb200_predict_batch_async is that call (asynchronous like the reference's, results behind sb200_sync); each timed
    # step copies its whole request host -> device and its whole result (ids, epochs, lengths, voting types, predicted
    # and observed boxes = the SortTrack columns) device -> host.
    t_e2e = new_tracker()
    pinned = []
    for f in frames:
        b = pinned_empty(f["boxes"].shape, np.float32)
        b[...] = f["boxes"]
        ft = None
        if visual:
            ft = pinned_empty(f["features"].shape, np.float32)
            ft[...] = f["features"]
        pinned.append((b, ft))
    max_total = cfg.n_scenes * cfg.n_objects   # same on every rank (all_gather needs equal shapes)
    RING = 5                                    # result buffers: one more than the frames the library keeps in flight
    out_ring = [{"ids": pinned_empty((max_total,), np.uint64), "epochs": pinned_empty((max_total,), np.uint32),
                 "lengths": pinned_empty((max_total,), np.uint32), "voting_types": pinned_empty((max_total,), np.uint8),
                 "predicted": pinned_empty((max_total, 6), np.float32),
                 "observed": pinned_empty((max_total, 6), np.float32)} for _ in range(RING)]
    h2d, d2h = [], []
    sampler = ClockSampler(local)   # runs through the warm-up steps and the timed region (both under load)
    sampler.start()
    t_e2e.prefetch_inputs(pinned[0][0], features=pinned[0][1])
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i, f in enumerate(frames[: W + K]):
        total = len(f["boxes"])
        out = {k: v[:total] for k, v in out_ring[i % RING].items()}
        if i == W:
            t_e2e.sync()
            timed_region_begin()
            sampler.mark_begin()
            ev0.record()
        t_e2e.prefetch_inputs(pinned[i + 1][0], features=pinned[i + 1][1])
        t_e2e.predict_batch(f["scene_ids"], f["det_offsets"], pinned[i][0], features=pinned[i][1], out=out, wait=False)
        if i >= W:
            h2d.append(total * 24 + (total * D * 4 if visual else 0))
            d2h.append(total * (8 + 4 + 4 + 1 + 24 + 24))
    t_e2e.sync()
    torch.cuda.synchronize()   # the prefetch issued by the last timed step has landed too
    ev1.record()
    ev1.synchronize()
    sampler.mark_end()
    e2e_total_ms = float(ev0.elapsed_time(ev1))
    n_last = len(frames[W + K - 1]["boxes"])
    e2e_last = {k: v[:n_last].copy() for k, v in out_ring[(W + K - 1) % RING].items()}
    ids_e2e_last = e2e_last["ids"]
    t_e2e.close()

    # ---------------------------------------------------------------- value: inputs resident in HBM
    # One sb200_predict_batch_device call per step, stream-ordered: nothing in the loop waits for the device, nothing is
    # queried per step.  Work (pair-associations, dot products) and kernel times come from the library's cumulative
    # counters, read before and after the timed region.
    t_dev = new_tracker()
    dboxes = [torch.from_numpy(np.ascontiguousarray(f["boxes"])).to(dev) for f in frames[: W + K]]
    dfeats = [torch.from_numpy(f["features"]).to(dev) if visual else None for f in frames[: W + K]]
    # two sets of output columns: frame i writes set i & 1, so the gather of frame i can read its ids while frame i + 1 runs
    d_ids = [torch.zeros(max_total, dtype=torch.int64, device=dev) for _ in range(2)]
    d_ep = [torch.zeros(max_total, dtype=torch.int32, device=dev) for _ in range(2)]
    d_len = [torch.zeros(max_total, dtype=torch.int32, device=dev) for _ in range(2)]
    d_vt = [torch.zeros(max_total, dtype=torch.uint8, device=dev) for _ in range(2)]
    main_stream = torch.cuda.current_stream()
    # the caller's stream does not wait for every frame (sb200_set_stream_join 0): successive frames overlap where they can;
    # whoever consumes device-resident outputs joins explicitly (sb200_stream_join)
    t_dev.set_stream(main_stream.cuda_stream, join_per_call=False)
    gather = None
    if world > 1:
        # NCCL gather of the assigned track ids (the one exchange of the path) on a side stream: that stream joins frame i
        # (sb200_stream_join) and gathers its ids while frame i + 1 computes; frame i + 2, which rewrites the same output
        # set, is ordered after that gather through the caller's stream
        gather = {"stream": torch.cuda.Stream(device=dev),
                  "buf": [torch.zeros(max_total * world, dtype=torch.int64, device=dev) for _ in range(2)],
                  "done": [None, None]}
    torch.cuda.synchronize()

    def step_dev(i):
        f = frames[i]
        b = i & 1
        if gather is not None and gather["done"][b] is not None:
            main_stream.wait_event(gather["done"][b])   # the gather that read this output set two steps ago
        t_dev.predict_batch_device(f["scene_ids"], f["det_offsets"], dboxes[i].data_ptr(),
                                   dfeats[i].data_ptr() if visual else 0, d_ids=d_ids[b].data_ptr(),
                                   d_epochs=d_ep[b].data_ptr(), d_lengths=d_len[b].data_ptr(),
                                   d_voting_types=d_vt[b].data_ptr())
        if gather is not None:
            t_dev.stream_join(gather["stream"].cuda_stream)
            with torch.cuda.stream(gather["stream"]):
                dist.all_gather_into_tensor(gather["buf"][b], d_ids[b])
                ev = torch.cuda.Event()
                ev.record(gather["stream"])
                gather["done"][b] = ev

    sampler_dev = ClockSampler(local)
    sampler_dev.start()
    for i in range(W):
        step_dev(i)
    c0 = t_dev.work_counters()          # waits for the warm-up frames
    timed_region_begin()
    l0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler_dev.mark_begin()
    h0 = t_dev.host_counters()
    th0 = time.perf_counter()
    ev0.record()
    for i in range(W, W + K):
        step_dev(i)
    th1 = time.perf_counter()
    h1 = t_dev.host_counters()
    t_dev.stream_join(main_stream.cuda_stream)   # the timed span ends when the last frame has ended
    if gather is not None:
        for e in gather["done"]:
            if e is not None:
                main_stream.wait_event(e)   # the last gathers are part of the timed work
    ev1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler_dev.mark_end()
    dev_ms = ev0.elapsed_time(ev1)
    clocks_dev = sampler_dev.stop()
    clocks = sampler.stop() if sampler else None
    launches = eng.launch_count() - l0
    c1 = t_dev.work_counters()
    b_last = (W + K - 1) & 1
    ids_dev_last = d_ids[b_last][:n_last].cpu().numpy().astype(np.uint64)
    assert np.array_equal(ids_dev_last, ids_e2e_last), "device-pointer and host-pointer paths disagree"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {
            "ids": ids_dev_last, "epochs": d_ep[b_last][:n_last].cpu().numpy(),
            "lengths": d_len[b_last][:n_last].cpu().numpy(), "voting_types": d_vt[b_last][:n_last].cpu().numpy(),
            "predicted_boxes": e2e_last["predicted"], "observed_boxes": e2e_last["observed"]})
    if gather is not None:   # every rank holds every shard's ids of the last step
        gl = gather["buf"][(W + K - 1) & 1].view(world, max_total)[rank][: len(ids_dev_last)].cpu().numpy().astype(np.uint64)
        assert np.array_equal(gl, ids_dev_last), "gathered ids differ from the local shard"
    t_dev.close()
    scatter_info = None
    if world > 1 and not args.no_scatter:
        try:
            scatter_info = run_scatter_arm(eng, torch, dist, new_tracker, frames, dboxes, dfeats, W, K, D, visual, max_total,
                                           rank, world, local, ids_dev_last)
        except Exception as e:   # the headline line must survive a failure of this arm
            scatter_info = {"error": f"{type(e).__name__}: {e}"}

    units = float(c1["pair_associations"] - c0["pair_associations"])
    dots = float(c1["visual_dot_products"] - c0["visual_dot_products"])
    assert c1["frames"] - c0["frames"] == K
    stage_ms = {k_: (c1["stage_ms"][k_] - c0["stage_ms"][k_]) / K for k_ in c1["stage_ms"]}
    tc_frames = c1["tc_frames"] - c0["tc_frames"]
    fallback_scenes = (c1["dense_fallback_scenes"] - c0["dense_fallback_scenes"]) / K
    if tc_frames:
        stage_ms["vis_screen"] = (c1["vis_screen_ms"] - c0["vis_screen_ms"]) / tc_frames
        stage_ms["vis_refine"] = (c1["vis_refine_ms"] - c0["vis_refine_ms"]) / tc_frames
    # max over ranks of the timed region, sum over ranks of the units
    if world > 1:
        tm = torch.tensor([dev_ms, e2e_total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        un = torch.tensor([units], dtype=torch.float64, device=dev)
        dist.all_reduce(un, op=dist.ReduceOp.SUM)
        dev_ms, e2e_total_ms = float(tm[0]), float(tm[1])
        units_all = float(un[0])
    else:
        units_all = units

    if rank == 0:
        value = units_all / (dev_ms * 1e-3)
        e2e_value = units_all / (e2e_total_ms * 1e-3)
        # roofline of the dominant cost-matrix kernel: the tensor-core kernel of the visual cost (bound: tensor pipe),
        # timed with CUDA events on the tracker's stream inside the timed region; positional-only configs report the
        # positional stage against HBM.  The HBM-side view of the whole visual stage is kept as `visual_stage_hbm`.
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        tf_peak = float(peaks.get("bf16_tflops", 1590.0))
        peak_src = "measured (MEASURED_PEAKS.json, burst)" if peaks else "fallback (B200_PROFILING.md)"
        Kobs = 3 if visual else 1
        tr = newest_traffic()
        if visual and tc_frames:
            fl = 2.0 * dots * D / K                       # algorithmic FLOP per launch: 2 * M * (feature rows) * D
            m_tot = float(np.mean([len(frames[i]["boxes"]) for i in range(W, W + K)]))
            kms = stage_ms["vis_screen"]
            achieved = fl / (kms * 1e-3) / 1e12
            floor_bytes = None
            traffic = None
            if tr:
                traffic = tr[1].get("dram_bytes_per_launch")
                floor_bytes = tr[1].get("operand_floor_bytes")
            roof = {"kernel": "tensor-core visual cost kernel (tcgen05 BF16, kernels_feat_tc.cu)", "bound": "tensor",
                    "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                    "traffic": traffic, "traffic_source": os.path.basename(tr[0]) if tr else None,
                    "traffic_over_operand_floor": (traffic / floor_bytes) if traffic and floor_bytes else None,
                    "peak_source": peak_src, "algorithmic_flops_per_launch": fl,
                    # the kernel runs a fraction of a millisecond inside a ~1 ms step at full clocks, so the burst peak is
                    # the denominator; against the sustained figure of MEASURED_PEAKS.json the fraction would be:
                    "frac_of_sustained_peak": (achieved / float(peaks["bf16_tflops_sustained"])
                                               if peaks.get("bf16_tflops_sustained") else None),
                    "kernel_ms": kms, "candidate_rows_per_launch": m_tot,
                    "visual_stage": {"stage_ms": stage_ms["visual_cost"], "refine_ms": stage_ms.get("vis_refine"),
                                     "frac_of_peak_whole_stage": fl / (stage_ms["visual_cost"] * 1e-3) / 1e12 / tf_peak}}
        elif visual:
            # exact SIMT kernel (small frames / SB200_VIS_KERNEL=simt): FP32 pipe, no tensor cores
            fl = 3.0 * dots * D / K
            kms = stage_ms["visual_cost"]
            roof = {"kernel": "vis_cost_kernel (exact f32 SIMT)", "bound": "fp32", "achieved": fl / (kms * 1e-3) / 1e12,
                    "peak": 75.0, "unit": "TFLOP/s", "frac": fl / (kms * 1e-3) / 1e12 / 75.0, "traffic": None,
                    "peak_source": "nominal FP32 (no measured figure)", "kernel_ms": kms}
        else:
            m_l = np.concatenate([np.diff(frames[i]["det_offsets"]) for i in range(W, W + K)]).astype(np.float64)
            n_mean = units / max(1.0, float(m_l.sum()))       # mean tracks per scene over the timed steps
            alg_bytes = float(((m_l + n_mean) * 24).sum() / K + units * 4 / K)
            kms = stage_ms["positional_cost"]
            achieved = alg_bytes / (kms * 1e-3) / 1e9
            roof = {"kernel": "positional_cost stage (pos_fill_none + pos_scan)", "bound": "hbm", "achieved": achieved,
                    "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kms}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(name, cfg, {"option_overrides": {k_: (float(v_) if isinstance(v_, float) else v_) for k_, v_ in over.items()},
                                              "feat_noise": cfg.feat_noise} if (over or args.feat_noise is not None) else None),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(np.mean(h2d)),
                    "d2h_bytes_per_step": int(np.mean(d2h)), "ms_per_step": e2e_total_ms / K,
                    "host_affinity": affinity_note,
                    "pipeline": "sb200_predict_batch_async + sb200_prefetch_inputs: the pinned-host -> device copy of "
                                "frame i+1 is issued at the start of step i and overlaps its kernels; each timed step "
                                "contains one full input copy and one full SortTrack read-back (65 B per detection)"},
            "gpu_launches": int(launches),
            "gpu_launches_per_step": float(launches) / K,
            "clocks": clocks_dev if clocks_dev and clocks_dev.get("samples") else clocks,
            "clocks_e2e": clocks,
            "stages_ms": stage_ms,
            "exact_fallback_scenes_per_step": fallback_scenes,
            "host_sync": "none inside the timed region (stream-ordered predict, per-frame tables built on the device)",
            # what one frame costs the calling thread: library time not blocked on the device, and the whole Python loop
            "host_ms_per_step": {"library_unblocked": (h1["ms_total"] - h1["ms_blocked"] - h0["ms_total"] + h0["ms_blocked"]) / K,
                                 "library_blocked_on_device": (h1["ms_blocked"] - h0["ms_blocked"]) / K,
                                 "python_loop_wall": 1e3 * (th1 - th0) / K},
            "roofline": roof,
        }
        if world > 1:
            line["id_gather"] = "NCCL all_gather of the assigned ids, one step behind on a side stream (included in the timed span)"
            if scatter_info is not None:
                if "ms_per_step" in scatter_info:
                    scatter_info["value"] = units_all / (scatter_info["ms_per_step"] * K * 1e-3)
                line["scatter_ingest"] = scatter_info
        if old_affinity is not None:
            os.sched_setaffinity(0, old_affinity)   # the CPU baseline uses every core
        if not args.no_cpu_baseline and world == 1:
            import oracle as orc

            orc.build()
            cores = usable_cores()
            sample = args.cpu_sample_scenes or min(cfg.n_scenes, max(cores, 64))
            ccfg, cframes = make_frames(name, 6, 0, sample, feat_noise=args.feat_noise)
            cu, cs, _ = cpu_port_run(name, cframes, 4, 2, cores, over)
            line["cpu_baseline"] = {"value": cu / cs, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{sample} of {cfg.n_scenes} scenes x 2 timed frames after 4 warm-up frames, "
                                              f"{cores} threads (scene-parallel), {cs:.1f} s"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
