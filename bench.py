#!/usr/bin/env python
"""bench.py — flow-pairs/s of the hot path on synthetic frame streams (BASELINE.json: tvl1 @ 1920x1080).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload tvl1_1080p|...] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: `--pairs` (default 16)
consecutive frame pairs of a seeded synthetic stream (17 gray frames), i.e. one call of the batch shape of
DenseFlow::calc_optflows_imp (/root/reference/src/denseflow_gpu.cpp:307-342).  Every rank works on its own
stream (weak scaling, no data-path collective); value = pairs of all ranks / max-over-ranks time.

  value     frames already resident in HBM (uint8), flows left in HBM; CUDA events on the launching stream
  e2e       same work through the reference-facing host call (dfb_calc_batch_host): pinned host frames in,
            pinned host float2 flows out, H2D/D2H inside the timed region (the reference's own shape:
            upload :317-318, calc :327, download :339)
  roofline  dominant kernel = the fused tvl1 pair kernel, timed live with CUDA events around every launch
  cpu_baseline / --impl reference
            the CPU restatement of the same algorithm (oracle/, kind "port": the reference itself cannot be
            built here — it needs OpenCV-CUDA + Boost — and OpenCV's CPU DualTVL1 lives in contrib, not installed)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (algorithm, W, H, stream seed, BASELINE.json config it mirrors)
    "tvl1_1080p": ("tvl1", 1920, 1080, 1, "synthetic 1920x1080 stream, -a=tvl1 -s=1 (BASELINE.json configs[2])"),
    "tvl1_340x256": ("tvl1", 340, 256, 100, "synthetic 340x256 clips, -a=tvl1 -s=1 (BASELINE.json configs[4])"),
    "tvl1_256": ("tvl1", 256, 256, 0, "synthetic 256x256 pair stream, -a=tvl1 -s=1 (BASELINE.json configs[1])"),
    "farn_720p": ("farn", 1280, 720, 2, "synthetic 1280x720 stream, -a=farn -s=1 (BASELINE.json configs[3])"),
    "tvl1_455x256": ("tvl1", 455, 256, 1, "synthetic 455x256 frames (a 1080p video with -ns=256), -a=tvl1 -s=1"),
}
METRIC = "tvl1 flow-pairs/sec at 1920x1080"
NWIN = 2  # distinct input windows of pairs+1 frames each, alternated between steps (both arms)
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
# captures (scripts/ncu_traffic.py writes this file from the raw CSV pages under profiles/)
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")
DUMP_MAX_BYTES = 64 << 20  # --dump-outputs: a larger batch of flows is written as a seeded sample of DUMP_SAMPLE flow vectors
DUMP_SAMPLE = 1 << 22


def ncu_traffic(workload, pairs_per_launch):
    """Measured DRAM bytes per launch for this workload at the capture whose pairs-per-launch is closest to the
    run's, scaled by the pair ratio; (None, reason) when no capture is committed."""
    try:
        caps = json.load(open(NCU_TRAFFIC_FILE)).get(workload, [])
    except Exception:
        caps = []
    if not caps:
        return None, "no ncu capture committed for this workload"
    best = min(caps, key=lambda c_: abs(c_["pairs_per_launch"] - pairs_per_launch))
    scale = pairs_per_launch / best["pairs_per_launch"]
    return best["dram_bytes_per_launch"] * scale, "%s (%d-pair launch, %.3f GB DRAM read+write; scaled x%.2f to this run's pairs per launch)" % (
        best["source"], best["pairs_per_launch"], best["dram_bytes_per_launch"] / 1e9, scale)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tvl1_1080p", choices=sorted(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=0, help="frame pairs per step (default 16; 63 = one 64-frame clip for the 340x256 / 256x256 workloads)")
    ap.add_argument("--cpu-sample-pairs", type=int, default=3, help="pairs timed for cpu_baseline (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    # BASELINE.json configs[4]: a fixed list of clips dispatched over the GPUs from one dynamic queue (strong scaling)
    ap.add_argument("--list", type=int, default=0, help="list mode: number of clips in the video list (e.g. 1024); a step = one pass over the list")
    ap.add_argument("--list-frames", type=int, default=64, help="frames per clip")
    ap.add_argument("--list-distinct", type=int, default=8, help="distinct synthetic clips the list cycles through")
    ap.add_argument("--list-bound", type=int, default=32, help="-b of the CLI (default 32): the uint8 planes come back")
    ap.add_argument("--workers-per-gpu", type=int, default=2, help="list mode: host threads (engine handles) per GPU")
    # the reference's per-batch chain minus decode / file IO: BGR frames -> gray -> resize -> flow -> quantise -> 2 JPEGs per pair
    ap.add_argument("--chain", action="store_true", help="chain mode: dfb_process_bgr_batch_host on BGR frames of --chain-src size")
    ap.add_argument("--chain-src", default="", help="WxH of the decoded BGR frames (default: the workload's size, i.e. no resize)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the flows the timed path returned in its last step (rank 0) to DIR/flow.npy, float32: [pairs,H,W,2] "
                         "up to 64 MB, else the flow vectors at %d seeded (pair, y, x) positions in increasing order, [n,2]" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.list or args.chain):
        ap.error("--dump-outputs writes the flows of the default timed path; it does not apply to --impl reference, --list or --chain")
    if args.pairs <= 0:
        args.pairs = 63 if args.workload in ("tvl1_340x256", "tvl1_256") else 16
    return args


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for ts, line in self.rows:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs"), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_flows(flows_dev, out_dir):
    """--dump-outputs: the float32 flows [P,H,W,2] of a step as out_dir/flow.npy, or a fixed sample of them when larger than
    DUMP_MAX_BYTES, so that two builds can be compared output for output on the same arguments."""
    import numpy as np
    import torch
    f = flows_dev
    if f.numel() * f.element_size() > DUMP_MAX_BYTES:
        idx = np.sort(np.random.default_rng(0).integers(0, f.numel() // 2, DUMP_SAMPLE))
        f = f.reshape(-1, 2)[torch.from_numpy(idx).to(f.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "flow.npy"), f.cpu().numpy())


def make_stream(W, H, n_frames, seed, rank):
    from denseflow_b200 import synth
    # every rank gets its own clip: different texture seed and motion phase (config-5 style sharding)
    return synth.stream(H, W, n_frames, seed + 1000 * rank, phase=7.0 * rank)


def usable_cores():
    """Cores this process may really use: scheduler affinity capped by the cgroup CPU quota (containers report the
    host's core count in os.cpu_count())."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def _cpu_worker(job):
    alg, a, b, threads = job
    if alg == "farn":
        # BASELINE.json configs[0] / BASELINE.md R1: OpenCV's own CPU Farneback with the create() defaults of
        # src/denseflow_gpu.cpp:301 — effectively single-threaded, so one pair per core
        import cv2
        cv2.setNumThreads(1)
        cv2.calcOpticalFlowFarneback(a, b, None, 0.5, 5, 13, 10, 5, 1.1, 0)
        return 1
    from oracle import pyoracle as O
    O.lib().orc_set_num_threads(threads)
    O.tvl1_calc(a, b)
    return 1


def cpu_split(alg):
    """(processes, threads per process) for the CPU arm: tvl1 = oracle port, OpenMP loops stop scaling past ~8 threads;
    farn = cv2.calcOpticalFlowFarneback, one single-threaded pair per core."""
    cores = usable_cores()
    threads = 1 if alg == "farn" else min(8, cores)
    return max(1, cores // threads), threads


def cpu_kind_note(alg):
    if alg == "farn":
        return ("cv2.calcOpticalFlowFarneback(a,b,None,0.5,5,13,10,5,1.1,0) (OpenCV %s CPU, the algorithm and defaults of "
                "cv::cuda::FarnebackOpticalFlow::create(); differs from the CUDA class only in the resize sampling convention)" % __import__("cv2").__version__)
    return ("CPU restatement of the CUDA algorithm (oracle/, -O2 scalar C + OpenMP: a soft baseline): OpenCV CPU DualTVL1 (contrib) is not "
            "installed and the reference itself needs OpenCV-CUDA")


def cpu_port_throughput(alg, frames, n_pairs_per_proc, warm=True):
    """The CPU restatement on ALL host cores: the per-pair OpenMP loops stop scaling long before 64 threads, so the
    cores are split into P processes x T threads working on different pairs concurrently (aggregate pairs/s)."""
    import multiprocessing as mp
    procs, threads = cpu_split(alg)
    n = len(frames) - 1
    jobs = [(alg, frames[i % n], frames[i % n + 1], threads) for i in range(procs * n_pairs_per_proc)]
    ctx = mp.get_context("spawn")
    pool = ctx.Pool(procs)
    try:
        if warm:
            pool.map(_cpu_worker, jobs[:procs])
        t0 = time.perf_counter()
        pool.map(_cpu_worker, jobs, chunksize=1)
        dt = time.perf_counter() - t0
    finally:
        pool.close()
        pool.join()
    return {"value": len(jobs) / dt, "unit": "pairs/s", "cores": procs * threads, "kind": "port",
            "sample": "%d pairs of the same stream (%d processes x %d threads, %d pairs each, after one warm-up pair per process); %s"
                      % (len(jobs), procs, threads, n_pairs_per_proc, cpu_kind_note(alg))}


# ---------------------------------------------------------------------------------------------------------
def bench_config(args, alg, W, H, desc):
    """The `config` object both arms print (same workload, same frames, same pairs per step)."""
    P = args.pairs
    return {"workload": desc, "algorithm": alg, "width": W, "height": H, "step": 1, "pairs_per_step": P,
            "frames_per_step": P + 1, "sharding": "one independent frame stream per rank, no collective",
            "l2": "no explicit flush: per-pair working set (16 fp32 planes x 5 levels, ~0.3 GB x lanes) exceeds the 126 MB L2 "
                  "and consecutive steps alternate between two input windows",
            "aee_tolerance_px": 0.01}


def run_reference(args, alg, W, H, seed, desc):
    """--impl reference: the reference path's CPU implementation (oracle port) on the host cores; rank 0 only.
    Same frames and the same pairs per step as the GPU arm: step i solves the P pairs of input window i % NWIN."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    P = args.pairs
    frames = make_stream(W, H, NWIN * (P + 1), seed, 0).reshape(NWIN, P + 1, H, W)
    procs, threads = cpu_split(alg)
    cores = procs * threads
    step_jobs = [[(alg, frames[w][i], frames[w][i + 1], threads) for i in range(P)] for w in range(NWIN)]
    ctx = mp.get_context("spawn")
    pool = ctx.Pool(procs)
    try:
        for i in range(args.warmup):
            pool.map(_cpu_worker, step_jobs[i % NWIN], chunksize=1)
        t0 = time.perf_counter()
        for i in range(args.steps):
            pool.map(_cpu_worker, step_jobs[(args.warmup + i) % NWIN], chunksize=1)
        dt = time.perf_counter() - t0
    finally:
        pool.close()  # let the workers exit on their own (a terminate() would lose their atexit records)
        pool.join()
    value = args.steps * P / dt
    sample = ("each step = the %d pairs of one input window of the workload stream (the GPU arm's frames), spread over %d processes x %d "
              "threads = %d usable host cores; %s" % (P, procs, threads, cores, cpu_kind_note(alg)))
    line = {
        "impl": "reference", "metric": METRIC if args.workload == "tvl1_1080p" else "%s flow-pairs/sec at %dx%d" % (alg, W, H),
        "value": value, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, alg, W, H, desc),
        "note": cpu_kind_note(alg) + "; the reference itself needs OpenCV-CUDA+Boost and cannot be built in this image",
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
def run_list_mode(args, alg, W, H, seed, desc):
    """--list N: a FIXED list of N clips (BASELINE.json configs[4]: 1024 x 340x256x64) drained from one dynamic work queue
    by all GPUs of the job: one process per GPU under torchrun (queue in POSIX shared memory), or one process with
    --gpus x --workers-per-gpu threads.  Unit of work = one video; host frames in, the convertFlowToImage planes back in
    host memory (what the jpg writer consumes); strong scaling; time = max over ranks of the wall time of the pass."""
    import numpy as np
    import torch
    import denseflow_b200 as d
    from denseflow_b200 import listrun, shard, synth
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank, local_rank, world = shard.init()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    wpg = max(1, args.workers_per_gpu)
    if world > 1:
        mode, n_gpus, devices = "one process per GPU, %d worker threads each, queue in POSIX shared memory" % wpg, world, [local_rank] * wpg
    else:
        mode, n_gpus = "one process, %d worker threads per GPU, in-process queue" % wpg, max(1, args.gpus)
        devices = [g for g in range(n_gpus) for _ in range(wpg)]
    N, F, NB, bound = args.list, args.list_frames, max(1, min(args.list_distinct, args.list)), args.list_bound
    base = [torch.from_numpy(synth.stream(H, W, F, seed + c, phase=float(c))).pin_memory() for c in range(NB)]
    base_np = [b.numpy() for b in base]
    clips = [[base_np[i % NB][t] for t in range(F)] for i in range(N)]
    runner = listrun.ListRunner(alg, devices, W, H)
    packed = runner.pack(clips)
    warm = runner.pack(clips[:2 * len(devices)])
    queue = None
    if world > 1:
        qname = "/dfb_bench_%s" % os.environ.get("MASTER_PORT", "0")
        if rank == 0:
            queue = listrun.WorkQueue(qname, create=True)
        shard.barrier()
        if rank != 0:
            queue = listrun.WorkQueue(qname, create=False)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 1)):  # private queue: every worker of every rank gets warm (lanes, pinned rings, clocks)
        runner.run(None, step=1, bound=bound, packed=warm)
    torch.cuda.synchronize(dev)
    tot = {"flows": 0, "clips": 0, "launches": 0, "h2d": 0, "d2h": 0}
    dts, last = [], None
    tmark0 = sampler.mark()
    for _ in range(args.steps):
        shard.barrier()
        if queue is not None and rank == 0:
            queue.reset()
        shard.barrier()
        t0 = time.perf_counter()
        last = runner.run(None, step=1, bound=bound, queue=queue, packed=packed)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        dts.append(shard.all_max(dt, dev))
        for k, key in (("flows", "flows"), ("clips", "clips"), ("launches", "kernel_launches"), ("h2d", "h2d_bytes"), ("d2h", "d2h_bytes")):
            tot[k] += last[key]
    tmark1 = sampler.mark()
    g = {k: shard.all_sum(v, dev) for k, v in tot.items()}
    per_rank_clips = [int(shard.all_sum(last["clips"] if r == rank else 0, dev)) for r in range(world)]
    finish = last["finish_seconds_per_worker"]
    tail = shard.all_max(max(finish), dev) - (-shard.all_max(-min(finish), dev))
    busy = shard.all_sum(sum(last["busy_seconds_per_worker"]), dev) / (max(dts[-1], 1e-9) * len(devices) * world)
    clocks = sampler.stop(tmark0, tmark1) if rank == 0 else None
    parity = None
    if rank == 0:
        from oracle import pyoracle as O
        e = d.create(alg, local_rank, W, H)
        a, b = base_np[0][0], base_np[0][1]
        got = e.calc_batch([a, b], 1)[0]
        qx, qy = e.calc_batch([a, b], 1, bound=bound)
        ref = (O.tvl1_calc if alg == "tvl1" else O.farn_calc)(a, b)
        ox, oy = O.quantise(ref, bound)
        parity = {"aee_px": synth.aee(got, ref), "pair": "clip 0, frames 0-1",
                  "quantised_planes_equal_fraction": float(((qx[0] == ox) & (qy[0] == oy)).mean()),
                  "quantised_max_level_diff": int(max(np.abs(qx[0].astype(int) - ox).max(), np.abs(qy[0].astype(int) - oy).max())),
                  "against": "oracle (CPU restatement)", "tolerance_px": 0.01}
        e.release()
    if rank == 0:
        total_s = sum(dts)
        value = g["flows"] / total_s
        line = {
            "metric": "%s flow-pairs/sec at %dx%d, %d-clip list" % (alg, W, H, N), "value": value, "unit": "pairs/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": total_s / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "algorithm": alg, "width": W, "height": H, "step": 1, "list_clips": N, "frames_per_clip": F,
                       "distinct_clips": NB, "bound": bound, "mode": mode, "queue": "dynamic (fetch-and-increment), unit = one video",
                       "completion": "a video is reported done after its last chunk's planes are in host memory (src/denseflow_gpu.cpp:456-470)",
                       "value_is": "end to end (there is no HBM-resident variant of a list job): pinned host frames in, uint8 planes out",
                       "l2": "each clip's frames and outputs are touched once; 16 lanes x ~20 MB of planes per launch"},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": g["h2d"] / args.steps, "d2h_bytes_per_step": g["d2h"] / args.steps,
                    "call": "dfb_list_run -> dfb_calc_batch_host_u8 per video"},
            "gpu_launches": int(g["launches"]), "clocks": clocks,
            "list": {"clips_per_rank_last_step": per_rank_clips, "clips_per_worker_rank0": last["clips_per_worker"],
                     "tail_seconds_last_step": tail, "worker_busy_fraction_last_step": busy, "seconds_per_step": dts},
        }
        if parity:
            line["parity_aee_px"] = parity["aee_px"]
            line["parity"] = parity
        print(json.dumps(line), flush=True)
    runner.close()
    if queue is not None:
        shard.barrier()
        queue.close()
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


def _cpu_chain_worker(job):
    """The reference's CPU stages around the flow for one pair: cvtColor + resize of one new frame (src/denseflow_gpu.cpp:163-170)
    and convertFlowToImage's output through two imencode(".jpg") calls (src/common.cpp:56-57)."""
    import cv2
    import numpy as np
    bgr, size, qx, qy, reps = job
    cv2.setNumThreads(1)
    t0 = time.perf_counter()
    for _ in range(reps):
        g = cv2.cvtColor(bgr, cv2.COLOR_BGR2GRAY)
        if size != (bgr.shape[1], bgr.shape[0]):
            g = cv2.resize(g, size)
    t1 = time.perf_counter()
    for _ in range(reps):
        cv2.imencode(".jpg", qx)
        cv2.imencode(".jpg", qy)
    t2 = time.perf_counter()
    return (t1 - t0) / reps, (t2 - t1) / reps


def run_chain_mode(args, alg, W, H, seed, desc):
    """--chain: the reference's per-batch chain minus decode and file IO through dfb_process_bgr_batch_host: pinned BGR frames in,
    two JPEG bitstreams per pair out; (W, H) of the workload is the size the flow runs at, --chain-src the decoded frame size."""
    import numpy as np
    import torch
    import denseflow_b200 as d
    from denseflow_b200 import shard, synth
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank, local_rank, world = shard.init()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    SW, SH = (int(x) for x in args.chain_src.split("x")) if args.chain_src else (W, H)
    P = args.pairs
    gray = synth.stream(SH, SW, P + 1, seed + 1000 * rank, phase=7.0 * rank)
    bgr_t = torch.from_numpy(np.stack([np.roll(gray, 2, 2), gray, 255 - np.roll(gray, 3, 1)], -1).copy()).pin_memory()
    bgr = [bgr_t[i].numpy() for i in range(P + 1)]
    e = d.create(alg, local_rank, W, H)
    new_size = None if (SW, SH) == (W, H) else (W, H)
    out = None
    for _ in range(max(args.warmup, 1)):
        out = e.process_bgr_batch(bgr, step=1, bound=20, new_size=new_size)
    torch.cuda.synchronize(dev)
    shard.barrier()
    e.reset_counters()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = e.process_bgr_batch(bgr, step=1, bound=20, new_size=new_size)
    torch.cuda.synchronize(dev)
    dt = shard.all_max(time.perf_counter() - t0, dev)
    c = e.counters()
    value = world * args.steps * P / dt
    if rank == 0:
        import cv2
        import multiprocessing as mp
        # parity of the chain's output: the decoded JPEGs against the quantised planes of the same engine on cv2-prepared frames
        frames = [cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr[:2]]
        if new_size:
            frames = [cv2.resize(f, new_size) for f in frames]
        qx, qy = e.calc_batch(frames, 1, bound=20)
        dx = cv2.imdecode(np.frombuffer(out[0][0], np.uint8), cv2.IMREAD_UNCHANGED)
        # CPU stages, one pair per core
        cores = usable_cores()
        jobs = [(bgr[i % (P + 1)], (W, H), qx[0], qy[0], 20) for i in range(cores)]
        pool = mp.get_context("spawn").Pool(cores)
        try:
            pool.map(_cpu_chain_worker, jobs[:cores])
            res = pool.map(_cpu_chain_worker, jobs)
        finally:
            pool.close()
            pool.join()
        prep = float(np.mean([r[0] for r in res]))
        enc = float(np.mean([r[1] for r in res]))
        line = {"metric": "%s chain pairs/sec: BGR %dx%d -> gray -> %dx%d -> flow -> quantise -> 2 JPEG" % (alg, SW, SH, W, H), "value": value,
                "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": dt / args.steps * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": desc + " as the flow size; decoded frames %dx%d BGR" % (SW, SH), "algorithm": alg, "pairs_per_step": P, "bound": 20,
                           "jpeg_quality": 95, "call": "dfb_process_bgr_batch_host"},
                "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": c["h2d_bytes"] / args.steps, "d2h_bytes_per_step": c["d2h_bytes"] / args.steps},
                "gpu_launches": int(c["kernel_launches"]),
                "jpeg_decoded_vs_planes": {"max_abs": int(np.abs(dx.astype(int) - qx[0].astype(int)).max()),
                                           "mean_abs": float(np.abs(dx.astype(int) - qx[0].astype(int)).mean())},
                "cpu_stages": {"cvtColor_resize_ms_per_frame": prep * 1e3, "two_imencode_ms_per_pair": enc * 1e3,
                               "pairs_per_s_all_cores": cores / (prep + enc), "cores": cores,
                               "note": "cv2 %s, one pair per core (the reference runs these stages on one thread each, include/dense_flow.h:76-80)" % cv2.__version__}}
        print(json.dumps(line), flush=True)
    e.release()


def main():
    args = parse()
    alg, W, H, seed, desc = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, alg, W, H, seed, desc)
    if args.list > 0:
        return run_list_mode(args, alg, W, H, seed, desc)
    if args.chain:
        return run_chain_mode(args, alg, W, H, seed, desc)

    import numpy as np
    import torch
    import denseflow_b200 as d
    from denseflow_b200 import shard

    # keep stdout to the one JSON line: NCCL's own log lines (e.g. "NCCL version ...") go to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank, local_rank, world = shard.init()
    if world != args.gpus and rank == 0:
        print("warning: WORLD_SIZE=%d but --gpus=%d" % (world, args.gpus), file=sys.stderr)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    P = args.pairs
    n_frames = P + 1
    frames_np = make_stream(W, H, NWIN * n_frames, seed, rank).reshape(NWIN, n_frames, H, W)
    frames_pin = [torch.from_numpy(frames_np[w]).pin_memory() for w in range(NWIN)]
    frames_dev = [f.to(dev) for f in frames_pin]
    flows_dev = torch.empty((P, H, W, 2), dtype=torch.float32, device=dev)
    flows_pin = torch.empty((P, H, W, 2), dtype=torch.float32).pin_memory()

    eng = d.create(alg, local_rank, W, H)
    eng.set("time_kernels", 1)
    stream = torch.cuda.current_stream(dev)

    def step_device(i):
        eng.calc_batch_device(frames_dev[i % NWIN], 1, flows_dev)

    fl_np = flows_pin.numpy()
    fr_lists = [[frames_pin[w][i].numpy() for i in range(n_frames)] for w in range(NWIN)]

    def step_host(i):
        eng.calc_batch(fr_lists[i % NWIN], 1, flows=fl_np)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---------------- value: inputs resident in HBM -------------------------------------------------------
    for i in range(args.warmup):
        step_device(i)
    torch.cuda.synchronize(dev)
    shard.barrier()
    eng.reset_counters()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tmark0 = sampler.mark()
    ev0.record(stream)
    for i in range(args.steps):
        step_device(args.warmup + i)
    ev1.record(stream)
    torch.cuda.synchronize(dev)
    tmark1 = sampler.mark()
    dt_dev = ev0.elapsed_time(ev1) / 1e3
    shard.barrier()
    dt_dev_max = shard.all_max(dt_dev, dev)
    c = eng.counters()
    launches = int(shard.all_sum(c["kernel_launches"], dev))
    total_pairs = world * args.steps * P
    value = total_pairs / dt_dev_max
    if args.dump_outputs and rank == 0:
        dump_flows(flows_dev, args.dump_outputs)  # before the unfused-schedule and parity runs below overwrite flows_dev

    # ---------------- roofline of the dominant kernel (rank 0's GPU) --------------------------------------
    roof = None
    if alg == "tvl1" and c["timed_kernel_launches"]:
        iters, sizes = eng.tvl1_stats()
        sum_px = sum(w_ * h_ for w_, h_ in sizes)
        warps = int(eng.get("warps"))
        npairs = c["timed_kernel_pairs"]
        k = int(eng.get("fused_k"))
        # algorithmic bytes (DESIGN.md §4): fused primal+dual iteration 64 B/px.iter (10 plane reads + 6 writes),
        # warp 44 B/px.warp, level start 28 B/px (I1 read, I1x/I1y + 4 p planes written), upsample 2*10 B/px_dst, merge 16 B/px
        b_iter = 64.0 * c["pixel_iters"]    # per-iteration formulation (k = 1): 64 B per pixel and iteration
        b_visit = 64.0 * c["pixel_chunks"]  # k-blocked formulation: 64 B per pixel and tile visit (<= k iterations on chip)
        b_other = npairs * (44.0 * warps * sum_px + 28.0 * sum_px + 20.0 * (sum_px - sizes[-1][0] * sizes[-1][1]) + 16.0 * W * H)
        kt = c["timed_kernel_ns"] / 1e9
        peak, peak_src = load_peaks()
        achieved = (b_visit + b_other) / kt / 1e9
        equiv = (b_iter + b_other) / kt / 1e9
        roof = {
            "bound": "hbm", "kernel": "k_tvl1_pair (persistent fused TV-L1 pair kernel)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures
            "traffic": ncu_traffic(args.workload, npairs / c["timed_kernel_launches"])[0],
            "traffic_source": ncu_traffic(args.workload, npairs / c["timed_kernel_launches"])[1],
            "peak_source": peak_src,
            "formulation": "SURVEY §8d, temporally blocked fused primal+dual: algorithmic bytes = 64 B per pixel per tile visit "
                           "(10 plane reads + 6 writes; up to k=%d iterations stay on chip per visit) x executed pixel-visits "
                           "+ 44 B/px per warp + level-start/upsample/merge.  The kernel is bound by instruction-level parallelism, "
                           "not by HBM (DESIGN.md §4.4), hence the low fraction; `per_iteration_equivalent` restates the same run "
                           "under the k=1 figure (64 B per pixel and iteration), i.e. the bandwidth an unblocked fused kernel "
                           "would need to match it" % k,
            "k": k,
            "algorithmic_bytes_per_launch": (b_visit + b_other) / c["timed_kernel_launches"],
            "per_iteration_equivalent": {"achieved": equiv, "frac": equiv / peak,
                                         "algorithmic_bytes_per_launch": (b_iter + b_other) / c["timed_kernel_launches"]},
            "avg_launch_ms": kt / c["timed_kernel_launches"] * 1e3,
            "pairs_per_launch": npairs / c["timed_kernel_launches"],
            "pixel_iters_per_pair": c["pixel_iters"] / max(npairs, 1),
            "pixel_visits_per_pair": c["pixel_chunks"] / max(npairs, 1),
            "kernel_share_of_step": kt / dt_dev,
        }

    if alg == "farn" and c["timed_kernel_launches"]:
        peak, peak_src = load_peaks()
        kt = c["timed_kernel_ns"] / 1e9
        nl = c["timed_kernel_launches"]
        npairs = c["timed_kernel_pairs"]
        # fused iteration kernel (box 13x13 -> 2x2 solve -> rebuild M): read M(5) + R0(5) + R1(5, gathered) + write M(5) + flow(2)
        # = 88 B per level pixel and iteration (SURVEY §8d, fused formulation); pixel_iters is counted by the engine
        b_alg = 88.0 * c["pixel_iters"]
        achieved = b_alg / kt / 1e9
        t = ncu_traffic(args.workload, min(8, P))  # pairs per launch = the engine's batch of up to 8 pairs (blockIdx.z)
        if t[0] is not None:
            # the capture is of a FULL-RESOLUTION launch (649 MB algorithmic for 8 pairs at 1280x720); the run's launches cover all
            # pyramid levels, so the measured bytes are scaled by the algorithmic bytes of an average launch over those of the captured one
            full = 88.0 * min(8, P) * W * H
            t = (t[0] * (b_alg / nl) / full, t[1] + "; a full-resolution launch, scaled by %.3f to the run's average launch over all levels" % ((b_alg / nl) / full))
        roof = {"bound": "hbm", "kernel": "k_box_solve_update<6> (13x13 box mean of M -> 2x2 solve -> rebuild M, one launch per iteration and level, up to 8 pairs per launch)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": t[0], "traffic_source": t[1],
                "peak_source": peak_src,
                "formulation": "SURVEY §8d fused-iteration figure: 88 B per level pixel and iteration x executed pixel-iterations (engine counter), "
                               "over the CUDA-event time of the iteration launches only (one event pair per level); the last iteration of a level "
                               "skips the rebuild (48 B) and is counted at 88 B too, i.e. the figure is an upper bound by ~4 %",
                "algorithmic_bytes_per_launch": b_alg / nl, "avg_launch_ms": kt / nl * 1e3,
                "launches": nl, "pixel_iters_per_pair": c["pixel_iters"] / max(npairs, 1), "kernel_share_of_step": kt / dt_dev}

    # ---------------- stand-alone primal / dual kernels of the unfused schedule vs the HBM roofline ------------
    kernels = None
    if alg == "tvl1" and rank == 0:
        peak, peak_src = load_peaks()
        kernels = {}
        for name, bpp in (("estimate_u", 48), ("estimate_dual", 40)):
            ms = eng.debug_time_kernel(name, W, H, sets=6, reps=60)
            gbs = bpp * W * H / (ms * 1e-3) / 1e9
            kernels["k_" + name] = {"bytes_per_px": bpp, "ms_per_launch": ms, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak,
                                    "note": "CUDA events over 60 launches rotating 6 operand sets (L2-busting), %dx%d" % (W, H)}

    # ---------------- the reference's launch structure on the same GPU (one kernel per half-step, host-side checks) ----
    unfused = None
    if alg == "tvl1" and rank == 0:
        eu = d.create(alg, local_rank, W, H)
        eu.set("fused", 0)
        nq = min(P, 4)
        eu.calc_batch_device(frames_dev[0][:nq + 1], 1, flows_dev[:nq])
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()  # host clock: this schedule synchronises with the host at every convergence check
        eu.calc_batch_device(frames_dev[1][:nq + 1], 1, flows_dev[:nq])
        torch.cuda.synchronize(dev)
        dtu = time.perf_counter() - t0
        cu = eu.counters()
        unfused = {"value": nq / dtu, "unit": "pairs/s", "kernel_launches_per_pair": cu["kernel_launches"] / (2 * nq),
                   "note": "same arithmetic, fused=0: ~2 000 launches and one stream sync per convergence check per pair, as "
                           "cv::cuda::OpticalFlowDual_TVL1 is structured (OpenCV-CUDA itself is not installable here)"}
        eu.release()

    # ---------------- e2e: host buffers through the reference-facing call ---------------------------------
    for i in range(max(args.warmup, 1)):
        step_host(i)
    torch.cuda.synchronize(dev)
    shard.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_host(args.warmup + i)
    torch.cuda.synchronize(dev)
    dt_host = time.perf_counter() - t0
    shard.barrier()
    dt_host_max = shard.all_max(dt_host, dev)
    e2e_value = total_pairs / dt_host_max
    # same end-to-end call, but the flow is bounded + quantised on the GPU and the two uint8 planes come back
    # (dfb_calc_batch_host_u8, SURVEY §8 f1: what the jpg path needs; 2 B/px instead of 8 B/px over PCIe)
    qx_pin = torch.empty((P, H, W), dtype=torch.uint8).pin_memory()
    qy_pin = torch.empty((P, H, W), dtype=torch.uint8).pin_memory()
    qx_np, qy_np = qx_pin.numpy(), qy_pin.numpy()

    def step_host_u8(i):
        eng.calc_batch_u8_into(fr_lists[i % NWIN], 1, 20, qx_np, qy_np)

    step_host_u8(0)
    torch.cuda.synchronize(dev)
    shard.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_host_u8(args.warmup + i)
    torch.cuda.synchronize(dev)
    dt_u8_max = shard.all_max(time.perf_counter() - t0, dev)
    clocks = sampler.stop(tmark0, tmark1) if rank == 0 else None

    # ---------------- parity of this run's output (outside the timed region): one flow of the timed workload vs the oracle ----
    parity = None
    if rank == 0:
        from oracle import pyoracle as O
        from denseflow_b200 import synth
        O.lib().orc_set_num_threads(min(16, usable_cores()))
        step_device(0)  # window 0 again: flows_dev[j] = flow(frame j -> j+1)
        torch.cuda.synchronize(dev)
        j = P - 1  # the last pair of the step (at 1080p it is in the partial launch)
        got = flows_dev[j].cpu().numpy()
        if alg == "tvl1":
            ref, ref_log = O.tvl1_calc(frames_np[0][j], frames_np[0][j + 1], return_iters=True)
            log = eng.tvl1_pair_stats(j)
            parity = {"aee_px": synth.aee(got, ref), "max_abs_px": float(np.abs(got - ref).max()), "pair": j, "against": "oracle/tvl1_oracle.c (CPU restatement, parity unpinned: no TV-L1 binary exists in this image)",
                      "iterations_engine": int(log.sum()), "iterations_oracle": int(ref_log.sum()),
                      "iteration_log_equal": bool(np.array_equal(log, ref_log)), "tolerance_px": 0.01}
        else:
            ref = O.farn_calc(frames_np[0][j], frames_np[0][j + 1])
            parity = {"aee_px": synth.aee(got, ref), "max_abs_px": float(np.abs(got - ref).max()), "pair": j,
                      "against": "oracle/farneback_oracle.c (pinned to cv2.calcOpticalFlowFarneback)", "tolerance_px": 0.01}

    # ---------------- cpu baseline: bounded sample of the same workload on the host cores -----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_port_throughput(alg, frames_np[0], args.cpu_sample_pairs)

    if rank == 0:
        line = {
            "metric": METRIC if args.workload == "tvl1_1080p" else "%s flow-pairs/sec at %dx%d" % (alg, W, H),
            "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt_dev_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args, alg, W, H, desc),
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": n_frames * W * H,
                    "d2h_bytes_per_step": P * W * H * 8, "ms_per_step": dt_host_max / args.steps * 1e3,
                    "call": "dfb_calc_batch_host (pinned host frames in, pinned host CV_32FC2 flows out)"},
            "e2e_quantised": {"value": total_pairs / dt_u8_max, "unit": "pairs/s", "h2d_bytes_per_step": n_frames * W * H,
                              "d2h_bytes_per_step": P * W * H * 2,
                              "call": "dfb_calc_batch_host_u8 (bound 20: the two uint8 planes convertFlowToImage would produce)"},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if parity:
            line["parity_aee_px"] = parity["aee_px"]
            line["parity"] = parity
        if roof:
            line["roofline"] = roof
        if kernels:
            line["unfused_kernels"] = kernels
        if unfused:
            line["unfused_schedule"] = unfused
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    shard.barrier()  # rank 0's parity check runs after the last timing collective: every rank leaves together
    eng.release()
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
