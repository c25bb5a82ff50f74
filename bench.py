#!/usr/bin/env python3
"""bench.py -- benchmark of the B200-native ORB front-end (BASELINE.json metric and configs).

Headline (the JSON line's top level): a "step" is one pass of extract+describe (ORBextractor::operator(), 8 levels,
scale 1.2, FAST 20/7, 1000 features) over one batch of synthetic 752x480 EuRoC-shaped frames on every rank's own GPU
(one agent stream set per GPU, no data-path collective: the path shards by agent -> "weak" scaling).

  value         frames/s, whole job, inputs and outputs resident in HBM (CUDA events on the launching stream)
  e2e           frames/s through the public host-buffer API (pinned host frames in, keypoints + descriptors out, H2D /
                D2H inside the timed region), with the box's measured H2D ceiling next to it
  roofline      pyramid + FAST kernels, algorithmic bytes / live event time, against the measured HBM peak
  cpu_baseline  the CPU oracle (port of the reference path) on this box's host cores, bounded sample

`workloads` holds one record per remaining BASELINE.json config, each with its own config.workload, device-timed
value, end-to-end value and a parity spot-check against the oracle made inside the run:
  config2_kitti      1241x376 / 2000 features extraction + SearchForInitialization(F_0, F_k), k = 1..10
  config34_tracking  per-frame tracking step of co-located agents: extract + resident frame + ComputeBoW +
                     SearchByBoW(KF, F) + SearchByProjection(cur, last, 15) + SearchByProjection(F, local map, th 1)
  config5_place      2000 query descriptors against 100 000 keyframes x 256 descriptors with 1 % planted copies,
                     strong-scaled over the ranks (NCCL all-gather of the per-shard top-2 inside the C ABI)

`--impl reference` times the reference path's CPU restatement (oracle/; the reference cannot be built as a whole,
SURVEY.md F3) with all host threads on the same workload and prints the same JSON line.

`--dump-outputs DIR` writes what the headline's device-resident path returned in its last timed step for a fixed,
seeded sample of the batch (dump_outputs below), so that two builds can be compared output for output on identical
inputs.  `--steps` sets the headline's timed steps (device-resident and end to end); the other workloads time fixed
counts.  bench.py runs the libraries build() left in the tree, stops if libswm_orb.so is older than its sources, and
writes nothing in the tree.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: the driver reads ONE JSON line

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, NFEAT = 752, 480, 1000
PYR_FAST_BYTES = 3912047   # SURVEY.md 8(d): pyramid R+W + FAST R per 752x480 frame
BLUR_BYTES = 2234734       # blur R+W per frame (fused into the same kernels)
METRIC = "orb_extract_frames_per_sec"  # BASELINE.json: ORB frames/sec (1000 feat, 752x480), whole job over all GPUs
UNIT = "frames/s"
WORKLOAD = "EuRoC-shaped 752x480 8-bit frames, ORBextractor(1000, 1.2, 8, 20, 7), extract+describe"
EUROC_CAM = (458.654, 457.296, 367.215, 248.375, -0.28340811, 0.07395907, 0.00019359, 1.76187114e-05, 0.0)


def _traffic_per_frame():
    """DRAM bytes per frame of the roofline kernels from the newest committed ncu --set full capture (profiles/)."""
    for name in ("r2_traffic.json", "r1k_traffic.json"):
        try:
            return float(json.load(open(os.path.join(ROOT, "profiles", name)))["dram_bytes_per_frame"]), name
        except Exception:
            continue
    return None, None


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

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
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_numa(local_rank, world):
    """Pin this rank to the host cores of its GPU's NUMA node BEFORE any pinned buffer is allocated (first touch then
    places the staging memory next to the GPU's PCIe root).  Returns a description for the JSON line."""
    info = {"bound": False, "nproc": os.cpu_count()}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        info["pci_bus"] = bus
        info["numa_node"] = node
        if node < 0:
            return info
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if not allowed:
            return info
        # ranks whose GPUs share this node split its cores evenly
        peers = []
        for r in range(world):
            try:
                b2 = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(r)).busId
                b2 = (b2.decode() if isinstance(b2, bytes) else b2).lower()
                if len(b2.split(":")[0]) == 8:
                    b2 = b2[4:]
                if int(open(f"/sys/bus/pci/devices/{b2}/numa_node").read()) == node:
                    peers.append(r)
            except Exception:
                pass
        k = peers.index(local_rank) if local_rank in peers else 0
        per = max(1, len(allowed) // max(1, len(peers)))
        mine = allowed[k * per:(k + 1) * per] or allowed
        os.sched_setaffinity(0, mine)
        info.update(bound=True, cores=len(mine), node_cores=len(allowed), ranks_on_node=len(peers))
    except Exception as e:  # binding is an optimisation, never fatal
        info["error"] = str(e)[:120]
    return info


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return ""


def cpu_oracle_rate(frames, seconds_budget, threads):
    """frames/s of the CPU oracle on `threads` host threads over a bounded sample."""
    import oracle_lib
    from concurrent.futures import ThreadPoolExecutor
    ex = [oracle_lib.Extractor(NFEAT, 1.2, 8, 20, 7) for _ in range(threads)]
    t0 = time.perf_counter()
    ex[0].time(frames[:1], 1)
    per = max(time.perf_counter() - t0, 1e-3)
    iters = max(2, min(200, int(seconds_budget / per)))

    def run(i):
        return ex[i].time(frames[i % len(frames):i % len(frames) + 1], iters)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as pool:
        list(pool.map(run, range(threads)))
    dt = time.perf_counter() - t0
    return threads * iters / dt, threads * iters


def cpu_protocol(seconds):
    """BASELINE.md section 3: oracle -O2 and -O1, 1 thread and A = 2/4/8 pinned threads, median + p95, each matcher."""
    out = {}
    for variant in ("O2", "O1"):
        env = dict(os.environ)
        env["SWM_ORACLE_VARIANT"] = variant
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "cpu_baseline.py"), "--seconds", str(seconds)],
                               capture_output=True, text=True, timeout=240, env=env)
            out[variant] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            out[variant] = {"error": str(e)[:200]}
    return out


def run_reference(args):
    from swarmmap_b200 import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    frames = synth.make_batch(max(8, threads), W, H, 20220410)
    for _ in range(max(args.warmup, 1) - 1):
        cpu_oracle_rate(frames, 0.5, threads)
    rates, n_total = [], 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r, n = cpu_oracle_rate(frames, 4.0, threads)
        rates.append(r)
        n_total += n
    dt = time.perf_counter() - t0
    value = statistics.median(rates)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frame": [W, H], "nfeatures": NFEAT},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{n_total} frames over {args.steps} steps, oracle -O2, one extractor per thread",
                             "cpu_model": cpu_model()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# =====================================================================================================================
class Ctx:
    """Per-rank state shared by the workloads."""

    def __init__(self, args):
        import torch
        self.torch = torch
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the ORB front-end has no CPU fallback")
        self.host = bind_numa(self.local_rank, self.world)
        torch.cuda.set_device(self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist
        self.dev = torch.device("cuda", self.local_rank)
        self.stream = torch.cuda.Stream(self.dev)
        torch.cuda.set_stream(self.stream)
        self.sptr = C.c_void_p(self.stream.cuda_stream)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, times_ms, counts=()):
        """max over ranks of the times, sum over ranks of the counts."""
        torch = self.torch
        t = torch.tensor(list(times_ms), dtype=torch.float64, device=self.dev)
        c = torch.tensor(list(counts) or [0.0], dtype=torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(c, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()], [float(x) for x in c.tolist()]


def h2d_ceiling(ctx, h2d_bytes, d2h_bytes):
    """What this box can move: plain pinned cudaMemcpyAsync on every rank at the same time, host->device alone and
    together with the device->host share of the end-to-end path (same byte ratio).  GB/s per GPU."""
    torch = ctx.torch
    n_h = 256 << 20
    n_d = max(1 << 20, int(n_h * d2h_bytes / h2d_bytes))
    hp = torch.empty(n_h, dtype=torch.uint8).pin_memory()
    dp = torch.empty(n_h, dtype=torch.uint8, device=ctx.dev)
    hq = torch.empty(n_d, dtype=torch.uint8).pin_memory()
    dq = torch.empty(n_d, dtype=torch.uint8, device=ctx.dev)
    s1, s2 = torch.cuda.Stream(ctx.dev), torch.cuda.Stream(ctx.dev)
    out = {}
    for name, both in (("h2d_alone_gbs", False), ("h2d_with_d2h_gbs", True)):
        for timed in (False, True):
            ctx.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 6 if timed else 2
            with torch.cuda.stream(s1):
                a.record(s1)
                for _ in range(reps):
                    dp.copy_(hp, non_blocking=True)
                b.record(s1)
            if both:
                with torch.cuda.stream(s2):
                    for _ in range(reps):
                        hq.copy_(dq, non_blocking=True)
            ctx.barrier()
            if timed:
                out[name] = reps * n_h / (a.elapsed_time(b) * 1e-3) / 1e9
    return out


class ExtractBench:
    """Device-resident and end-to-end extraction throughput for one frame size / feature count."""

    def __init__(self, ctx, frames, nfeat, B, handle_batch=64, nh=4):
        torch = ctx.torch
        from swarmmap_b200.orb import ORBextractor, KP_DTYPE
        self.ctx, self.B = ctx, B
        self.h, self.w = frames.shape[1], frames.shape[2]
        reps = (B + len(frames) - 1) // len(frames)
        self.h_img = torch.from_numpy(frames).repeat(reps, 1, 1)[:B].contiguous().pin_memory()
        self.d_img = self.h_img.to(ctx.dev)
        self.nh = nh if B % (nh * handle_batch) == 0 else 1
        self.hb = handle_batch if B % (self.nh * handle_batch) == 0 else B
        self.dex = [ORBextractor(nfeat, 1.2, 8, 20, 7, device=ctx.local_rank, max_batch=self.hb) for _ in range(self.nh)]
        self.cap = self.dex[0].max_keypoints()
        self.d_kps = torch.empty((B, self.cap, 7), dtype=torch.float32, device=ctx.dev)
        self.d_desc = torch.empty((B, self.cap, 32), dtype=torch.uint8, device=ctx.dev)
        self.d_n = torch.zeros(B, dtype=torch.int32, device=ctx.dev)
        self.wstreams = [torch.cuda.Stream(ctx.dev) for _ in range(self.nh)]
        self.wptrs = [C.c_void_p(ws.cuda_stream) for ws in self.wstreams]
        self.KP = KP_DTYPE
        self.nfeat = nfeat
        self.launches = 0

    def step_device(self):
        """One pass over the B resident frames: chunks of `hb` frames round-robin over the handles / streams, as
        co-located agents would run (one handle's quadtree / describe tail overlaps another's pyramid / FAST)."""
        w, h, hb = self.w, self.h, self.hb
        for c in range(self.B // hb):
            i, f0 = c % self.nh, c * hb
            self.dex[i].extract_batch_device(self.d_img[f0:].data_ptr(), hb, w, h, w, w * h, self.d_kps[f0:].data_ptr(),
                                             self.d_desc[f0:].data_ptr(), self.cap, self.d_n[f0:].data_ptr(), self.wptrs[i])
            self.launches += self.dex[i].last_launches()

    def time_device(self, steps, warmup):
        torch, ctx = self.ctx.torch, self.ctx
        for _ in range(warmup):
            self.step_device()
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ctx.stream)
        for ws in self.wstreams:
            ws.wait_event(e0)
        self.launches = 0   # kernels launched by the timed steps
        for _ in range(steps):
            self.step_device()
        for ws in self.wstreams:
            done = torch.cuda.Event()
            done.record(ws)
            ctx.stream.wait_event(done)
        e1.record(ctx.stream)
        ctx.barrier()
        return e0.elapsed_time(e1), int(self.d_n.sum().item())

    def setup_e2e(self, nslot=8, eb=32):
        torch = self.ctx.torch
        from swarmmap_b200.orb import ORBextractor
        self.nslot, self.eb = nslot, min(eb, self.B)
        self.exs = [ORBextractor(self.nfeat, 1.2, 8, 20, 7, device=self.ctx.local_rank, max_batch=self.eb) for _ in range(nslot)]
        self.h_np = self.h_img.numpy()
        self.outs = []
        for _ in range(nslot):
            k = torch.empty((self.eb, self.cap, 7), dtype=torch.float32).pin_memory()
            d = torch.empty((self.eb, self.cap, 32), dtype=torch.uint8).pin_memory()
            n = torch.zeros(self.eb, dtype=torch.int32).pin_memory()
            self.outs.append((k.numpy().view(self.KP).reshape(self.eb, self.cap), d.numpy(), n.numpy(), (k, d, n)))
        self.chunks = [(i, min(self.eb, self.B - i)) for i in range(0, self.B, self.eb)]

    def run_e2e(self, steps):
        """`steps` passes over the B pinned host frames as one stream of chunks: each chunk is uploaded, extracted and its
        keypoints / descriptors / counts downloaded; a slot is synchronised (and its result consumed on the host) only
        when it is reused, and everything is drained at the end."""
        total, pending, ci = 0, [None] * self.nslot, 0
        for _ in range(steps):
            for f0, nb in self.chunks:
                s = ci % self.nslot
                ci += 1
                if pending[s] is not None:
                    self.exs[s].sync()
                    total += int(self.outs[s][2][:pending[s]].sum())
                self.exs[s].extract_batch_async(self.h_np[f0:f0 + nb], (self.outs[s][0][:nb], self.outs[s][1][:nb], self.outs[s][2][:nb]))
                pending[s] = nb
        for s in range(self.nslot):
            if pending[s] is not None:
                self.exs[s].sync()
                total += int(self.outs[s][2][:pending[s]].sum())
        return total

    def time_e2e(self, steps, warmup):
        self.run_e2e(warmup)
        self.ctx.barrier()
        t0 = time.perf_counter()
        kp = self.run_e2e(steps)
        self.ctx.torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, kp

    def bytes_per_frame(self):
        return self.w * self.h, self.cap * (28 + 32) + 4


def headline_frames(batch, rank=0):
    """The headline's distinct synthetic frames (at most 512, tiled to the batch: inputs >> L2); frame i of the batch
    is frames[i % len(frames)]."""
    from swarmmap_b200 import synth
    return synth.make_batch(min(batch, 512), W, H, 20220410 + rank)


DUMP_FRAMES = 256    # x at most ~1030 keypoints x (7 + 32) float32 per frame: about 41 MB
DUMP_BYTES = 64 << 20


def dump_outputs(eb, out_dir):
    """Writes the device-resident path's outputs of its last timed step for a fixed, seeded sample of DUMP_FRAMES
    frames of the batch (every frame when the batch is smaller), as float32 arrays:
      frames.npy       (S,)        batch indices of the sample, ascending
      n_keypoints.npy  (S,)        keypoints per frame
      keypoints.npy    (sum n, 7)  x, y, size, angle, response, octave, class_id (KP_DTYPE order; the integers are exact)
      descriptors.npy  (sum n, 32) descriptor bytes
    Keypoints and descriptors are the frames' valid rows, concatenated in sample order."""
    torch = eb.ctx.torch
    idx = np.sort(np.random.default_rng(0).choice(eb.B, min(eb.B, DUMP_FRAMES), replace=False))
    sel = torch.from_numpy(idx).to(eb.ctx.dev)
    n = eb.d_n[sel].cpu().numpy()
    m = max(int(n.max()), 1)
    kps = eb.d_kps[sel, :m].cpu().numpy().view(eb.KP).reshape(len(idx), m)
    desc = eb.d_desc[sel, :m].cpu().numpy()
    kp = np.concatenate([k[:c] for k, c in zip(kps, n)])
    out = {"frames": idx.astype(np.float32), "n_keypoints": n.astype(np.float32),
           "keypoints": np.stack([kp[f].astype(np.float32) for f in eb.KP.names], 1),
           "descriptors": np.concatenate([d[:c] for d, c in zip(desc, n)]).astype(np.float32)}
    assert sum(a.nbytes for a in out.values()) <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------- config 2
def workload_kitti(ctx, cpu):
    """BASELINE config 2: KITTI-shaped 1241x376 sequence, extraction at 2000 features and the monocular initialiser's
    matcher SearchForInitialization(F_0, F_k, prev, matches, 100), ORBmatcher(0.9, true), k = 1..10 with vbPrevMatched
    carried from call to call (Tracking.cc:470-472), frames extracted with 4000 features (Tracking.cc:123)."""
    torch = ctx.torch
    from swarmmap_b200 import synth
    from swarmmap_b200.matcher import Frame, ORBmatcher, ResidentFrame
    from swarmmap_b200.orb import ORBextractor
    wk, hk = 1241, 376
    seq = synth.make_sequence(100, wk, hk, 20220405 + 1000 * ctx.rank)
    eb = ExtractBench(ctx, seq, 2000, 1000, handle_batch=50, nh=4)
    ms_dev, nkp = eb.time_device(4, 3)
    eb.setup_e2e(8, 25)
    ms_e2e, nkp2 = eb.time_e2e(4, 2)
    assert nkp2 == 4 * nkp, (nkp2, nkp)
    h2d, d2h = eb.bytes_per_frame()
    # ---- init matching: chains s = 0..P-1 over the 100-frame sequence: F_0 = frame s, F_k = frame s + k
    ex4k = ORBextractor(4000, 1.2, 8, 20, 7, device=ctx.local_rank, max_batch=100)
    kps, desc, n = ex4k.extract_batch(seq)
    sf = ex4k.GetScaleFactors()
    fs = [Frame.from_keypoints(kps[i, :n[i]].copy(), desc[i, :n[i]].copy(), wk, hk, sf) for i in range(100)]
    res = [ResidentFrame(ctx.local_rank).upload(f) for f in fs]
    P, K = 89, 10
    m = ORBmatcher(0.9, True, device=ctx.local_rank)

    def run_chains(store=None):
        prev = [np.stack([fs[s].x, fs[s].y], 1).astype(np.float32).copy() for s in range(P)]
        dev_ms = 0.0
        for k in range(1, K + 1):
            got = m.SearchForInitializationBatch([(res[s], res[s + k], prev[s]) for s in range(P)], 100)
            dev_ms += float(m._lib.swm_matcher_last_device_ms(m._h))
            if store is not None:
                store.append(got)
        return dev_ms

    run_chains()
    ctx.barrier()
    store = []
    t0 = time.perf_counter()
    dev_ms = run_chains(store)
    wall_ms = (time.perf_counter() - t0) * 1e3
    # parity spot-check inside the run: chain 0 and chain 37 against the oracle, all ten calls
    parity = None
    if cpu:
        import oracle_lib
        ok, t_cpu = True, 0.0
        for s in (0, 37):
            prev = np.stack([fs[s].x, fs[s].y], 1).astype(np.float32).copy()
            for k in range(1, K + 1):
                t1 = time.perf_counter()
                on, om12, prev = oracle_lib.search_for_initialization(fs[s], fs[s + k], prev, 100, 0.9, True)
                t_cpu += time.perf_counter() - t1
                gn, gm12 = store[k - 1][s]
                ok = ok and gn == on and np.array_equal(gm12, om12)
        parity = {"checked": "chains 0 and 37, k = 1..10: match count and vnMatches12 against the oracle", "identical": bool(ok),
                  "cpu_oracle_ms_per_call": 1e3 * t_cpu / (2 * K)}
        assert ok, "SearchForInitialization batch differs from the oracle"
    (ms_dev, ms_e2e, dev_ms, wall_ms), (frames_n, calls) = ctx.reduce([ms_dev, ms_e2e, dev_ms, wall_ms], [4.0 * 1000, float(P * K)])
    return {
        "config": {"workload": "BASELINE config 2: KITTI-shaped 1241x376 synthetic sequence (100 frames), ORBextractor(2000, 1.2, 8, 20, 7) "
                               "extract+describe; SearchForInitialization(F_0, F_k, window 100), ORBmatcher(0.9, true), k = 1..10 on "
                               "4000-feature frames", "frame": [wk, hk], "chains_per_gpu": P},
        "extract": {"metric": METRIC, "unit": UNIT, "value": frames_n / (ms_dev * 1e-3),
                    "e2e": {"value": frames_n / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_frame": h2d, "d2h_bytes_per_frame": d2h},
                    "keypoints_per_frame": nkp / 1000.0,
                    "roofline_note": "same kernels as the headline; algorithmic pyramid+FAST bytes 5 057 039 per frame"},
        "init_matching": {"metric": "search_for_initialization_calls_per_sec", "unit": "calls/s",
                          "value": calls / (dev_ms * 1e-3), "e2e": {"value": calls / (wall_ms * 1e-3), "unit": "calls/s"},
                          "note": f"{P} independent chains per GPU advance together: one batched call per k (resident frames, "
                                  "vbPrevMatched up and vnMatches12 down every call); value = CUDA-event time of the six kernels, "
                                  "e2e = host clock around the ten calls", "keypoints_per_frame": float(np.mean(n)),
                          "parity": parity},
    }


# ---------------------------------------------------------------------------------------------------- configs 3 / 4
def workload_tracking(ctx, cpu):
    """BASELINE configs 3 and 4: the per-frame tracking matchers of agents pinned to this GPU.  One "tracking step" =
    one frame of one agent: ORBextractor::operator() -> Frame (undistort + grid on the device) -> [ComputeBoW ->
    SearchByBoW(KF = previous frame, F), ratio 0.7 (Tracking.cc:619-626)] -> SearchByProjection(cur, last, 15)
    (Tracking.cc:715-737) -> SearchByProjection(F, local map points, th 1), ORBmatcher(0.8) (Tracking.cc:998-1005).
    Map points: the previous frame's keypoints, projected with the generator's ground-truth motion + 1 px noise; the
    local map adds the points of the frame before.  P agents advance together: every stage is one batched call."""
    torch = ctx.torch
    from swarmmap_b200 import _lib, synth
    from swarmmap_b200._lib import BowJob, BowOut, FeatVec, WindowJob, WindowQuery, ptr
    from swarmmap_b200.bow import ORBVocabulary
    from swarmmap_b200.matcher import Camera, ORBmatcher, ResidentFrame
    from swarmmap_b200.orb import ORBextractor, KP_DTYPE
    lib = _lib.load()
    S, T, P = 8, 10, 128                      # sequences, timed steps, agents per GPU
    seqs, warps = [], []
    for s in range(S):
        fr, hs = synth.make_sequence(T + 2 + P // S, W, H, 20220406 + s + 100 * ctx.rank, return_h=True)
        seqs.append(fr)
        warps.append(hs)
    ex = ORBextractor(NFEAT, 1.2, 8, 20, 7, device=ctx.local_rank, max_batch=P)
    cap = ex.max_keypoints()
    sf = ex.GetScaleFactors()
    cam = Camera(*EUROC_CAM)
    bounds = cam.bounds(W, H, ctx.local_rank)
    vblob = synth.make_vocabulary(10, 5, seed=20220407)
    voc = ORBVocabulary(vblob, device=ctx.local_rank)
    m7, m9, m8 = (ORBmatcher(r, o, device=ctx.local_rank) for r, o in ((0.7, True), (0.9, True), (0.8, True)))

    def frame_of(a, t):   # agent a at step t looks at frame (a // S) + t of sequence a % S
        return a % S, a // S + t

    # pinned host frames per step, and the extraction of every frame any step touches (setup, untimed)
    h_steps = [torch.from_numpy(np.stack([seqs[frame_of(a, t)[0]][frame_of(a, t)[1]] for a in range(P)])).pin_memory()
               for t in range(T + 2)]
    feats = []
    for t in range(T + 2):
        k, d, n = ex.extract_batch(h_steps[t].numpy())
        feats.append((k.copy(), d.copy(), n.copy()))
    rng = np.random.default_rng(7 + ctx.rank)

    def warp_points(s, i_from, i_to, x, y):
        """frame i_from pixel -> canvas -> frame i_to pixel (the generator's affine maps are frame -> canvas)."""
        A, B2 = np.vstack([warps[s][i_from], [0, 0, 1]]), np.vstack([warps[s][i_to], [0, 0, 1]])
        Mx = np.linalg.inv(B2) @ A
        return (Mx[0, 0] * x + Mx[0, 1] * y + Mx[0, 2]).astype(np.float32), (Mx[1, 0] * x + Mx[1, 1] * y + Mx[1, 2]).astype(np.float32)

    # two sets of resident frames alternate between "current" and "last"
    rf = [[ResidentFrame(ctx.local_rank) for _ in range(P)] for _ in range(2)]
    rf_h = [(C.c_void_p * P)(*[f._h for f in rf[b]]) for b in range(2)]
    keep = []

    def window_jobs(t, mode):
        """Prebuilt swm_window_job array of step t (cur = step t frames in rf[t % 2]); mode 0 = SearchByProjection(cur,
        last, 15), mode 1 = SearchByProjection(F, local map points, th 1)."""
        arr = (WindowJob * P)()
        outs = []
        for a in range(P):
            s, i = frame_of(a, t)
            srcs = [t - 1] if mode == 0 else [t - 1, t - 2]
            us, vs, descs, octs, angs = [], [], [], [], []
            for tt in srcs:
                k, d, n = feats[tt]
                kk = k[a, :n[a]]
                x, y = warp_points(s, frame_of(a, tt)[1], i, kk["x"], kk["y"])
                us.append(x + rng.normal(0, 1.0, len(x)).astype(np.float32))
                vs.append(y + rng.normal(0, 1.0, len(x)).astype(np.float32))
                descs.append(d[a, :n[a]])
                octs.append(kk["octave"])
                angs.append(kk["angle"])
            u, v = np.concatenate(us), np.concatenate(vs)
            desc = np.ascontiguousarray(np.concatenate(descs))
            octv = np.concatenate(octs).astype(np.int32)
            ang = np.ascontiguousarray(np.concatenate(angs), np.float32)
            M = len(u)
            valid = ((u >= bounds[0]) & (u <= bounds[1]) & (v >= bounds[2]) & (v <= bounds[3])).astype(np.uint8)
            if mode == 0:
                radius = (np.float32(15.0) * sf[octv]).astype(np.float32)
                lo, hi = (octv - 1).astype(np.int32), (octv + 1).astype(np.int32)
                th_dist, ratio_mode, nnr, ori = 100, 0, 0.9, 1
            else:
                radius = (np.float32(2.5) * sf[octv]).astype(np.float32)   # RadiusByViewingCos(1.0) * th(1) (:123-128)
                lo, hi = (octv - 1).astype(np.int32), octv.copy()
                th_dist, ratio_mode, nnr, ori = 100, 1, 0.8, 0
            blocks = np.ones(M, np.uint8)
            q = WindowQuery(M, ptr(desc).value, ptr(u).value, ptr(v).value, ptr(radius).value, ptr(lo).value, ptr(hi).value,
                            ptr(valid).value, ptr(ang).value, ptr(blocks).value)
            asg = np.full(cap, -1, np.int32)
            keep.extend([u, v, desc, octv, ang, valid, radius, lo, hi, blocks, q, asg])
            arr[a] = WindowJob(None, rf[t % 2][a]._h, C.addressof(q), None, th_dist, ratio_mode, nnr, ori, ptr(asg).value, 0)
            outs.append((asg, dict(desc=desc, u=u, v=v, radius=radius, lo=lo, hi=hi, valid=valid, ang=ang, th=th_dist,
                                   rm=ratio_mode, nnr=nnr, ori=ori)))
        return arr, outs

    steps = list(range(2, T + 2))
    proj_jobs = {t: window_jobs(t, 0) for t in steps}
    map_jobs = {t: window_jobs(t, 1) for t in steps}
    # BoW: per-set output slabs of the vocabulary transform, FeatVec views into them, prebuilt job arrays
    bow = []
    for b in range(2):
        o = dict(word_ids=np.zeros((P, cap), np.uint32), word_values=np.zeros((P, cap), np.float64), n_words=np.zeros(P, np.int32),
                 node_ids=np.zeros((P, cap), np.uint32), node_offsets=np.zeros((P, cap + 1), np.int32),
                 feats=np.zeros((P, cap), np.uint32), n_nodes=np.zeros(P, np.int32))
        view = BowOut(*[ptr(o[k]).value for k in ("word_ids", "word_values", "n_words", "node_ids", "node_offsets", "feats", "n_nodes")])
        fvs = (FeatVec * P)()
        for a in range(P):
            fvs[a] = FeatVec(0, ptr(o["node_ids"][a]).value, ptr(o["node_offsets"][a]).value, ptr(o["feats"][a]).value)
        bow.append((o, view, fvs))
    valid_all = np.ones(cap, np.uint8)
    bow_out = [[np.full(cap, -1, np.int32) for _ in range(P)] for _ in range(2)]
    bow_jobs = []
    for b in range(2):   # cur set b, KF = the other set
        arr = (BowJob * P)()
        for a in range(P):
            arr[a] = BowJob(None, None, rf[1 - b][a]._h, rf[b][a]._h, C.addressof(bow[1 - b][2][a]), C.addressof(bow[b][2][a]),
                            ptr(valid_all).value, None, 0, 0.7, 1, ptr(bow_out[b][a]).value, 0)
        bow_jobs.append(arr)
    # extraction outputs (pinned) of the timed loop
    o_k = torch.empty((P, cap, 7), dtype=torch.float32).pin_memory()
    o_d = torch.empty((P, cap, 32), dtype=torch.uint8).pin_memory()
    o_n = torch.zeros(P, dtype=torch.int32).pin_memory()
    out_np = (o_k.numpy().view(KP_DTYPE).reshape(P, cap), o_d.numpy(), o_n.numpy())
    bptr = ptr(np.ascontiguousarray(bounds, np.float32))
    b_np = np.ascontiguousarray(bounds, np.float32)
    stage = {"extract": 0.0, "frames": 0.0, "bow_transform": 0.0, "search_by_bow": 0.0, "proj_last": 0.0, "proj_map": 0.0}
    dev_ms = {"search_by_bow": 0.0, "proj_last": 0.0, "proj_map": 0.0}

    def check(rc, h, what):
        if rc != 0:
            raise RuntimeError(f"{what}: {lib.swm_matcher_last_error(h)}")

    def do_step(t, with_bow, acc):
        b = t % 2
        t0 = time.perf_counter()
        ex.extract_batch_async(h_steps[t].numpy(), out_np)
        ex.sync()
        t1 = time.perf_counter()
        rc = lib.swm_frames_from_extractor(rf_h[b], P, ex._h, None, C.byref(cam.c), ptr(b_np))
        if rc != 0:
            raise RuntimeError("swm_frames_from_extractor failed")
        t2 = time.perf_counter()
        if with_bow:
            rc = lib.swm_bow_transform(voc._h, ptr(out_np[1]), ptr(out_np[2]), P, cap, 4, C.byref(bow[b][1]))
            if rc != 0:
                raise RuntimeError("swm_bow_transform failed")
            nn = bow[b][0]["n_nodes"]
            for a in range(P):
                bow[b][2][a].n_nodes = int(nn[a])
            t3 = time.perf_counter()
            if t > 2:   # the keyframe's FeatureVector exists from the previous step on
                check(lib.swm_match_bow_batch(m7._h, bow_jobs[b], P), m7._h, "swm_match_bow_batch")
                if acc:
                    dev_ms["search_by_bow"] += float(lib.swm_matcher_last_device_ms(m7._h))
            t4 = time.perf_counter()
        else:
            t3 = t4 = t2
        check(lib.swm_match_window_batch(m9._h, proj_jobs[t][0], P), m9._h, "swm_match_window_batch")
        if acc:
            dev_ms["proj_last"] += float(lib.swm_matcher_last_device_ms(m9._h))
        t5 = time.perf_counter()
        check(lib.swm_match_window_batch(m8._h, map_jobs[t][0], P), m8._h, "swm_match_window_batch")
        if acc:
            dev_ms["proj_map"] += float(lib.swm_matcher_last_device_ms(m8._h))
        t6 = time.perf_counter()
        if acc:
            for k, dt in zip(("extract", "frames", "bow_transform", "search_by_bow", "proj_last", "proj_map"),
                             (t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4, t6 - t5)):
                stage[k] += dt * 1e3

    def reset_outputs():
        for t in steps:
            for jobs in (proj_jobs[t], map_jobs[t]):
                for asg, _ in jobs[1]:
                    asg.fill(-1)

    results = {}
    for variant, with_bow in (("projection_only", False), ("with_bow", True)):
        for k in stage:
            stage[k] = 0.0
        for k in dev_ms:
            dev_ms[k] = 0.0
        for t in steps[:3]:
            do_step(t, with_bow, False)
        reset_outputs()
        ctx.barrier()
        t0 = time.perf_counter()
        for t in steps:
            do_step(t, with_bow, True)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        results[variant] = (wall, dict(stage), dict(dev_ms))
    # ---- parity spot-check: agent 5 at the last step, all three matchers against the oracle
    parity = None
    if cpu:
        import oracle_lib
        from swarmmap_b200.matcher import FeatureVector, Frame
        t, a = steps[-1], 5
        k, d, n = feats[t]
        und = oracle_lib.undistort_points(np.stack([k[a, :n[a]]["x"], k[a, :n[a]]["y"]], 1).astype(np.float32),
                                          np.array(EUROC_CAM, np.float32))
        curF = Frame(und[:, 0], und[:, 1], k[a, :n[a]]["octave"], k[a, :n[a]]["angle"], d[a, :n[a]],
                     (float(bounds[0]), float(bounds[2]), float(bounds[1]), float(bounds[3])), sf)
        ok = True
        for jobs in (proj_jobs[t], map_jobs[t]):
            asg, q = jobs[1][a]
            on, oasg = oracle_lib.match_window(curF, q["desc"], q["u"], q["v"], q["radius"], q["lo"], q["hi"], q["valid"],
                                               np.ones(len(q["u"]), np.uint8), q["th"], q["rm"], q["nnr"], bool(q["ori"]), q["ang"])
            ok = ok and np.array_equal(asg[:curF.N], oasg) and int(jobs[0][a].nmatches) == on
        kp, dp, npv = feats[t - 1]
        undp = oracle_lib.undistort_points(np.stack([kp[a, :npv[a]]["x"], kp[a, :npv[a]]["y"]], 1).astype(np.float32),
                                           np.array(EUROC_CAM, np.float32))
        kfF = Frame(undp[:, 0], undp[:, 1], kp[a, :npv[a]]["octave"], kp[a, :npv[a]]["angle"], dp[a, :npv[a]], curF.bounds, sf)
        ov = oracle_lib.Vocabulary(vblob)
        f1 = ov.transform(dp[a, :npv[a]], 4)
        f2 = ov.transform(d[a, :n[a]], 4)
        fv1, fv2 = FeatureVector.__new__(FeatureVector), FeatureVector.__new__(FeatureVector)
        fv1.node_ids, fv1.offsets, fv1.feats = f1[2], f1[3], f1[4]
        fv2.node_ids, fv2.offsets, fv2.feats = f2[2], f2[3], f2[4]
        on, oout = oracle_lib.search_by_bow(kfF, fv1, np.ones(kfF.N, np.uint8), curF, fv2, None, 0, 0.7, True)
        ok = ok and np.array_equal(bow_out[t % 2][a][:curF.N], oout) and int(bow_jobs[t % 2][a].nmatches) == on
        parity = {"checked": f"agent {a}, last step: SearchByProjection(cur,last), SearchByProjection(F,map points) and SearchByBoW "
                             "indices + counts against the oracle (resident undistorted frame vs oracle undistortion)",
                  "identical": bool(ok)}
        assert ok, "tracking-step matchers differ from the oracle"
    rec = {"config": {"workload": "BASELINE configs 3 and 4: per-frame tracking step of agents pinned to the GPU, 752x480, 1000 features: "
                                  "extract + resident Frame + [ComputeBoW + SearchByBoW(KF,F) 0.7] + SearchByProjection(cur,last,15) + "
                                  "SearchByProjection(F, local map points, th 1)", "agents_per_gpu": P, "steps_timed": len(steps),
                      "vocabulary": f"synthetic k=10 L=5 ({voc.n_nodes} nodes), levelsup 4",
                      "map_points_per_frame": "previous frame's keypoints (projection), previous two frames' (local map)"},
           "metric": "tracking_steps_per_sec", "unit": "steps/s", "parity": parity, "variants": {}}
    for variant, (wall, st, dv) in results.items():
        (wall_r,), (steps_n,) = ctx.reduce([wall], [float(P * len(steps))])
        rec["variants"][variant] = {
            "e2e": {"value": steps_n / (wall_r * 1e-3), "unit": "steps/s",
                    "note": "host clock around the synchronised loop: pinned host frames in, keypoints + descriptors + every match array out"},
            "stage_ms_per_step_of_%d_agents" % P: {k: v / len(steps) for k, v in st.items()},
            "matcher_kernels_device_ms_per_step": {k: v / len(steps) for k, v in dv.items()},
        }
    # device-timed value of the tracking step = extraction (CUDA events, headline kernels) + matcher kernels (CUDA events)
    po = rec["variants"]["projection_only"]
    wb = rec["variants"]["with_bow"]
    rec["value_note"] = ("value = agents x steps / (device time of extraction at the headline rate + CUDA-event time of the matcher "
                         "kernels); the headline's frames/s gives the extraction share")
    rec["_matcher_ms"] = {"projection_only": sum(po["matcher_kernels_device_ms_per_step"].values()),
                          "with_bow": sum(wb["matcher_kernels_device_ms_per_step"].values())}
    rec["_agents"] = P
    return rec


# ---------------------------------------------------------------------------------------------------- config 5
def workload_place(ctx, cpu):
    """BASELINE config 5 as written: Q = 2000 descriptors of one keyframe against 100 000 keyframes x 256 descriptors
    (25.6 M, 819 MB), bytes i.i.d. uniform (seed 99) with 1 % of the keyframes planted as noisy copies of Q (10 % of the
    bits flipped), STRONG-scaled: the database is partitioned by keyframe id over the ranks, every rank scans its shard
    (tcgen05 kernel), one NCCL all-gather of the (2000, 2) key blocks, merge + votes."""
    torch = ctx.torch
    from swarmmap_b200 import _lib, place
    NQ, DPK, NKF = 2000, 256, 100000
    parts = place.partition(NKF, ctx.world)
    first_kf, n_kf = parts[ctx.rank]
    gq = torch.Generator(device=ctx.dev)
    gq.manual_seed(99)
    q = torch.randint(0, 256, (NQ, 32), dtype=torch.uint8, device=ctx.dev, generator=gq)
    gen = torch.Generator(device=ctx.dev)
    gen.manual_seed(990 + ctx.rank)
    db = torch.randint(0, 256, (n_kf * DPK, 32), dtype=torch.uint8, device=ctx.dev, generator=gen)
    # planted keyframes: every 100th keyframe id (globally) holds noisy copies of 256 consecutive query descriptors
    planted = [kf for kf in range(first_kf, first_kf + n_kf) if kf % 100 == 0]
    for kf in planted:
        j0 = (kf * 7) % (NQ - DPK)
        flips = torch.rand((DPK, 256), device=ctx.dev, generator=gen) < 0.10
        bits = torch.zeros((DPK, 32), dtype=torch.uint8, device=ctx.dev)
        for bit in range(8):
            bits |= (flips[:, bit::8].to(torch.uint8) << bit)
        lo = (kf - first_kf) * DPK
        db[lo:lo + DPK] = q[j0:j0 + DPK] ^ bits
    shard = place.PlaceShard(db, DPK, first_kf, device=ctx.local_rank)
    comm = nccl = None
    if ctx.world > 1:
        comm, nccl = place.nccl_comm_from_torch(ctx.local_rank)

    # N > 1: the exchange runs over peer memory inside the merge kernel (swm_db_query_peers); the NCCL form
    # (swm_db_query_sharded: scan, ncclAllGather, merge) is timed beside it and must give the same keys and votes
    peers = False
    if ctx.world > 1:
        try:
            shard.enable_peers(nq_max=NQ)
            peers = True
        except Exception as e:  # no peer access between these GPUs: the NCCL form is the product path
            if ctx.rank == 0:
                print(f"place: peer-memory exchange unavailable ({e}); NCCL exchange", file=sys.stderr)
        (_,), (npeers,) = ctx.reduce([0.0], [1.0 if peers else 0.0])
        peers = int(npeers) == ctx.world  # a collective: all ranks or none

    def query_nccl():
        return shard.query_sharded(q, comm, ctx.world, 2, 50)

    def query():
        if ctx.world > 1:
            return shard.query_peers(q, 2, 50) if peers else query_nccl()
        return shard.query(q, 2, 50)

    def timed(fn):
        for _ in range(2):
            fn()
        ctx.barrier()
        reps_ = 10
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps_):
            out = fn()
        b.record()
        ctx.barrier()
        return a.elapsed_time(b) / reps_, out

    reps = 10
    ms, (keys, votes) = timed(query)
    ms_nccl, same_as_nccl = None, None
    if ctx.world > 1 and peers:
        ms_nccl, (keys_n, votes_n) = timed(query_nccl)
        same_as_nccl = bool(torch.equal(keys, keys_n) and torch.equal(votes, votes_n))
    # e2e: host query descriptors in, host keys + votes out
    hq = q.cpu().pin_memory()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        dq = hq.to(ctx.dev, non_blocking=True)
        if ctx.world > 1:
            k2, v2 = shard.query_peers(dq, 2, 50) if peers else shard.query_sharded(dq, comm, ctx.world, 2, 50)
        else:
            k2, v2 = shard.query(dq, 2, 50)
        k_h, v_h = k2.cpu(), v2.cpu()
    wall = (time.perf_counter() - t0) * 1e3 / reps
    # ---- checks inside the run: votes land on the planted keyframes; sampled queries against the oracle
    v = votes.cpu().numpy()
    d0, i0 = place.unpack_keys(keys[:, 0].cpu())
    low = d0.numpy() <= 50
    is_planted = np.zeros(n_kf, bool)
    is_planted[np.array(planted, np.int64) - first_kf] = True
    # every query votes once, for the keyframe of its GLOBAL best match: all votes must land on planted keyframes and
    # (summed over the shards) there must be exactly one per query whose best distance is <= TH_LOW
    (_,), (votes_total, stray) = ctx.reduce([0.0], [float(v.sum()), float(v[~is_planted].sum())])
    votes_ok = stray == 0 and int(votes_total) == int(low.sum()) and low.mean() > 0.8
    frac_low = float(low.mean())
    parity = {"votes_on_planted_keyframes": bool(votes_ok), "queries_with_best_distance_le_50": frac_low}
    if cpu and ctx.rank == 0:
        import oracle_lib
        sel = np.arange(0, NQ, 97)[:16]
        sub = db[:2048 * DPK].cpu().numpy()
        keys_sub, _ = place.PlaceShard(sub, DPK, first_kf, device=ctx.local_rank).query_local(q[sel], 2, 50)
        dd, ii = place.unpack_keys(keys_sub.cpu())
        obf = oracle_lib.bruteforce_top2(q[sel].cpu().numpy(), sub)
        parity["oracle_sample"] = {"checked": "16 queries x the first 2048 keyframes (524 288 descriptors): top-2 distance and index",
                                   "identical": bool(np.array_equal(dd.numpy()[:, 0], obf[:, 0]) and np.array_equal(ii.numpy()[:, 0] - first_kf * DPK, obf[:, 1])
                                                     and np.array_equal(dd.numpy()[:, 1], obf[:, 2]) and np.array_equal(ii.numpy()[:, 1] - first_kf * DPK, obf[:, 3]))}
    assert votes_ok, "place-recognition votes do not single out the planted keyframes"
    peak = C.c_double(0)
    peak256 = C.c_double(0)
    lib = _lib.load()
    lib.swm_i8_peak(ctx.local_rank, 0, 4096, C.byref(peak))
    lib.swm_i8_peak(ctx.local_rank, 1, 4096, C.byref(peak256))
    if comm is not None:
        nccl.ncclCommDestroy(comm)
    (ms_r, wall_r, ms_nccl_r), (same_all,) = ctx.reduce([ms, wall, ms_nccl or 0.0], [1.0 if same_as_nccl in (None, True) else 0.0])
    if ctx.world > 1 and peers:
        parity["peer_exchange_identical_to_nccl_exchange"] = int(same_all) == ctx.world
    pairs = float(NQ) * NKF * DPK
    ops = pairs * 512 / (ms_r * 1e-3) / 1e12
    return {"config": {"workload": "BASELINE config 5: 2000 query descriptors x 100 000 keyframes x 256 descriptors (25.6 M, 819 MB), 1 % "
                                   "planted noisy copies, top-2 + per-keyframe votes, database sharded by keyframe id over the ranks",
                       "scaling": "strong", "n_gpus": ctx.world,
                       "exchange": ("none (one shard)" if ctx.world == 1 else
                                    "peer-memory stores of the (2000, 2) 64-bit key blocks + flags over NVLink inside the merge kernel "
                                    "(swm_db_query_peers: scan + ONE fused kernel)" if peers else
                                    "ncclAllGather of (2000, 2) 64-bit keys inside swm_db_query_sharded"),
                       "ms_per_query_batch_nccl_exchange": (ms_nccl_r if ctx.world > 1 and peers else None)},
            "metric": "hamming_matches_per_sec", "unit": "256-bit pairs/s", "value": pairs / (ms_r * 1e-3),
            "ms_per_query_batch": ms_r, "e2e": {"value": pairs / (wall_r * 1e-3), "unit": "256-bit pairs/s", "ms_per_query_batch": wall_r,
                                                "h2d_bytes_per_step": NQ * 32, "d2h_bytes_per_step": NQ * 16 + n_kf * 4},
            "kernel": "db_top2_umma_kernel (tcgen05 kind::i8, A in TMEM, accumulators in TMEM) + db_merge_kernel / db_merge_peers_kernel",
            "roofline": {"bound": "tensor", "unit": "TOP/s (int8)", "achieved": ops / ctx.world, "peak": max(peak.value, peak256.value),
                         "frac": ops / ctx.world / max(peak.value, peak256.value, 1e-9),
                         "issued": ops / ctx.world * 288.0 / 256.0,
                         "frac_issued": ops / ctx.world * 288.0 / 256.0 / max(peak.value, peak256.value, 1e-9),
                         "peak_source": "MEASURED on this GPU by swm_i8_peak (pure tcgen05 kind::i8 issue loops, no epilogue, one CTA per SM): "
                                        "the larger of 128x64x32 .ts with six accumulators in rotation (the scan's own shape) and 128x256x32 .ss; "
                                        "per GPU.  achieved = algorithmic ops (2 x 256 per pair), issued = what the kernel executes "
                                        "(2 x 288: the constant K block that turns the accumulator into the sort key)",
                         "peak_128x64x32_ts": peak.value, "peak_128x256x32_ss": peak256.value, "nominal_dense_int8": 4500.0},
            "parity": parity}


# =====================================================================================================================
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline, device-resident and end to end (the other workloads time fixed counts)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8192, help="frames per step per GPU (8192 x 20 steps = a timed region above 1 s)")
    ap.add_argument("--impl", default="swm", choices=["swm", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only", default="", help="comma list of workloads to run besides the headline (kitti,tracking,place); default all")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the headline's outputs of its last timed step (rank 0, sampled frames) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "swm":
        ap.error("--dump-outputs writes the outputs of --impl swm")
    args.warmup = max(args.warmup, 3) if args.impl == "swm" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return

    from swarmmap_b200 import build, synth
    if build.needs_build():
        raise SystemExit(f"{build.LIB} is missing or older than its sources: rebuild it (python -m swarmmap_b200.build)")
    from swarmmap_b200 import _lib
    from swarmmap_b200.orb import ORBextractor
    ctx = Ctx(args)
    torch = ctx.torch
    rank, world, B = ctx.rank, ctx.world, args.batch
    cpu = not args.no_cpu_baseline
    only = set(x for x in args.only.split(",") if x) or {"kitti", "tracking", "place"}

    # ---- headline: extraction of B frames per step
    frames = headline_frames(B, rank)
    distinct = len(frames)
    eb = ExtractBench(ctx, frames, NFEAT, B, handle_batch=256, nh=4)  # 256-frame calls round-robin over 4 handles / streams (64-frame calls: 151 k instead of 158 k frames/s)
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    ms_total, n_kp = eb.time_device(args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(eb, args.dump_outputs)
    launches = eb.launches
    eb.setup_e2e(8, 64)
    ms_e2e, kp_e2e = eb.time_e2e(args.steps, args.warmup)
    assert kp_e2e == n_kp * args.steps, (kp_e2e, n_kp, args.steps)  # the streamed path produced the same keypoints
    clocks = sampler.stop()
    h2d_pf, d2h_pf = eb.bytes_per_frame()
    ceiling = h2d_ceiling(ctx, h2d_pf, d2h_pf)

    # ---- per-stage device times and the roofline launch set (one 256-frame handle, events on the bench stream)
    SB = min(256, B)
    ex = ORBextractor(NFEAT, 1.2, 8, 20, 7, device=ctx.local_rank, max_batch=SB)
    ex.extract_batch_device(eb.d_img.data_ptr(), SB, W, H, W, W * H, eb.d_kps.data_ptr(), eb.d_desc.data_ptr(), eb.cap,
                            eb.d_n.data_ptr(), ctx.sptr)
    torch.cuda.synchronize()
    stage_ms = {}
    for name, mask in (("pyramid_border_blur", _lib.STAGE_PYRAMID), ("fast_both_passes", _lib.STAGE_NMS),
                       ("quadtree", _lib.STAGE_OCTREE), ("angle_describe", _lib.STAGE_DESCRIBE)):
        reps = 10
        ex.run_stage(mask, SB, ctx.sptr)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            ex.run_stage(mask, SB, ctx.sptr)
        b.record()
        torch.cuda.synchronize()
        stage_ms[name] = a.elapsed_time(b) / reps
    del ex

    # ---- the other BASELINE configs
    workloads = {}
    if "kitti" in only:
        workloads["config2_kitti"] = workload_kitti(ctx, cpu)
    if "tracking" in only:
        workloads["config34_tracking"] = workload_tracking(ctx, cpu)
    if "place" in only:
        workloads["config5_place"] = workload_place(ctx, cpu)

    # ---- single-call latencies of the drop-in API (rank 0, informational)
    latency = {}
    if rank == 0:
        ex1 = ORBextractor(NFEAT, 1.2, 8, 20, 7, device=ctx.local_rank, max_batch=1)
        for _ in range(5):
            ex1(frames[0])
        t0 = time.perf_counter()
        for i in range(50):
            ex1(frames[i % distinct])
        latency["single_frame_operator_ms"] = (time.perf_counter() - t0) / 50 * 1e3
        del ex1
        # stereo front-end (Frame::ComputeStereoMatches, Frame.cc:516-690): 32 rectified pairs per call, both views
        # resident from their extractors; informational, checked against the oracle on pair 0
        sl, sr = synth.make_stereo_pair(W, H, 20220421)
        SBT = 32
        exl = ORBextractor(NFEAT, 1.2, 8, 20, 7, device=ctx.local_rank, max_batch=SBT)
        exr = ORBextractor(NFEAT, 1.2, 8, 20, 7, device=ctx.local_rank, max_batch=SBT)
        kl, dl, nl = exl.extract_batch(np.repeat(sl[None], SBT, 0))
        kr, dr, nr = exr.extract_batch(np.repeat(sr[None], SBT, 0))
        bf, bl = 47.90639384423901, 47.90639384423901 / 458.654
        u, z = exl.stereo_match(exr, bf, bl, SBT)
        t0 = time.perf_counter()
        for _ in range(10):
            u, z = exl.stereo_match(exr, bf, bl, SBT)
        latency["stereo_match_ms_per_pair"] = (time.perf_counter() - t0) / 10 / SBT * 1e3
        latency["stereo_matches_per_pair"] = int((u[0, :nl[0]] >= 0).sum())
        if cpu:
            import oracle_lib

            def comp(ex):
                out = []
                for l in range(8):
                    buf = ex.debug_plane(0, l, 0).copy()
                    buf[19:-19, 19:-19] = ex.debug_plane(0, l, 1)
                    out.append(buf)
                return out
            sf_, isf_, _, _ = oracle_lib.scale_tables(1.2, 8)
            u0, z0, _ = oracle_lib.stereo_matches(kl[0, :nl[0]], dl[0, :nl[0]], kr[0, :nr[0]], dr[0, :nr[0]], comp(exl), comp(exr),
                                           sf_, isf_, bf, bl)
            latency["stereo_identical_to_oracle"] = bool(np.array_equal(u[0, :nl[0]].view(np.uint32), u0.view(np.uint32)) and
                                                         np.array_equal(z[0, :nl[0]].view(np.uint32), z0.view(np.uint32)))
        del exl, exr

    # ---- reduce over ranks (max time), rank 0 prints
    (ms_total, ms_e2e, ms_pf, c_h2d, c_both), (cnt,) = ctx.reduce(
        [ms_total, ms_e2e, stage_ms["pyramid_border_blur"] + stage_ms["fast_both_passes"], -ceiling["h2d_alone_gbs"],
         -ceiling["h2d_with_d2h_gbs"]], [float(n_kp)])
    c_h2d, c_both = -c_h2d, -c_both       # min over ranks
    frames_total = world * B * args.steps
    value = frames_total / (ms_total * 1e-3)
    e2e_value = frames_total / (ms_e2e * 1e-3)
    peak, peak_src = _peaks()
    achieved = PYR_FAST_BYTES * SB / (ms_pf * 1e-3) / 1e9
    traffic_pf, traffic_src = _traffic_per_frame()
    ceil_fps = world * c_both * 1e9 / h2d_pf
    if "config34_tracking" in workloads:
        tr = workloads["config34_tracking"]
        per_gpu_fps = value / world
        for variant, mms in tr.pop("_matcher_ms").items():
            P = tr["_agents"]
            ms_step = P / per_gpu_fps * 1e3 + mms
            tr["variants"][variant]["value"] = world * P / (ms_step * 1e-3)
        tr.pop("_agents")

    cpu_rec = None
    protocol = None
    if rank == 0 and cpu:
        v, n = cpu_oracle_rate(frames[:8], 12.0, 1)
        cpu_rec = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "cpu_model": cpu_model(), "nproc": os.cpu_count(),
                   "sample": f"{n} frames of the same workload, single thread, oracle -O2 (the reference extractor is single-threaded per agent)"}
        protocol = cpu_protocol(2.5)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frame": [W, H], "nfeatures": NFEAT, "batch_per_gpu": B,
                       "agents": world, "handles_per_gpu": eb.nh, "frames_per_handle_call": eb.hb,
                       "cache": f"inputs per step {B * W * H / 1e6:.0f} MB + plane sets >> 126 MB L2, no reuse across steps",
                       "timed_region_s": ms_total * 1e-3},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * h2d_pf, "d2h_bytes_per_step": B * d2h_pf,
                    "note": f"pinned host buffers, {eb.nslot} extractor handles x {eb.eb}-frame chunks in flight",
                    "timed_region_s": ms_e2e * 1e-3,
                    "h2d_ceiling": {"h2d_alone_gbs_per_gpu": c_h2d, "h2d_with_d2h_share_gbs_per_gpu": c_both,
                                    "frames_per_s_at_ceiling": ceil_fps, "e2e_frac_of_ceiling": e2e_value / ceil_fps,
                                    "how": "plain pinned cudaMemcpyAsync of 256 MiB x 6 on every rank at once (min over ranks), alone and "
                                           "with the device-to-host share of the path running beside it"}},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (traffic_pf * SB if traffic_pf else None),
                         "traffic_source": f"ncu dram__bytes_read+write of the same launch set (profiles/{traffic_src})" if traffic_src else None,
                         "peak_source": peak_src,
                         "kernel": "pyr_walk_kernel x8 (pyramid + border + fused blur, column walk, tensor-map TMA source rows) + fast_tile_kernel x2 "
                                   "(FAST quick reject + score + tile retry + NMS, tensor-map TMA windows), 256-frame launches",
                         "bytes_per_frame": PYR_FAST_BYTES, "ms_per_launch_set": ms_pf,
                         "frac_counting_fused_blur_bytes": (PYR_FAST_BYTES + BLUR_BYTES) * SB / (ms_pf * 1e-3) / 1e9 / peak},
            "cpu_baseline": cpu_rec,
            "cpu_baseline_protocol": protocol,
            "clocks": clocks,
            "host": ctx.host,
            "stages_ms_per_256_frames": stage_ms,
            "keypoints_per_frame": cnt / (world * B),
            "latency": latency,
            "workloads": workloads,
        }
        if "config5_place" in workloads:   # kept at the top level too: BASELINE.json's second metric
            p5 = workloads["config5_place"]
            line["hamming"] = {"metric": p5["metric"], "value": p5["value"], "unit": p5["unit"], "roofline": p5["roofline"],
                               "config": p5["config"]["workload"]}
        print(json.dumps(line), flush=True)
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
