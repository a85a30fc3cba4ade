#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 delay-Doppler hot path.

Workload (BASELINE.json configs[1]): one "step" = one 1 s CPI @ 2 MS/s through
WienerHopf (410 taps) -> Ambiguity (300 delay x 257 Doppler) -> Map::set_metrics ->
CfarDetector1D -> Centroid -> Interpolate on synthetic IQ (blah2_b200/scene.py).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Contract (one JSON line on rank 0):
  value   IQ Msamples/s, whole job over all N GPUs, inputs resident in HBM (float2), CUDA-event
          timed on the launching stream, max over ranks;  maps_per_s = value / (N_samples/1e6).
  e2e     same metric through the public host API (Pipeline.submit_host / fetch = C ABI
          b200dd_pipeline_submit_host / _fetch, PINNED complex128 host buffers): H2D of x and y and D2H of
          the map + detections inside the timed region, every step.
  roofline  the kernel with the largest SM-time share of the step (CUDA events around every stage, live:
          b200dd_wh_profile_device / b200dd_caf_profile_device; the single-CTA solve is a latency chain on one SM and
          is not a candidate): its ALGORITHMIC bytes per launch / its time against MEASURED_PEAKS.json hbm_gbs, plus --
          for the FP64 FFT kernels -- nominal FFT flops against the FP64 FMA rate measured in this run
          (b200dd_ubench_fp64_tflops: builder-measured).  `step` uses SURVEY.md s8(d)'s fused-chain bytes
          2 (16 N) + 8 nDop nDel = 64 616 800; `cfg3` times BASELINE configs[2] (CAF, 2e7 samples, 512 x 1025).
  cpu_baseline  the reference's own src/process code (oracle/_ref, unmodified sources + our FFT /
          Armadillo shims) on ONE host thread for ONE CPI of the same workload.
  --impl reference: the same reference code, one host process per concurrent CPI (time-bounded).
Multi-GPU: independent CPIs sharded over ranks ("weak" scaling, no data-path collective); the only
communication is the gather of EVERY finished map to rank 0 (C ABI b200dd_comm_gather_async: NCCL send/recv on a
dedicated stream, overlapped with the next CPI's kernels, inside the timed region).
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

FS = 2_000_000
N = 2_000_000
GEOM = dict(delayMin=0, delayMax=299, dopplerMin=-128, dopplerMax=128, fs=FS, nSamples=N, roundHamming=True)
CLUTTER = (-10, 400)
DET = dict(pfa=1e-5, nGuard=2, nTrain=6, minDelay=5, minDoppler=15.0, nCentroid=6)
WORKLOAD = ("cfg2: WienerHopf(410 taps)+Ambiguity(300 delay x 257 Doppler)+set_metrics+CFAR/Centroid/Interpolate, "
            "1 s CPI @ 2 MS/s, N=2e6 per channel")
KERNELS_PER_STEP = 4 + 2 + 2 + 3 + 1  # wh(corr,solve,wspec,apply) caf(range,doppler) metrics(2) cfar(flag,scan,emit) tail(centroid+interp)


def ncu_traffic(kernel="caf_range_", capture="cfg2"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` in the `capture` section of the committed
    ncu --set full extract (profiles/r02_kernels.json, else round 1's), or None."""
    for name in ("r02_kernels.json", "r01z_kernels.json"):
        try:
            ks = json.load(open(os.path.join(ROOT, "profiles", name)))["kernels"]
            for k in ks:
                if kernel in k["name"] and capture in str(k.get("capture", capture)):
                    return int(k["dram_bytes_read"] + k["dram_bytes_write"])
        except Exception:
            pass
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _cpu_chain():
    """(run(x, y) -> (stage_ms, n_detections), kind): the compiled reference (oracle/_ref) when it was built,
    else the numpy port of the same algorithm (oracle/blah2_oracle.py)."""
    from oracle import refpath as R
    if R.available():
        ch = R.Chain(GEOM["delayMin"], GEOM["delayMax"], GEOM["dopplerMin"], GEOM["dopplerMax"], FS, N, True, clutter=CLUTTER,
                     **DET)

        def run(x, y):
            r = ch.run(x, y, want_map=False)
            return [float(v) for v in r["stage_ms"]], int(len(r["detections"][0]))
        return run, "reference"
    from oracle import blah2_oracle as O
    g = O.ambiguity_geometry(GEOM["delayMin"], GEOM["delayMax"], GEOM["dopplerMin"], GEOM["dopplerMax"], FS, N, True)

    def run(x, y):
        t0 = time.perf_counter()
        r = O.chain(x, y, g, clutter=CLUTTER, det=DET)
        return [0.0, (time.perf_counter() - t0) * 1e3, 0.0], int(len(r["detections"][0]))
    return run, "port"


def _ref_worker(conn, seed):
    """One host process = one stream of CPIs through the reference's own classes (separate address spaces:
    the reference's per-sample deque traffic makes threads contend on the allocator)."""
    from blah2_b200.scene import make_scene

    sc = make_scene(N, FS, seed=seed)
    run, kind = _cpu_chain()
    conn.send("ready:" + kind)
    while True:
        cmd = conn.recv()
        if cmd == "stop":
            break
        conn.send(run(sc.x, sc.y)[0])


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores."""
    if rank != 0:
        return
    import multiprocessing as mp

    cores = os.cpu_count() or 1
    try:
        avail_gb = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE") / 2**30
    except Exception:
        avail_gb = 16.0
    procs_n = int(max(1, min(cores, 32, avail_gb // 3)))  # ~2 GB of FFT plans + buffers per process
    ctx = mp.get_context("spawn")
    workers = []
    for i in range(procs_n):
        a, b = ctx.Pipe()
        p = ctx.Process(target=_ref_worker, args=(b, 20260923))
        p.start()
        workers.append((p, a))
    kind = "reference"
    for _, c in workers:
        msg = c.recv()
        assert msg.startswith("ready:")
        kind = msg.split(":", 1)[1]

    def step():
        for _, c in workers:
            c.send("run")
        return [c.recv() for _, c in workers]

    # bounded: a CPI takes seconds on the CPU; warm-up is capped at one step and the timed steps stop
    # after ~150 s (steps actually timed are reported as "steps")
    for _ in range(min(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    stages = []
    done = 0
    for _ in range(args.steps):
        stages += step()
        done += 1
        if time.perf_counter() - t0 > 150.0:
            break
    dt = time.perf_counter() - t0
    for p, c in workers:
        c.send("stop")
    for p, c in workers:  # let them run their exit handlers (the driver records the libraries they loaded)
        p.join(timeout=30)
        if p.is_alive():
            p.terminate()
    requested = args.steps
    args.steps = done
    cpis = procs_n * args.steps
    value = cpis * N / dt / 1e6
    st = np.mean(np.array(stages), axis=0)
    line = {
        "impl": "reference", "metric": "iq_msamples_per_s", "value": round(value, 4), "unit": "Msamples/s",
        "maps_per_s": round(cpis / dt, 4), "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "step": f"{procs_n} CPIs, one per host process", "steps_requested": requested},
        "cpu_baseline": {"value": round(value, 4), "unit": "Msamples/s", "cores": procs_n, "kind": kind,
                         "sample": f"{cpis} full CPIs ({procs_n} concurrent host processes); " +
                                   ("unmodified reference src/process sources linked to this repo's FFTW/Armadillo shims "
                                    "(stock FFTW not in the image)" if kind == "reference" else
                                    "numpy port of the reference algorithm (oracle/_ref was not built)"),
                         "stage_ms": {"clutter_filter": round(float(st[0]), 1),
                                      "ambiguity_processing": round(float(st[1]), 1),
                                      "detector": round(float(st[2]), 2)}, "host_cores": cores},
        "e2e": {"value": round(value, 4), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dropin_leg(sc, cpis=3):
    """Level-1 drop-in, end to end (VERDICT r1 item 7): the C++ classes of blah2_b200/dropin driven exactly as the
    reference's process thread drives its own (src/blah2.cpp:268-287: WienerHopf::process -> Ambiguity::process ->
    Map::set_metrics -> CfarDetector1D -> Centroid -> Interpolate on IqData deques, Map and Detection objects),
    through the same harness source that drives the reference (oracle/ref_capi.cpp compiled against the drop-in
    headers: tests/native, built into oracle/_ref beside the reference library).  Stage times are the harness's own
    (the reference's stage names); the IqData fill is the caller's deque traffic (blah2.cpp:254-258) and is timed
    apart."""
    import importlib.util
    harness = os.path.join(ROOT, "oracle", "_ref", "libdropin_harness.so")
    if not os.path.exists(harness):
        return {"unavailable": "oracle/_ref/libdropin_harness.so not built (needs the blah2 sources at build time)"}
    try:
        from oracle import refpath as R
        spec = importlib.util.spec_from_file_location("dropin_binding", R.__file__)
        D = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(D)
        D.LIB_PATH = harness
        ch = D.Chain(GEOM["delayMin"], GEOM["delayMax"], GEOM["dopplerMin"], GEOM["dopplerMax"], FS, N, True, clutter=CLUTTER, **DET)
        ch.run(sc.x, sc.y, want_map=False)   # warm-up (allocations, first launches)
        t, stages, ndet = [], [], 0
        for _ in range(cpis):
            t0 = time.perf_counter()
            r = ch.run(sc.x, sc.y, want_map=False)
            t.append((time.perf_counter() - t0) * 1e3)
            stages.append([float(v) for v in r["stage_ms"]])
            ndet = len(r["detections"][0])
        st = np.mean(np.array(stages), axis=0)
        ms = float(np.mean(t))
        ch.close()
        return {"value": round(N / (ms * 1e-3) / 1e6, 2), "unit": "Msamples/s", "ms_per_step": round(ms, 3), "steps": cpis,
                "stage_ms": {"clutter_filter": round(float(st[0]), 3), "ambiguity_processing": round(float(st[1]), 3),
                             "detector": round(float(st[2]), 3),
                             "iqdata_fill_and_result_copy": round(ms - float(np.sum(st)), 3)},
                "n_detections": ndet,
                "api": "C++ drop-in classes (libblah2dropin.so) on std::deque IqData / Map / Detection, one host thread"}
    except Exception as e:  # the headline line must not die on the side leg
        return {"unavailable": f"{type(e).__name__}: {e}"}


def dump_outputs(out_dir, res, d_map, pipe):
    """What a caller of the timed path receives for one CPI, as DIR/<name>.npy: the device map (complex64
    [nDoppler][nDelay], stored as float32 [..., 2] = real, imag), set_metrics' noise and max power with the skip flag,
    the detection list ([3][nDetections]: delay, Doppler, SNR) and the map's axes."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    det = res["detections"]
    arrays = {
        "map": torch.view_as_real(d_map).cpu().numpy().astype(np.float32),
        "metrics": np.array([res["noisePower"], res["maxPower"], float(res["skipped"])], dtype=np.float64),
        "detections": np.stack([det.delay, det.doppler, det.snr]).astype(np.float64),
        "delay": pipe.delay.astype(np.float64),
        "doppler": pipe.doppler.astype(np.float64),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true", help="launch every kernel of every CPI instead of replaying the chain as a CUDA graph")
    ap.add_argument("--streams", type=int, default=6, help="CPIs in flight per GPU (independent pipelines on their own streams)")
    ap.add_argument("--no-gather", action="store_true", help="diagnostic: N > 1 without the map gather (not a bench mode)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (map, metrics, detections) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    args.graph = not args.eager

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import ctypes

    from blah2_b200 import capi
    from blah2_b200.process import Ambiguity, Pipeline, WienerHopf
    from blah2_b200.scene import make_scene
    from blah2_b200.shard import Comm

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # the submitting thread and its pinned staging buffers on the GPU's NUMA node (the end-to-end path is PCIe-bound)
    cpulist = ctypes.create_string_buffer(256)
    numa_rc = capi.load().b200dd_bind_host_to_device(local_rank, cpulist, 256)
    host_cpus = cpulist.value.decode() if numa_rc == 0 else None
    # stdout carries exactly ONE line, the JSON: keep the real stdout aside and point file descriptor 1 at stderr, so
    # that anything a library prints there (NCCL's "NCCL version ..." banner, which it writes at WARN level too)
    # lands on stderr instead
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    comm = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        comm = Comm(rank, world, local_rank)

    NPIPE = max(1, args.streams)
    pipes = [Pipeline(**GEOM, clutter=CLUTTER, detection=DET, device=local_rank) for _ in range(NPIPE)]
    pipe = pipes[0]
    g = pipe.geometry
    cells = g.n_doppler_bins * g.n_delay_bins

    # ---- inputs: NB distinct CPIs resident in HBM (> 2x the 126 MB L2) + 2 pinned host CPIs ----
    sc = make_scene(N, FS, seed=20260923 + rank)
    NB = 10
    x0 = torch.from_numpy(sc.x.astype(np.complex64)).cuda()
    y0 = torch.from_numpy(sc.y.astype(np.complex64)).cuda()
    xs = [torch.roll(x0, 977 * b) for b in range(NB)]
    ys = [torch.roll(y0, 977 * b) for b in range(NB)]
    hx = [torch.from_numpy(np.roll(sc.x, 977 * b)).pin_memory() for b in range(2)]
    hy = [torch.from_numpy(np.roll(sc.y, 977 * b)).pin_memory() for b in range(2)]
    hmap = torch.empty((g.n_doppler_bins, g.n_delay_bins), dtype=torch.complex128).pin_memory()
    streams = [torch.cuda.Stream() for _ in range(NPIPE)]
    stream = streams[0]
    st = stream.cuda_stream

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Map gather (N > 1): every CPI of the region writes its map into its OWN slot of a device-resident ring (no slot is
    # reused inside the region, so the compute streams never wait for the communicator); the maps of a chunk of NPIPE
    # consecutive CPIs travel to rank 0 in ONE exchange (b200dd_comm_gather_async: NCCL send/recv on the communicator's
    # stream) as soon as the chunk's CPIs have finished, beside the next chunk's kernels.  (One exchange per CPI cost
    # 13 % of the step at N = 2 -- the NCCL calls take longer on the submitting thread than the CPI's graph launch;
    # profiles/r02_summary.md.)
    map_bytes = cells * 8
    NMAPS = max(args.steps, args.warmup) if comm is not None else NPIPE
    ring = torch.empty((NMAPS, g.n_doppler_bins, g.n_delay_bins), dtype=torch.complex64, device="cuda")
    dmaps = [ring[k] for k in range(NMAPS)]
    dmap = dmaps[0]
    n_chunks = (NMAPS + NPIPE - 1) // NPIPE
    recv_all = None
    if comm is not None and rank == 0:   # [chunk][world][NPIPE] maps, allocated once
        recv_all = torch.empty((n_chunks, world, NPIPE, g.n_doppler_bins, g.n_delay_bins), dtype=torch.complex64, device="cuda")

    def slot_of(i):
        return i if comm is not None else i % NPIPE

    def gather_chunk(first, count):
        """maps of the CPIs [first, first + count) -> rank 0, behind the pipelines that produced them"""
        for q in range(count):
            comm.wait_stream(streams[(first + q) % NPIPE])
        c = first // NPIPE
        comm.gather_async(ring[first:first + count], recv_all[c].view(-1)[: world * count * cells].view(world, count, g.n_doppler_bins, g.n_delay_bins) if rank == 0 else None, 0, after=None)

    def submit(i, n_total):
        p = i % NPIPE
        with torch.cuda.stream(streams[p]):
            pipes[p].submit_device(xs[i % NB], ys[i % NB], dmaps[slot_of(i)], streams[p].cuda_stream)
        if comm is not None and not args.no_gather and ((i + 1) % NPIPE == 0 or i == n_total - 1):
            first = (i // NPIPE) * NPIPE
            gather_chunk(first, i - first + 1)

    # ---- device-resident throughput: a stream of independent CPIs, NPIPE in flight ----
    # Plan creation (untimed, before the warm-up steps): the CUDA graph of the chain for every (input set, pipeline)
    # pair the loop below submits -- one launch per CPI instead of 13.  (Round 1 measured replay 3 % slower than eager
    # launches at 111 us per CPI; at this round's ~60 us per CPI the 13 launches of a CPI are what the submitting
    # thread cannot keep up with.)  --eager turns it off.
    if args.graph:
        n_prep = NB * NPIPE if comm is None else NMAPS   # 1 GPU: (i % NB, i % NPIPE) repeats after lcm(NB, NPIPE) steps
        for i in range(n_prep):
            p = i % NPIPE
            pipes[p].prepare_device(xs[i % NB], ys[i % NB], dmaps[slot_of(i)], streams[p].cuda_stream)
    for i in range(args.warmup):
        submit(i, args.warmup)   # (also warms the communicator and the gather path)
    for p in range(NPIPE):
        last = pipes[p].fetch(streams[p].cuda_stream)
    if comm is not None:
        comm.sync()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if comm is not None:
        # start line on the DEVICE timelines: every rank's streams wait for one tiny all-reduce, which completes on all
        # ranks within microseconds of each other (host-side barrier skew would otherwise be charged to the region)
        tick = torch.zeros(2, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        comm.allreduce_f64_async(tick, after=None)
        comm.join(stream)
    e0.record(stream)
    for s_ in streams[1:]:
        s_.wait_event(e0)
    t_host0 = time.perf_counter()
    for i in range(args.steps):
        submit(i, args.steps)
    host_submit_us = (time.perf_counter() - t_host0) / args.steps * 1e6   # the submitting thread's time per CPI
    fetched = [None] * NPIPE
    for p in reversed(range(NPIPE)):  # synchronises each stream; detections + metrics of the final CPIs on the host
        last = fetched[p] = pipes[p].fetch(streams[p].cuda_stream)
    with torch.cuda.stream(stream):
        if comm is not None:  # the last gathers (rank 0: every rank's maps have arrived) end the region
            comm.join(stream)
        e1.record(stream)
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    gather_check = None
    if comm is not None and rank == 0 and not args.no_gather:   # rank 0's own block of the last chunk equals its device maps: the gather really ran
        first = ((args.steps - 1) // NPIPE) * NPIPE
        count = args.steps - first
        got = recv_all[first // NPIPE].view(-1)[: world * count * cells].view(world, count, g.n_doppler_bins, g.n_delay_bins)
        gather_check = bool(torch.equal(got[0], ring[first:first + count])) and bool(torch.isfinite(torch.view_as_real(got)).all())
    if args.dump_outputs is not None and rank == 0:   # before anything below reuses the map slots
        dump_outputs(args.dump_outputs, fetched[(args.steps - 1) % NPIPE], dmaps[slot_of(args.steps - 1)], pipe)

    # ---- end to end through the host API (pinned complex128 in, complex128 map out) ----
    # Two pipelines alternate: submit_host(i) enqueues H2D + kernels + D2H, fetch(i-1) collects the
    # previous CPI's map/detections, so PCIe transfers of one CPI overlap the kernels of the other.
    hmaps = [torch.empty((g.n_doppler_bins, g.n_delay_bins), dtype=torch.complex128).pin_memory() for _ in range(NPIPE)]
    for i in range(2 * NPIPE):
        pipes[i % NPIPE].process(hx[i % 2], hy[i % 2], map_out=hmaps[i % NPIPE])
    barrier()
    e2e_steps = max(6, min(args.steps, 30))
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        p = i % NPIPE
        if i >= NPIPE:
            r_e2e = pipes[p].fetch()          # result of CPI i - NPIPE is now in host memory
        pipes[p].submit_host(hx[i % 2], hy[i % 2], map_out=hmaps[p])
    for i in range(e2e_steps, e2e_steps + NPIPE):
        r_e2e = pipes[i % NPIPE].fetch()
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())

    # ---- the same, fed with the reference's replay layout (int16 I1 Q1 I2 Q2, 8 B per instant) ----
    def to_i16(b):
        x_, y_ = np.roll(sc.x, 977 * b), np.roll(sc.y, 977 * b)
        iq = np.empty((N, 4), dtype="<i2")
        iq[:, 0], iq[:, 1], iq[:, 2], iq[:, 3] = x_.real, x_.imag, y_.real, y_.imag
        return torch.from_numpy(iq).pin_memory()

    hq = [to_i16(b) for b in range(2)]
    for i in range(NPIPE):
        pipes[i].submit_host_rspduo(hq[i % 2], map_out=hmaps[i])
        pipes[i].fetch()
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        p = i % NPIPE
        if i >= NPIPE:
            r_i16 = pipes[p].fetch()
        pipes[p].submit_host_rspduo(hq[i % 2], map_out=hmaps[p])
    for i in range(e2e_steps, e2e_steps + NPIPE):
        r_i16 = pipes[i % NPIPE].fetch()
    torch.cuda.synchronize()
    i16_s = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(i16_s, op=dist.ReduceOp.MAX)
    i16_s = float(i16_s.item())

    clocks = sampler.stop() if rank == 0 else None  # sampled over the device-resident AND the end-to-end timed regions

    # ---- per-kernel durations for the roofline (CUDA events around each kernel) ----
    amb = Ambiguity(GEOM["delayMin"], GEOM["delayMax"], GEOM["dopplerMin"], GEOM["dopplerMax"], FS, N, True,
                    device=local_rank)
    wh = WienerHopf(CLUTTER[0], CLUTTER[1], N, device=local_rank)
    yf = torch.empty_like(ys[0])
    prof = {"range": [], "doppler": [], "wh_corr": [], "wh_solve": [], "wh_apply": []}
    with torch.cuda.stream(stream):
        for i in range(3 + min(args.steps, 30)):
            c, s_, a_ = wh.profile_device(xs[i % NB], ys[i % NB], yf, st)
            r_, d_ = amb.profile_device(xs[i % NB], yf, dmap, st)
            if i >= 3:
                prof["range"].append(r_); prof["doppler"].append(d_)
                prof["wh_corr"].append(c); prof["wh_solve"].append(s_); prof["wh_apply"].append(a_)
    kms = {k: float(np.mean(v)) for k, v in prof.items()}

    # ---- SpectrumAnalyser(n, 2000) (blah2.cpp:198,263-265) on the resident reference channel: not part of the
    # step above (BASELINE's configs do not include it); its folding pass is the path's purely HBM-bound kernel ----
    spectrum = None
    if rank == 0:
        from blah2_b200.process import SpectrumAnalyser
        spectrum = {"api": "SpectrumAnalyser(n, 2000.0).process_device(float2 x)", "kernel": "spec_fold_kernel",
                    "algorithmic_bytes": "8 nfft (x read once)"}
        big = [torch.randn(20_000_000, dtype=torch.complex64, device="cuda") for _ in range(2)]
        for label, n_, bufs in (("n2e6", N, xs), ("n2e7", 20_000_000, big)):
            sa = SpectrumAnalyser(n_, 2000.0, device=local_rank)
            f_, r_ = [], []
            with torch.cuda.stream(stream):
                for i in range(3 + 20):
                    a_, b_ = sa.profile_device(bufs[i % len(bufs)], st)
                    if i >= 3:
                        f_.append(a_); r_.append(b_)
            fm, rm = float(np.mean(f_)), float(np.mean(r_))
            spectrum[label] = {"n_spectrum": sa.nSpectrum, "decimation": sa.decimation, "fold_ms": round(fm, 5),
                               "reduce_dft_ms": round(rm, 5), "achieved_gbs": round(8 * sa.nfft / (fm * 1e-3) / 1e9, 1)}
            sa.close()

    # ---- BASELINE configs[2] (the configuration designated for the HBM capture): CAF alone, 2 s CPI @ 10 MS/s,
    # 512 delay x 1025 Doppler, device-resident float2 IQ (2 x 160 MB per map > L2), CUDA events around each kernel ----
    cfg3 = None
    fp64_peak = None
    if rank == 0:
        tf = ctypes.c_double()
        capi.check(capi.load().b200dd_ubench_fp64_tflops(local_rank, ctypes.byref(tf)))
        fp64_peak = float(tf.value)
        amb3 = Ambiguity(0, 511, -256, 256, 10_000_000, 20_000_000, True, device=local_rank)
        g3 = amb3.geometry
        bigy = [torch.randn(20_000_000, dtype=torch.complex64, device="cuda") for _ in range(2)]
        out3 = torch.empty((g3.n_doppler_bins, g3.n_delay_bins), dtype=torch.complex64, device="cuda")
        r3, d3 = [], []
        with torch.cuda.stream(stream):
            for i in range(3 + 10):
                a_, b_ = amb3.profile_device(big[i % 2], bigy[i % 2], out3, st)
                if i >= 3:
                    r3.append(a_); d3.append(b_)
        torch.cuda.synchronize()
        cfg3 = {"workload": "cfg3: Ambiguity 512 delay x 1025 Doppler, 2 s CPI @ 10 MS/s, N=2e7 per channel",
                "range_ms": round(float(np.mean(r3)), 5), "doppler_ms": round(float(np.mean(d3)), 5),
                "algorithmic_bytes": 16 * g3.n_used + 8 * g3.n_doppler_bins * g3.n_delay_bins,
                "range_fft": f"M={g3.range_fft_len} x{g3.range_segments} segments, hop {g3.range_hop}"}
        amb3.close()
        del big, bigy, out3

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    for label in ("n2e6", "n2e7"):
        spectrum[label]["frac"] = round(spectrum[label]["achieved_gbs"] / peak, 4)
    # ---- roofline: the kernel that owns the SMs (largest CUDA-event time among the full-grid kernels) ----
    plan = wh.plan
    fft_flop = lambda m: 5.0 * m * np.log2(m)   # nominal flops of one m-point complex transform
    cand = {
        "wh_corr": dict(kernel="wh_corr_kernel", ms=kms["wh_corr"], bytes=16 * N,
                        flop=(3 * plan.corr_segments + 2 * plan.corr_ctas) * fft_flop(plan.corr_fft_len), dtype="f64"),
        "wh_apply": dict(kernel="wh_apply_kernel", ms=kms["wh_apply"], bytes=16 * N + 8 * N,
                         flop=(2 * plan.filter_blocks + 1) * fft_flop(plan.filter_fft_len), dtype="f64"),
        "range": dict(kernel="caf_range_grouped_kernel" if g.range_groups > 1 else "caf_range_kernel", ms=kms["range"],
                      bytes=16 * g.n_used + 8 * g.range_parts * cells, flop=None, dtype="f32"),
        "doppler": dict(kernel="caf_doppler_kernel", ms=kms["doppler"], bytes=8 * cells, flop=None, dtype="f32"),
    }
    dom_key = max(cand, key=lambda k: cand[k]["ms"])
    dom = cand[dom_key]
    ach = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9
    bytes_caf = 16 * g.n_used + 8 * cells                   # SURVEY s8(d) B_caf (map written; R stays in L2)
    bytes_step = 2 * 16 * N + 8 * cells                     # SURVEY s8(d) B_wh+caf: two compulsory passes over x, y + the map
    roofline = {"kernel": dom["kernel"], "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                "frac": round(ach / peak, 4), "traffic": ncu_traffic(dom["kernel"].replace("_grouped_kernel", "_").replace("_kernel", "")),
                "peak_source": peak_src, "algorithmic_bytes": dom["bytes"], "kernel_ms": round(dom["ms"], 5),
                "chosen_by": "largest CUDA-event time among the full-grid kernels of the step (wh_solve is one CTA on one SM: "
                             "a latency chain that overlaps the other CPIs' kernels, no roofline applies)",
                "share_of_kernel_time": round(dom["ms"] / sum(c["ms"] for c in cand.values()), 3)}
    if dom["flop"]:
        tfl = dom["flop"] / (dom["ms"] * 1e-3) / 1e12
        roofline["fp64"] = {"achieved_tflops": round(tfl, 2), "peak_tflops": round(fp64_peak, 2), "frac": round(tfl / fp64_peak, 4),
                            "flops": "5 M log2 M per transform (nominal), transforms per launch from b200dd_wh_get_plan",
                            "peak_source": "b200dd_ubench_fp64_tflops in this run (builder-measured DFMA rate)"}
    roofline["per_kernel"] = {k: {"ms": round(c["ms"], 5), "hbm_frac": round(c["bytes"] / (c["ms"] * 1e-3) / 1e9 / peak, 4),
                                  **({"fp64_frac": round(c["flop"] / (c["ms"] * 1e-3) / 1e12 / fp64_peak, 4)} if c["flop"] else {})}
                              for k, c in cand.items()}
    roofline["caf_total"] = {"ms": round(kms["range"] + kms["doppler"], 5),
                             "frac": round(bytes_caf / ((kms["range"] + kms["doppler"]) * 1e-3) / 1e9 / peak, 4)}
    roofline["step"] = {"algorithmic_bytes": bytes_step, "frac": round(bytes_step / (ms_total / args.steps * 1e-3) / 1e9 / peak, 4)}
    cfg3["ms"] = round(cfg3["range_ms"] + cfg3["doppler_ms"], 5)
    cfg3["achieved_gbs"] = round(cfg3["algorithmic_bytes"] / (cfg3["ms"] * 1e-3) / 1e9, 1)
    cfg3["frac"] = round(cfg3["achieved_gbs"] / peak, 4)
    cfg3["range_kernel_frac"] = round(cfg3["algorithmic_bytes"] / (cfg3["range_ms"] * 1e-3) / 1e9 / peak, 4)
    cfg3["traffic"] = ncu_traffic("caf_range_", "cfg3")
    cfg3["msamples_per_s"] = round(20_000_000 / (cfg3["ms"] * 1e-3) / 1e6, 1)
    value = world * args.steps * N / (ms_total * 1e-3) / 1e6
    e2e_value = world * e2e_steps * N / e2e_s / 1e6
    line = {
        "metric": "iq_msamples_per_s", "value": round(value, 2), "unit": "Msamples/s",
        "maps_per_s": round(world * args.steps / (ms_total * 1e-3), 2),
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 5),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (CAF) / f64 (WienerHopf, detection)",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "cpis_per_step_per_gpu": 1, "parallelism": f"independent CPIs x{world}",
                   "l2": f"{NB} distinct CPI input sets rotated ({NB * 32} MB > L2)", "cpis_in_flight": NPIPE, "submission": "cuda graph replay (b200dd_pipeline_prepare_device)" if args.graph else "eager launches",
                   "host_cpus": host_cpus, "map_gather": (f"every finished map to rank 0, one b200dd_comm_gather_async (NCCL send/recv on a dedicated stream) per chunk of {NPIPE} CPIs, check {gather_check}" if world > 1 else "none (1 GPU)"),
                   "host_submit_us_per_step": round(host_submit_us, 1),
                   "range_fft": f"M={g.range_fft_len} x{g.range_segments} segments, hop {g.range_hop}, "
                                f"{g.range_groups} warp group(s) x {g.range_parts} part(s) per batch",
                   "doppler_fft": f"Bluestein M2={g.doppler_fft_len}"},
        "e2e": {"value": round(e2e_value, 2), "unit": "Msamples/s", "h2d_bytes_per_step": 2 * 16 * N,
                "d2h_bytes_per_step": 16 * cells + 3 * 8 * int(r_e2e["detections"].get_nDetections()) + 32,
                "ms_per_step": round(e2e_s / e2e_steps * 1e3, 4), "steps": e2e_steps,
                "api": "Pipeline.submit_host(pinned complex128 x, y) / fetch() -> complex128 map + detections, "
                       f"{NPIPE} CPIs in flight"},
        "e2e_rspduo_int16": {"value": round(world * e2e_steps * N / i16_s / 1e6, 2), "unit": "Msamples/s",
                             "h2d_bytes_per_step": 8 * N, "ms_per_step": round(i16_s / e2e_steps * 1e3, 4),
                             "api": "Pipeline.submit_host_rspduo(pinned int16 I1 Q1 I2 Q2) / fetch()",
                             "n_detections": int(r_i16["detections"].get_nDetections())},
        "gpu_launches": KERNELS_PER_STEP * args.steps,
        "clocks": clocks,
        "roofline": roofline,
        "cfg3": cfg3,
        "kernel_ms": {k: round(v, 5) for k, v in kms.items()},
        "spectrum": spectrum,
        "result": {"n_detections": int(last["detections"].get_nDetections()), "noisePower": round(last["noisePower"], 4),
                   "maxPower": round(last["maxPower"], 4), "filter_ok": not last["skipped"]},
    }
    if world == 1 and not args.no_cpu_baseline:
        run, kind = _cpu_chain()
        t0 = time.perf_counter()
        stage_ms, n_det = run(sc.x, sc.y)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": round(N / dt / 1e6, 4), "unit": "Msamples/s", "cores": 1, "kind": kind,
                                "sample": "1 full CPI of the same workload on 1 host thread (" +
                                          ("reference src/process sources unmodified + this repo's FFTW/Armadillo shims"
                                           if kind == "reference" else "numpy port, oracle/_ref was not built") + ")",
                                "stage_ms": {"clutter_filter": round(stage_ms[0], 1),
                                             "ambiguity_processing": round(stage_ms[1], 1),
                                             "detector": round(stage_ms[2], 2)},
                                "host_cores": os.cpu_count(), "n_detections": n_det}
        try:  # the reference's SpectrumAnalyser on the same reference channel (blah2.cpp:263-265), for the `spectrum` block
            from oracle import refpath as R
            if R.available():
                t0 = time.perf_counter()
                R.spectrum_process(sc.x, N, 2000.0)
                line["cpu_baseline"]["spectrum_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
        except Exception:
            pass
    if world == 1:
        line["e2e_dropin"] = dropin_leg(sc)
    print(json.dumps(line), file=json_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
