#!/usr/bin/env python
"""bench.py -- headline benchmark of the spectral watermark hot path (BASELINE.json).

metric   audio frames/sec embed+detect, 44.1 kHz stereo (PCM sample-frames per second of
         `add` + `get` wall time; decoded payload checked against the embedded one)
workload BASELINE.json configs[1]: 1 h stereo 44.1 kHz per GPU (weak scaling: every rank owns
         one hour of the N-hour stream; ranks exchange nothing but the final result gather)
step     one `add` (embed + limiter) followed by one `get` (chunked sync search, block decode,
         Viterbi, result merge) over the whole hour, through the host-side C++ drivers
         (audiowmark_b200/host -> C ABI -> sm_100a kernels)

value  : inputs resident in HBM (device pointers), timed with CUDA events on the context stream
e2e    : the same call with pinned HOST buffers holding 16 bit PCM (the sample format of the reference arm's WAV
         files; converted on the device with the reference's rules): H2D of the input for add, D2H of the marked
         audio, H2D of the marked audio for get and D2H of the results are all inside the timed region
e2e_f32: the same with fp32 host buffers (twice the PCIe bytes)
roofline / kernels : per-kernel CUDA-event times of the timed steps (awm_profile_*)
cpu_baseline       : the reference's own CPU implementation (oracle/_ref/audiowmark, unmodified
                     sources, FFT = in-repo shim with AVX2 passes) on the same 60 min workload, rank 0 at N=1 only
add / get          : the two halves of a step timed separately (north_star's target is on `get`)
cli_e2e            : `bin/audiowmark add` + `cmp` as processes on a tmpfs WAV: process start, CUDA context creation, file I/O included

python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--minutes M] [--dump-outputs DIR]

--dump-outputs DIR : after the timed steps, what the last timed resident step returned, as DIR/<name>.npy (float32 / float64,
                     about 16 MB in all; the input is a pure function of the arguments, so two builds compare output for output):
  marked_frame, marked_audio      a fixed, seeded sample of 2^20 frame numbers of the marked audio `add` wrote and their samples
                                  (frames x channels; with several GPUs, of rank 0's range)
  match_pos_s, match_quality, match_error, match_rating, match_speed
                                  the fields of the matches of the `get --json` document, in its order (pos in seconds)
  match_type                      index of the type string in MATCH_TYPES
  match_bits                      the decoded payload, one 0 / 1 entry per bit (matches x 128)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

RATE = 44100
PAYLOAD = "0123456789abcdef0011223344556677"
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "audiowmark")


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


# ----------------------------------------------------------------------------- clocks

class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
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
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- reference arm

def run_reference(steps, warmup, minutes):
    """The reference's own CPU `add` + `get` (unmodified sources in oracle/_ref) on a bounded sample."""
    import numpy as np
    import awm_oracle as O
    if not os.path.exists(REF_BIN):           # built by __graft_entry__.build(); the benchmark itself writes nothing into the tree
        raise RuntimeError("oracle/_ref/audiowmark is missing (__graft_entry__.build() makes it where the reference sources are available)")
    seconds = minutes * 60.0
    n = int(seconds * RATE)
    tmp = tempfile.mkdtemp(prefix="awm_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    src, dst = os.path.join(tmp, "in.wav"), os.path.join(tmp, "wm.wav")
    rng = np.random.default_rng(1)
    x = (rng.random((n, 2), dtype=np.float32) - 0.5).astype(np.float32)
    O.write_wav16(src, x)
    del x
    times = []
    ok = True
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        subprocess.run([REF_BIN, "-q", "add", src, dst, PAYLOAD], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        t1 = time.perf_counter()
        p = subprocess.run([REF_BIN, "-q", "cmp", dst, PAYLOAD], capture_output=True, text=True)
        t2 = time.perf_counter()
        ok = ok and p.returncode == 0
        if it >= warmup:
            times.append((t1 - t0, t2 - t1))
    for f in (src, dst):
        try:
            os.remove(f)
        except OSError:
            pass
    os.rmdir(tmp)
    t_add = sum(t[0] for t in times) / len(times)
    t_get = sum(t[1] for t in times) / len(times)
    return {"value": n / (t_add + t_get), "t_add_s": t_add, "t_get_s": t_get, "n_frames": n, "payload_ok": ok,
            "add_value": n / t_add, "get_value": n / t_get, "fft": fft_shim_vs_pocketfft(),
            "cores": os.cpu_count(), "sample": "%g min stereo 44.1 kHz s16 WAV on tmpfs: `audiowmark add` (1 thread) + `audiowmark cmp` (all threads), wall time incl. process start and file I/O" % minutes}


def fft_shim_vs_pocketfft():
    """The reference build's FFT is the in-repo shim (FFTW is not installed).  To quantify how far that is from a tuned library:
    microseconds per 1024-point real transform, one thread, shim vs scipy's pocketfft (C++, SIMD)."""
    try:
        import ctypes
        import numpy as np
        import scipy.fft
        import awm_oracle as O
        L = O.lib()
        L.orc_fft_r2c_us.restype = ctypes.c_double
        L.orc_fft_r2c_us(ctypes.c_int(2000))
        t_shim = L.orc_fft_r2c_us(ctypes.c_int(100000))
        xs = (np.random.default_rng(0).random((4096, 1024), dtype=np.float32) - 0.5).astype(np.float32)
        scipy.fft.rfft(xs, axis=1)
        t0 = time.perf_counter()
        for rep in range(5):
            scipy.fft.rfft(xs, axis=1)
        t_pf = (time.perf_counter() - t0) / (5 * len(xs)) * 1e6
        return {"shim_us_per_r2c_1024": round(t_shim, 3), "pocketfft_us_per_r2c_1024": round(t_pf, 3)}
    except Exception as e:
        return {"error": str(e)}


def run_cli_e2e(minutes):
    """`audiowmark add` + `audiowmark cmp` of THIS repo as separate processes on a tmpfs WAV: what a user of the CLI sees, with process
    start, CUDA context creation, WAV parsing and file I/O inside the time (the reference arm pays the same minus CUDA)."""
    import numpy as np
    import awm_oracle as O
    from audiowmark_b200 import hostapi as H
    n = int(minutes * 60 * RATE)
    tmp = tempfile.mkdtemp(prefix="awm_cli_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    src, dst = os.path.join(tmp, "in.wav"), os.path.join(tmp, "wm.wav")
    try:
        rng = np.random.default_rng(1)
        O.write_wav16(src, (rng.random((n, 2), dtype=np.float32) - 0.5).astype(np.float32))
        best = None
        for _ in range(2):
            t0 = time.perf_counter()
            subprocess.run([H.CLI_PATH, "-q", "add", src, dst, PAYLOAD], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            t1 = time.perf_counter()
            p = subprocess.run([H.CLI_PATH, "-q", "cmp", dst, PAYLOAD], capture_output=True, text=True)
            t2 = time.perf_counter()
            if best is None or t2 - t0 < best[0] + best[1]:
                best = (t1 - t0, t2 - t1, p.returncode == 0)
        return {"value": n / (best[0] + best[1]), "unit": "PCM frames/s", "t_add_s": round(best[0], 3), "t_get_s": round(best[1], 3), "payload_ok": best[2],
                "what": "bin/audiowmark add + cmp, %g min stereo s16 WAV on tmpfs, best of 2, incl. process start, CUDA context creation and file I/O" % minutes}
    finally:
        for f in (src, dst):
            try:
                os.remove(f)
            except OSError:
                pass
        os.rmdir(tmp)


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    minutes = args.minutes if args.minutes else 60.0
    r = run_reference(args.steps, args.warmup, minutes)
    line = {
        "impl": "reference", "metric": "audio frames/sec embed+detect, 44.1 kHz stereo; decoded-bit match vs ref", "value": r["value"],
        "unit": "PCM frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * (r["t_add_s"] + r["t_get_s"]), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "payload_ok": r["payload_ok"],
        "config": {"workload": "%g min stereo 44.1 kHz embed+detect per GPU (BASELINE.json configs[1]%s)" % (minutes, "" if minutes == 60 else ", shortened"),
                   "pcm_frames_per_gpu": r["n_frames"], "channels": 2, "payload_bits": 128, "get_chunks": "30 min, 134.4 s overlap"},
        "add": {"value": r["add_value"], "unit": "PCM frames/s", "s_per_step": r["t_add_s"], "threads": 1},
        "get": {"value": r["get_value"], "unit": "PCM frames/s", "s_per_step": r["t_get_s"], "threads": r["cores"]},
        "cpu_baseline": {"value": r["value"], "unit": "PCM frames/s", "cores": r["cores"], "kind": "reference", "sample": r["sample"], "fft": r["fft"]},
        "e2e": {"value": r["value"], "unit": "PCM frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm

def bind_to_gpu_numa_node(gpu_index):
    """8 ranks pulling their PCM through one socket's memory controllers was the end-to-end bottleneck of the 8 GPU run (GPUs 0-3 hang
    off NUMA node 0, 4-7 off node 1): restrict this process to the CPUs NVML reports as local to its GPU, so that first-touch places the
    pinned buffers there.  Best effort: returns what was done."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return "cpu affinity set to the GPU's local CPUs (%d)" % len(os.sched_getaffinity(0))
    except Exception as e:
        return "not bound: %s" % e


DUMP_FRAMES = 1 << 20                     # 8 MB of stereo float32 + 8 MB of frame numbers (the marked hour is 1.27 GB)
MATCH_TYPES = [c + b + s for c in ("", "CLIP-") for b in ("A", "B", "AB", "ALL") for s in ("", "-SPEED")]


def step_outputs(y_dev, n_frames, doc):
    """What a caller of the timed step receives, as arrays (see --dump-outputs): a seeded sample of the marked audio and the
    matches of the `get --json` document `doc` (None: no document on this rank)."""
    import numpy as np
    import torch
    idx = np.sort(np.random.default_rng(2024).choice(n_frames, min(n_frames, DUMP_FRAMES), replace=False))
    out = {"marked_frame": idx.astype(np.float64),
           "marked_audio": y_dev.index_select(0, torch.from_numpy(idx).to(y_dev.device)).cpu().numpy()}
    matches = json.loads(doc)["matches"] if doc is not None else []
    out["match_pos_s"] = np.array([sum(int(v) * 60 ** i for i, v in enumerate(reversed(m["pos"].split(":")))) for m in matches], np.float64)
    for f in ("quality", "error", "rating", "speed"):
        out["match_" + f] = np.array([m[f] for m in matches], np.float64)
    out["match_type"] = np.array([MATCH_TYPES.index(m["type"]) for m in matches], np.float64)
    out["match_bits"] = np.array([[(int(c, 16) >> (3 - b)) & 1 for c in m["bits"] for b in range(4)] for m in matches],
                                 np.float32).reshape(len(matches), 4 * len(PAYLOAD))
    return out


def main_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from audiowmark_b200 import hostapi as H

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout when the first communicator is created: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            torch.cuda.set_device(local)
            dist.all_reduce(torch.zeros(1, device=torch.device("cuda", local)))
            torch.cuda.synchronize()
            H.set_params(gpu_device=local)
            H.dist_init_from_torch()          # NCCL communicator of the C++ sharded get (its exchanges run on the context stream)
        finally:
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)       # pinned buffers and the host threads of this rank on the GPU's own NUMA node
    H.set_params(gpu_device=local)

    from audiowmark_b200 import sharding as S
    minutes = args.minutes if args.minutes else 60.0
    n = int(minutes * 60 * RATE)          # PCM frames per GPU (weak scaling: the stream is world * n frames long)
    ch = 2
    n_total = n * world
    mx, ov = H.chunk_geometry(RATE)
    plan = S.chunk_plan(n_total, mx, ov, RATE)
    assert H.frames_per_block() == S.T_BLOCK          # the Python plan functions below are written for the default block length
    if world == 1:
        e0, e1, ffn = 0, n, 0
    else:
        # frame-balanced shard: this rank searches an equal share of the start frames of every chunk (S.rank_slices) and
        # embeds exactly the PCM those slices read (+ the halo that makes its interior identical to the unsharded `add`)
        sl = S.rank_slices(plan, rank, world, n_total)
        own = (min(s.lo for s in sl), max(s.hi for s in sl))
        e0, e1, ffn = S.embed_range(own[0], own[1], n_total, RATE)
    n_loc = e1 - e0                       # frames this rank embeds (its chunks + halo)

    # synthetic input: uniform noise at -6 dBFS, a pure function of the stream position (blocks of 2^22 frames seeded by
    # block number) so that the ranges of neighbouring ranks agree where they overlap
    BLK = 1 << 22
    x_dev = torch.empty((max(n_loc, 1), ch), device=dev, dtype=torch.float32)
    g = torch.Generator(device=dev)
    for b in range(e0 // BLK, (max(e1, 1) - 1) // BLK + 1):
        g.manual_seed(1234 + b)
        blk = torch.rand((BLK, ch), device=dev, generator=g, dtype=torch.float32) - 0.5
        lo, hi = max(e0, b * BLK), min(e1, (b + 1) * BLK)
        if hi > lo:
            x_dev[lo - e0:hi - e0] = blk[lo - b * BLK:hi - b * BLK]
    del blk
    y_dev = torch.empty_like(x_dev)
    x_host = torch.empty((max(n_loc, 1), ch), dtype=torch.float32, pin_memory=True)
    y_host = torch.empty((max(n_loc, 1), ch), dtype=torch.float32, pin_memory=True)
    x_host.copy_(x_dev)
    # the same audio as 16 bit PCM (what a WAV file of the reference arm holds): floor (x * 32768), cf. src/sfoutputstream.cc:148-155
    x16_host = torch.empty((max(n_loc, 1), ch), dtype=torch.int16, pin_memory=True)
    y16_host = torch.empty((max(n_loc, 1), ch), dtype=torch.int16, pin_memory=True)
    x16_host.copy_(torch.floor(x_dev * 32768.0).clamp_(-32768, 32767).to(torch.int16))
    torch.cuda.synchronize()

    stream = torch.cuda.ExternalStream(H.gpu_stream(), device=dev)

    if world == 1:
        def step_resident():
            H.add(x_dev.data_ptr(), PAYLOAD, None, y_dev.data_ptr(), n, ch)
            return H.get(y_dev.data_ptr(), n_frames=n, channels=ch, parse=False)

        def step_e2e():
            H.add(x_host.numpy(), PAYLOAD, None, y_host.numpy())
            return H.get(y_host.numpy(), parse=False)

        def step_e2e_s16():
            H.add_s16(x16_host.numpy(), PAYLOAD, None, y16_host.numpy())
            return H.get_s16(y16_host.numpy(), parse=False)
    else:
        # one N-hour stream: `add` by frame blocks with halo (bit identical to the unsharded run), `get` by the C++ sharded driver
        # (host/awm_balanced.cc): three ncclAllGather exchanges of small lists, no PCM crosses NVLink
        def step_resident():
            H.add(x_dev.data_ptr(), PAYLOAD, None, y_dev.data_ptr(), n_loc, ch, first_frame_number=ffn)
            return H.balanced_get(y_dev.data_ptr(), e0, n_total, n_frames=n_loc, channels=ch, parse=False)

        def step_e2e():
            H.add(x_host.numpy(), PAYLOAD, None, y_host.numpy(), first_frame_number=ffn)
            return H.balanced_get(y_host.numpy(), e0, n_total, parse=False)

        def step_e2e_s16():
            H.add_s16(x16_host.numpy(), PAYLOAD, None, y16_host.numpy(), first_frame_number=ffn)
            return H.balanced_get(y16_host.numpy(), e0, n_total, parse=False)

    # A step ends with the `--json` document of `audiowmark get` as text (what the CLI writes); it is parsed and checked here, after the
    # timed region -- turning 100 to 900 patterns into Python objects is the checker's work, not the library's
    def check(doc):
        if doc is None:                       # sharded run: the merged result lives on rank 0
            return True, 0
        doc = json.loads(doc)
        real = [m for m in doc["matches"] if m["quality"] > 0.35]
        return len(real) > 0 and all(m["bits"] == PAYLOAD for m in real), len(real)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile):
        barrier()
        if profile:
            H.profile_enable(True)
        l0 = H.gpu_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        doc = None
        for _ in range(steps):
            doc = fn()
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        prof = H.profile_report() if profile else None
        if profile:
            H.profile_enable(False)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), wall, doc, H.gpu_launches() - l0, prof

    # the timed region of K steps lasts tens of milliseconds, less than nvidia-smi needs to deliver its first sample: the sampler
    # runs from before the warm-up until after the last timed e2e step (the GPU is under this load all the time)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    for _ in range(args.warmup):
        step_resident()
    ms, wall, doc, launches, prof = timed(step_resident, args.steps, True)
    dumped = step_outputs(y_dev, n_loc, doc) if args.dump_outputs and rank == 0 else None
    ok, n_real = check(doc)
    if args.resident_only:
        ms_e2e = ms_e2e16 = float("nan")
        ok2 = True
    else:
        for _ in range(min(args.warmup, 1)):
            step_e2e()
        ms_e2e, wall_e2e, doc2, _, _ = timed(step_e2e, args.steps, False)
        ok2, _ = check(doc2)
        for _ in range(min(args.warmup, 1)):
            step_e2e_s16()
        ms_e2e16, _, doc3, _, _ = timed(step_e2e_s16, args.steps, False)
        ok3, _ = check(doc3)
        ok2 = ok2 and ok3
    # the two halves of a step on their own (north_star's >= 100x target is on `get`); single GPU only
    halves = None
    if world == 1 and not args.resident_only:
        def sync_after(fn):
            def run():
                fn()
                H.synchronize()
            return run
        ms_add, _, _, _, _ = timed(sync_after(lambda: H.add(x_dev.data_ptr(), PAYLOAD, None, y_dev.data_ptr(), n, ch)), args.steps, False)
        ms_get, _, _, _, _ = timed(lambda: H.get(y_dev.data_ptr(), n_frames=n, channels=ch, parse=False), args.steps, False)
        ms_add16, _, _, _, _ = timed(sync_after(lambda: H.add_s16(x16_host.numpy(), PAYLOAD, None, y16_host.numpy())), args.steps, False)
        ms_get16, _, _, _, _ = timed(lambda: H.get_s16(y16_host.numpy(), parse=False), args.steps, False)
        halves = {"add_ms": ms_add / args.steps, "get_ms": ms_get / args.steps, "add_e2e_ms": ms_add16 / args.steps, "get_e2e_ms": ms_get16 / args.steps}
    if world == 1 and len(clocks.rows) < 8:         # very short runs: keep the load up until a few samples exist (single process only: the sharded step is collective)
        t_end = time.time() + 1.0
        while time.time() < t_end and len(clocks.rows) < 8:
            step_resident()
    clk = clocks.stop() if rank == 0 else None
    if clk is not None:
        clk["window"] = "warm-up + timed resident steps + e2e steps (nvidia-smi -lms 20)"

    sharded_equals_single = None
    if world > 1 and not args.resident_only:
        if rank == 0:
            # the whole N-hour stream once more on this GPU alone (the input is a pure function of the position): the merged document
            # of the sharded run has to be the single-GPU document, pattern for pattern
            try:
                xf = torch.empty((n_total, ch), device=dev, dtype=torch.float32)
                for b in range(0, (n_total - 1) // BLK + 1):
                    g.manual_seed(1234 + b)
                    blk = torch.rand((BLK, ch), device=dev, generator=g, dtype=torch.float32) - 0.5
                    hi = min(n_total, (b + 1) * BLK)
                    xf[b * BLK:hi] = blk[:hi - b * BLK]
                del blk
                yf = torch.empty_like(xf)
                torch.cuda.synchronize()
                H.add(xf.data_ptr(), PAYLOAD, None, yf.data_ptr(), n_total, ch)
                single = H.get(yf.data_ptr(), n_frames=n_total, channels=ch)
                sharded_equals_single = bool(single == json.loads(doc))
                del xf, yf
            except Exception as e:
                sharded_equals_single = "check failed: %s" % e
        barrier()
    det = torch.tensor([n_real, int(ok), int(ok2)], device=dev, dtype=torch.int64)
    if world > 1:
        gathered = [torch.zeros_like(det) for _ in range(world)]
        dist.all_gather(gathered, det)
        det_all = torch.stack(gathered).cpu().tolist()
    else:
        det_all = [det.cpu().tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_frames = n_total
    ms_step = ms / args.steps
    value = total_frames / (ms_step / 1e3)
    e2e_value = total_frames / (ms_e2e / args.steps / 1e3)
    e2e16_value = total_frames / (ms_e2e16 / args.steps / 1e3)
    # per-kernel picture and the roofline of the dominant kernel.
    # Algorithmic bytes follow SURVEY.md section 8(d): embed reads and writes every sample once (16 B per stereo PCM frame);
    # detect reads every chunk sample once (8 B) and writes + reads the four 81-band dB matrices (2 * 4 * 81 * 4 B per 1024 frames
    # = 2.53 B per frame): 10.53 B per frame of chunked input, 1.0747 x the stream length at 1 h.  Everything else a kernel moves
    # (the entry-sum matrix this implementation puts between spectrogram and search, refine / decode windows) is NOT algorithmic;
    # it shows up in `achieved_incl_intermediates` and in the measured DRAM traffic instead.
    peaks = measured_peaks()
    peak_gbs = (peaks or {}).get("hbm_gbs", 6650.0)
    overlap = 1.0747 if minutes >= 59 else 1.0                   # chunk overlap of `get` (SURVEY 8d)
    n_chunk_frames = n * overlap
    db_rw = 2 * 4 * 81 * 4 / 1024.0                              # 2.53 B / frame: dB matrices written once, read once
    survey_bytes = {                                             # per step and GPU
        "k_embed": 4.0 * ch * 2 * n,
        "k_embed_strip": 4.0 * ch * 2 * n,
        "k_stft_mags_tc": (4.0 * ch + db_rw / 2) * n_chunk_frames,   # PCM once + the dB matrices once
        "k_stft_mags": (4.0 * ch + db_rw / 2) * n_chunk_frames,
        "k_sync_gather": (db_rw / 2) * n_chunk_frames,               # the dB matrices read back
    }
    builder_bytes = {                                            # what the kernels of this implementation have to move
        "k_stft_mags_tc": (4.0 * ch + 4 * 510 * 8 / 1024.0) * n_chunk_frames,    # PCM once + entry sums (U, D) of 510 entries, 4 shifts
        "k_stft_mags": (4.0 * ch + 4 * 510 * 8 / 1024.0) * n_chunk_frames,
        "k_sync_gather": (4 * 510 * 8 / 1024.0) * n_chunk_frames,
        "k_embed": 4.0 * ch * 2 * n,
        "k_embed_strip": 4.0 * ch * 2 * n,
    }
    # dram__bytes_read.sum + dram__bytes_write.sum per PCM frame of kernel input, ncu --set full on a 10 min launch
    # (profiles/r2_ncu_full_final_add_get_10min.md; k_embed from profiles/r1_ncu_full_v4_all_kernels_10min.md)
    dram_per_frame = {"k_stft_mags_tc": (213.25e6 + 365.00e6) / 26.46e6, "k_embed": (213.32e6 + 170.57e6) / 26.46e6,
                      "k_embed_strip": (239.64e6 + 171.13e6) / 26.46e6}
    kernels = {}
    for name, r in (prof or {}).items():
        per_launch_ms = r["ms"] / max(r["launches"], 1)
        sb = survey_bytes.get(name, 0.0) * args.steps
        bb = (r.get("algo_bytes") or builder_bytes.get(name, 0.0) * args.steps)
        if name == "k_limiter":
            bb = 0.0                                             # CTAs whose blocks stay below the ceiling return at once: no meaningful byte count
        kernels[name] = {"launches": r["launches"], "ms_total": round(r["ms"], 4), "ms_per_launch": round(per_launch_ms, 5),
                         "share_of_step": round(r["ms"] / ms, 4),
                         "algo_GBps": round(sb / (r["ms"] / 1e3) / 1e9, 2) if sb else None,
                         "moved_GBps": round(bb / (r["ms"] / 1e3) / 1e9, 2) if bb else None}
    dominant = max(kernels, key=lambda k: kernels[k]["ms_total"]) if kernels else None
    roofline = None
    if dominant:
        k = kernels[dominant]
        a = k["algo_GBps"] or 0.0
        limiter = {"k_stft_mags_tc": "instruction latency / fp32 issue of the FFT warps (12 of the 17 warps, 3 per scheduler; ~1800 warp instructions per 1024-point stereo transform); the tcgen05 contraction, the TMA copies and the epilogue stores run underneath",
                   "k_refine_slide": "fp32 issue rate; the PCM window is re-read from L2",
                   "k_sync_gather": "HBM: one streaming pass over the entry-sum matrix",
                   "k_embed": "fp32 issue rate / latency of two FFTs per frame",
                   "k_embed_strip": "fp32 issue rate of two FFTs per frame (12 warps per SM, 167 registers)",
                   "k_viterbi": "serial dependency of 143 trellis steps"}
        launches_per_step = k["launches"] / args.steps
        traffic = dram_per_frame.get(dominant)
        if traffic is not None:
            traffic = traffic * (n if dominant.startswith("k_embed") else n_chunk_frames) / launches_per_step
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": a, "peak": peak_gbs, "unit": "GB/s", "frac": round(a / peak_gbs, 5),
                    "traffic": traffic,
                    "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture (10 min launch), scaled to this kernel's average launch of the step",
                    "achieved_incl_intermediates": k["moved_GBps"],
                    "actual_limiter": limiter.get(dominant),
                    "byte_model": "SURVEY.md 8(d): algorithmic bytes per launch / CUDA-event launch time",
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s"}
        # the whole path against the same roofline: 16 B / frame for embed + 10.53 B / frame of chunked input for detect
        path_bytes = 16.0 * n + 10.53 * n_chunk_frames
        roofline["path"] = {"algorithmic_bytes_per_step": path_bytes, "achieved": round(path_bytes / (ms_step / 1e3) / 1e9, 2),
                            "frac": round(path_bytes / (ms_step / 1e3) / 1e9 / peak_gbs, 5)}
        for ek in ("k_embed_strip", "k_embed"):
            if ek in kernels:
                roofline["embed_kernel"] = {"kernel": ek, "achieved": kernels[ek]["algo_GBps"], "frac": round((kernels[ek]["algo_GBps"] or 0.0) / peak_gbs, 4)}
                break
        if "k_sync_gather" in kernels:
            roofline["hbm_bound_kernel"] = {"kernel": "k_sync_gather", "moved_GBps": kernels["k_sync_gather"]["moved_GBps"],
                                            "frac_of_peak_moved": round((kernels["k_sync_gather"]["moved_GBps"] or 0.0) / peak_gbs, 4)}
    cpu = None
    if world == 1 and not args.no_cpu_baseline and not args.resident_only:
        try:
            r = run_reference(1, 0, minutes)
            cpu = {"value": r["value"], "unit": "PCM frames/s", "cores": r["cores"], "kind": "reference", "sample": r["sample"],
                   "t_add_s": round(r["t_add_s"], 3), "t_get_s": round(r["t_get_s"], 3), "add_value": r["add_value"], "get_value": r["get_value"],
                   "payload_ok": r["payload_ok"], "fft": r["fft"]}
        except Exception as e:          # the bench line must still print
            cpu = {"value": None, "unit": "PCM frames/s", "cores": os.cpu_count(), "kind": "reference", "sample": "unavailable: %s" % e}
    cli = None
    if world == 1 and not args.no_cpu_baseline and not args.resident_only:
        try:
            cli = run_cli_e2e(minutes)
        except Exception as e:
            cli = {"error": str(e)}
    add_get = None
    if halves:
        add_get = {"add": {"value": n / (halves["add_ms"] / 1e3), "ms_per_step": halves["add_ms"], "e2e_value": n / (halves["add_e2e_ms"] / 1e3), "e2e_ms_per_step": halves["add_e2e_ms"]},
                   "get": {"value": n / (halves["get_ms"] / 1e3), "ms_per_step": halves["get_ms"], "e2e_value": n / (halves["get_e2e_ms"] / 1e3), "e2e_ms_per_step": halves["get_e2e_ms"]},
                   "unit": "PCM frames/s"}
        if cpu and cpu.get("value"):
            add_get["add"]["e2e_vs_cpu_reference"] = round(add_get["add"]["e2e_value"] / cpu["add_value"], 1)
            add_get["get"]["e2e_vs_cpu_reference"] = round(add_get["get"]["e2e_value"] / cpu["get_value"], 1)
    line = {
        "metric": "audio frames/sec embed+detect, 44.1 kHz stereo; decoded-bit match vs ref",
        "value": value, "unit": "PCM frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%g min stereo 44.1 kHz embed+detect per GPU (BASELINE.json configs[1]%s)" % (minutes, "" if minutes == 60 else ", shortened"),
                   "pcm_frames_per_gpu": n, "channels": ch, "payload_bits": 128, "get_chunks": "30 min, 134.4 s overlap",
                   "parallelism": ("one %d h stream (%d chunks): every rank owns an equal span of positions -- `add` by frame blocks with halo, `get` by start-frame slices of each chunk (C++ driver, 3 ncclAllGather exchanges of small lists, no PCM exchanged)" % (world, len(plan))) if world > 1 else "1 GPU",
                   "l2": "inputs (%.2f GB per pass) larger than L2" % (n * ch * 4 / 1e9),
                   "result": "every step returns the `get --json` document as text (rank 0); parsed and checked after the timed region"},
        "analysis_frames_per_s": value / 1024.0,
        "payload_ok": bool(all(d[1] for d in det_all)), "detections": det_all[0][0],
        "sharded_equals_single_gpu": sharded_equals_single,
        # headline e2e: 16 bit PCM host buffers in and out -- what the WAV files of the reference arm hold; the int <-> float conversions of
        # SFInputStream / SFOutputStream run on the device (bit identical to converting on the host, tests/test_gpu_e2e.py)
        "e2e": {"value": e2e16_value, "unit": "PCM frames/s", "ms_per_step": ms_e2e16 / args.steps,
                "h2d_bytes_per_step": 2 * n_loc * ch * 2, "d2h_bytes_per_step": n_loc * ch * 2, "payload_ok": bool(all(d[2] for d in det_all)),
                "pcm": "s16 pinned host buffers (input, marked output, input of get)",
                "api": "hostapi.add_s16 + hostapi.get_s16 (C++ add_watermark_buffer_s16 / get_watermark_buffer_s16 -> awm_embed_s16, awm_pcm_prefetch_s16 ...)"},
        # the same with fp32 host buffers (what AudioInputStream::read_frames hands over inside the reference): twice the PCIe bytes
        "e2e_f32": {"value": e2e_value, "unit": "PCM frames/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": 2 * n_loc * ch * 4, "d2h_bytes_per_step": n_loc * ch * 4,
                    "api": "hostapi.add + hostapi.get (C++ add_watermark_buffer / get_watermark_buffer) on pinned fp32 host buffers"},
        "gpu_launches": launches,
        "add_get": add_get,
        "cli_e2e": cli,
        "roofline": roofline,
        "kernels": kernels,
        "host_wall_ms_per_step": 1e3 * wall / args.steps,
        "numa": numa,
        "cpu_baseline": cpu,
        "clocks": clk,
    }
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--minutes", type=float, default=0.0, help="audio length per GPU (default 60 = BASELINE configs[1], both arms)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--resident-only", action="store_true", help="only the resident legs (for the ncu launch list: every launch it sees belongs to a warm-up or timed resident step)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.impl == "reference":
        main_reference(args)
    else:
        main_gpu(args)


if __name__ == "__main__":
    main()
