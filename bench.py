#!/usr/bin/env python
"""bench.py -- throughput of the ns-nnsp streaming hot path on B200, next to the reference's CPU path.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --steps K --warmup W --dump-outputs DIR  (also writes the result records of the last timed step)

Headline workload (BASELINE.json `metric`, configs[4] at its per-GPU share): the full VAD -> KWS -> S2I gated cascade
(nnCntrlClass_exec, evb/src/nnCntrlClass.c:152-272) over 8,192 independent synthetic 16 kHz streams per GPU -- 65,536 at
N = 8 -- one step = 100 frames (1.0 s of audio) of every stream. The single-model configurations of BASELINE.json
(VAD x 4,096; KWS x 16,384 with ACC32BIT_OPT; S2I x 32,768 in total) are measured in the same run and reported in the
`configs` block of the same line.

One JSON line on stdout (rank 0):
  value         audio-seconds per second, PCM already resident in HBM; exactly K steps (after W warm-up steps, W raised to
                at least 3) timed with CUDA events on the engine's stream, MAX over ranks
  e2e           the same metric through the C ABI call with HOST (pinned) buffers: H2D + kernels + D2H inside
  roofline      the dominant kernel (feat_kernel) against the resource that binds it (issue slots), the HBM line next to it
  cpu_baseline  the reference's own C (oracle/_ref, unmodified sources, gcc -O2) on this host's cores, same PCM, same
                controller state per stream carried from step to step
  bit_exact_frame_pct   result records of a stream sample against that reference, taken outside the timed region

--dump-outputs DIR writes what the headline path returned to its caller in the last timed step: every field of the
[streams, frames] cascade result records of rank 0 (the only rank when N = 1) as DIR/<field>.npy in float32 (exact for
these integer fields, 23 MB in all).
The PCM is synthesised from fixed seeds and every step count is fixed by the arguments, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import hashlib
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME = 160
FRAMES_PER_STEP = 100
AUDIO_S_PER_FRAME = FRAME / 16000.0
CASCADE_STREAMS_PER_GPU = 8192                   # 65,536 / 8: BASELINE.json configs[4]
MODEL_FILE = {0: "s2i.nnspm", 1: "vad.nnspm", 2: "kws_galaxy.nnspm"}
# SURVEY.md section 8(d), algorithmic bytes per stream-frame of the whole path (one-frame-per-launch design):
#   S2I 2 872, KWS 2 824, VAD 2 608; the cascade adds the PCM ring (write 320 + look-back read 320) to the S2I figure
ALGO_BYTES = {"cascade": 2872 + 640, "vad": 2608, "kws": 2824, "s2i": 2872}
# single-model configurations of BASELINE.json: (name, nn_id, acc32, streams, how the streams scale with N)
SIDE_CONFIGS = [("vad", 1, False, 4096, "weak"), ("kws", 2, True, 16384, "weak"), ("s2i", 0, False, 32768, "strong")]
BIT_EXACT_SAMPLE = 48                            # streams of rank 0 compared with the reference, 300 frames each
REF_SAMPLE_PER_CORE = 96                         # CPU arms: sampled streams per core (about 0.5 s per step and core)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def capture(kernel, workload):
    """counters of one launch of `kernel` on `workload` from the committed ncu --set full capture (profiles/traffic.json:
    DRAM bytes, warp instructions, pipe utilisation), plus whether the kernel's sources still hash to what was captured"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            d = json.load(f)["%s@%s" % (kernel, workload)]
    except Exception:
        return None
    h = hashlib.sha256()
    for fn in d.get("source_files", []):
        try:
            with open(os.path.join(ROOT, fn), "rb") as f:
                h.update(f.read())
        except OSError:
            h.update(b"missing")
    d["capture_is_current"] = (h.hexdigest() == d.get("source_sha256"))
    return d


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed regions: NVML in-process (a sample every millisecond),
    nvidia-smi as the fall-back when pynvml is not importable."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device, self.sm, self.mx, self.reasons, self._stop_evt = device, [], [], set(), threading.Event()
        self.nvml = self.handle = None
        try:
            import pynvml
            from nnsp_b200.shard import nvml_handle
            self.nvml, self.handle = pynvml, nvml_handle(device)      # the GPU the kernels run on, by PCI bus id
            self.mx.append(int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(device):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x for x in vis.split(",") if x.strip() != ""]
            if device < len(ids) and ids[device].strip().isdigit():
                return int(ids[device])
        return device

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(int(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        r = int(get(self.handle))
        for name, bit in (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self._physical_index(self.device)), "--query-gpu=" + self.FIELDS,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [x.strip() for x in out.strip().split(",")]
        if len(parts) >= 6 and parts[0].isdigit():
            self.sm.append(int(parts[0]))
            if parts[1].isdigit():
                self.mx.append(int(parts[1]))
            for i in range(4):
                if parts[2 + i].lower().startswith("active"):
                    self.reasons.add(self.NAMES[i])

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop_evt.wait(0.001 if self.nvml is not None else 0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        return {"sm_mhz": int(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------
# the reference's own C implementation of the cascade on the host cores (cpu_baseline / --impl reference)
# ---------------------------------------------------------------------------------------------
_REF_PCM = None          # [2][n, T*160], set before the workers fork: they inherit the sample instead of receiving it


def _cpu_worker(conn, lo, hi):
    """One process = one instance of the (single-instance, SURVEY.md section 0.3) reference. It serves streams lo..hi-1
    in turn, every step continuing each stream's controller from where the previous step left it."""
    try:
        from oracle import pyoracle
        ref = pyoracle.RefLib.available(False)
        if ref:
            R = pyoracle.RefLib(False)
            states = np.zeros((hi - lo, R.cascade_state_bytes()), np.uint8)
        else:
            O = pyoracle.Oracle()
            models = [O.model(i, False) for i in range(3)]
        conn.send("reference" if ref else "port")
        while True:
            msg = conn.recv()
            if msg is None:
                break
            buf, fresh = msg
            t0 = time.perf_counter()
            if ref:
                R.cascade_batch(_REF_PCM[buf][lo:hi], states, fresh)
            else:                                         # the restatement keeps no state across calls: every step from reset
                O.cascade_batch_run(models, _REF_PCM[buf][lo:hi], n_threads=1)
            conn.send(time.perf_counter() - t0)
    except Exception as e:                                # noqa: BLE001
        conn.send("error: %r" % (e,))


class CpuCascade:
    def __init__(self, pcm_pair, cores):
        global _REF_PCM
        _REF_PCM = pcm_pair
        n = pcm_pair[0].shape[0]
        ctx = mp.get_context("fork")
        self.n, self.cores, self.procs, self.conns = n, cores, [], []
        for k in range(cores):
            lo, hi = n * k // cores, n * (k + 1) // cores
            if hi <= lo:
                continue
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(b, lo, hi), daemon=True)
            p.start()
            self.procs.append(p)
            self.conns.append(a)
        kinds = [c.recv() for c in self.conns]
        if any(str(k).startswith("error") for k in kinds):
            raise RuntimeError(kinds)
        self.kind = kinds[0]
        self.step_no = 0

    def step(self):
        """all sampled streams advance by one step (FRAMES_PER_STEP frames); returns wall seconds"""
        t0 = time.perf_counter()
        for c in self.conns:
            c.send((self.step_no & 1, self.step_no == 0))
        rep = [c.recv() for c in self.conns]
        dt = time.perf_counter() - t0
        if any(isinstance(r, str) for r in rep):
            raise RuntimeError(rep)
        self.step_no += 1
        return dt

    def close(self):
        global _REF_PCM
        for c in self.conns:
            try:
                c.send(None)
            except Exception:
                pass
        for p in self.procs:
            p.join(timeout=5)
        _REF_PCM = None


def cascade_pcm(rank, n_streams):
    """the two alternating PCM sets of a rank (consecutive steps never re-read L2-resident input)"""
    from nnsp_b200.synth import synth_pcm
    S = CASCADE_STREAMS_PER_GPU
    return [synth_pcm(n_streams, FRAMES_PER_STEP, first_stream=rank * S + k * 1000003) for k in range(2)]


def cpu_sample_size(cores):
    return min(CASCADE_STREAMS_PER_GPU, REF_SAMPLE_PER_CORE * cores)


def cpu_sample_text(n, cores, kind):
    return ("%d of rank 0's %d cascade streams x %d frames per step (the same PCM, each stream's controller state carried "
            "from step to step), %d forked processes, %s" % (
                n, CASCADE_STREAMS_PER_GPU, FRAMES_PER_STEP, cores,
                "oracle/_ref = unmodified reference C (nnCntrlClass_exec, gcc -O2)" if kind == "reference"
                else "oracle/nnsp_oracle.c port (restarts every step)"))


def workload_config(n_gpus):
    S, T = CASCADE_STREAMS_PER_GPU, FRAMES_PER_STEP
    return {"workload": "full VAD -> KWS -> S2I gated cascade (nnCntrlClass {vad, kws_galaxy, s2i}, thresholds of ParamsNNCntrl.h, "
                        "acc64) x %d streams per GPU x %d frames (%.1f s audio) per step; FeatureClass -> NeuralNetClass -> NNSPClass "
                        "-> controller, bit-exact vs reference C" % (S, T, T * AUDIO_S_PER_FRAME),
            "streams_per_gpu": S, "frames_per_step": T, "total_streams": S * n_gpus,
            "partition": "streams block-partitioned over GPUs, no data-path collective",
            "cache": "two alternating %d MB PCM buffers per GPU (larger than the 126 MB L2)" % (S * T * FRAME * 2 // 1000000)}


METRIC = "audio-sec/sec (16 kHz streams, VAD+KWS+S2I cascade)"
DTYPE = "int16 activations x int8 weights, int32/int64 accumulate (bit-exact integer path)"


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n = cpu_sample_size(cores)
    arm = CpuCascade(cascade_pcm(0, n), cores)
    for _ in range(args.warmup):
        arm.step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.step()
    dt = time.perf_counter() - t0
    arm.close()
    value = args.steps * n * FRAMES_PER_STEP * AUDIO_S_PER_FRAME / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": arm.kind,
                             "sample": cpu_sample_text(n, cores, arm.kind)},
            "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
class Timer:
    """W warm-up steps (W >= 3, see main), then exactly K steps between two CUDA events on the handle's stream, a barrier + synchronize on
    both sides; the time is the MAX over ranks."""

    def __init__(self, nb, device, dist):
        self.nb, self.device, self.dist = nb, device, dist
        self.ev0, self.ev1 = nb.Event(device), nb.Event(device)

    def barrier(self, h):
        h.sync()
        if self.dist is not None:
            self.dist.barrier()
        h.sync()

    def allmax(self, values):
        if self.dist is None:
            return [float(v) for v in values]
        import torch
        t = torch.tensor(list(values), dtype=torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def once(self, h, step, K):
        self.barrier(h)
        self.ev0.record(h.stream)
        for i in range(K):
            step(i)
        h.sync()                                       # every stream of the handle (calls are pipelined over several)
        self.ev1.record(h.stream)
        h.sync()
        return self.ev0.elapsed_ms_to(self.ev1)

    def run(self, h, step, K, W):
        for i in range(W):
            step(i)
        return self.allmax([self.once(h, step, K)])[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps before each timed region (at least 3 for the b200 implementation)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the cascade results of the last timed step as DIR/<field>.npy "
                    "(b200 implementation only; under torchrun rank 0's streams only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 implementation; the reference arm only times its steps")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import nnsp_b200 as nb
    from nnsp_b200.synth import synth_pcm

    S, T, K, W = CASCADE_STREAMS_PER_GPU, FRAMES_PER_STEP, args.steps, args.warmup
    host_pcm = cascade_pcm(rank, S)

    # CPU baseline first (rank 0, N = 1 only), before the GPU context makes fork() unsafe: ~15-25 core-seconds
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        n = cpu_sample_size(cores)
        arm = CpuCascade([p[:n] for p in host_pcm], cores)
        arm.step(); arm.step()                          # from reset into the steady stage mix
        dts = [arm.step() for _ in range(3)]
        kind = arm.kind
        arm.close()
        cpu_baseline = {"value": n * T * AUDIO_S_PER_FRAME / min(dts), "unit": "audio-s/s", "cores": cores, "kind": kind,
                        "sample": cpu_sample_text(n, cores, kind) + "; best of 3 steps after 2 warm-up steps"}

    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the one JSON line
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    device = local_rank

    bound = set()
    if os.environ.get("NNSP_BENCH_BIND", "1") != "0":
        from nnsp_b200.shard import bind_host_to_device
        bound = bind_host_to_device(device)

    tm = Timer(nb, device, dist)
    models = [nb.Model.from_blob(os.path.join(nb.MODEL_DIR, MODEL_FILE[i])) for i in range(3)]
    casc = nb.Cascade(models, S, device=device)
    dev_pcm = [nb.DeviceArray.from_host(p, device) for p in host_pcm]
    dev_res = nb.DeviceArray((S, T), nb.CASCADE_RESULT_DT, device)

    # ---- bit-exact frame % : the first 300 frames of a stream sample against the reference, outside any timed region --
    parts = []
    for i in range(3):
        casc.exec_device(dev_pcm[i & 1], T * FRAME, T, dev_res)
        casc.sync()
        parts.append(dev_res.to_host())
    bit_exact = None
    if rank == 0:
        from oracle import pyoracle
        got = np.concatenate(parts, axis=1)
        idx = np.unique(np.linspace(0, S - 1, BIT_EXACT_SAMPLE).astype(np.int64))
        use_ref = pyoracle.RefLib.available(False)
        chk = pyoracle.RefLib(False) if use_ref else pyoracle.Oracle()
        om = None if use_ref else [chk.model(i, False) for i in range(3)]
        same = total = 0
        for s in idx:
            x = np.concatenate([host_pcm[0][s], host_pcm[1][s], host_pcm[0][s]])
            want = chk.cascade_run(x, taps=False)[0] if use_ref else chk.cascade_run(om, x, taps=False)[0]
            ok = np.ones(len(want), bool)
            for f in want.dtype.names:
                ok &= (got[s][f] == want[f]).reshape(len(want), -1).all(axis=1)
            same += int(ok.sum()); total += len(want)
        bit_exact = {"pct": 100.0 * same / total, "frames": total,
                     "sample": "%d streams of rank 0 x 300 frames from reset, every field of the 12-byte result record "
                               "(stage, position, detection, outputs, time-out counter) against %s; every layer tap is "
                               "compared by tests/ (test_gpu_cascade.py, test_gpu_fullsize.py)" % (
                                   len(idx), "oracle/_ref (unmodified reference C)" if use_ref else "oracle/nnsp_oracle.c")}
    del parts

    # ---- headline: device-resident cascade -------------------------------------------------------------------------
    def step(i):
        casc.exec_device(dev_pcm[i & 1], T * FRAME, T, dev_res)

    sampler = ClockSampler(device)
    sampler.start()
    ms_total = tm.run(casc, step, K, W)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:                  # dev_res holds the last timed step's records until the next step
        last = dev_res.to_host()
        os.makedirs(args.dump_outputs, exist_ok=True)
        for f in last.dtype.names:
            np.save(os.path.join(args.dump_outputs, f + ".npy"), last[f].astype(np.float32))
        del last
    km = []
    for i in range(5):                                  # per-kernel durations: CUDA events the engine records around its launches
        step(i)
        casc.sync()
        km.append(casc.last_kernel_ms())
    feat_ms = float(np.mean([k[0] for k in km]))
    nn_ms = float(np.mean([k[1] for k in km]))
    stage = np.bincount(dev_res.to_host()["stage_id"].ravel().astype(np.int64), minlength=3).tolist()
    n0 = nb.kernel_launches()
    tm.once(casc, step, K)
    gpu_launches = int(nb.kernel_launches() - n0)

    # ---- end to end through the host-buffer entry point (pinned host memory -> H2D -> kernels -> D2H) ----------------
    pin = [nb.PinnedArray((S, T * FRAME), np.int16) for _ in range(2)]
    for k in range(2):
        pin[k].array[...] = host_pcm[k]
    pin_res = [nb.PinnedArray((S, T), nb.CASCADE_RESULT_DT) for _ in range(2)]
    det = [r.array["detected"] for r in pin_res]

    def e2e_loop(n):
        fired, prev = 0, None
        for i in range(n):
            tk = casc.exec_host_async(pin[i & 1].array, pin_res[i & 1].array)
            if prev is not None:
                casc.wait_host(prev)
                fired += int(np.count_nonzero(det[(i - 1) & 1]))       # the host reads the step's result
            prev = tk
        casc.wait_host(prev)
        return fired + int(np.count_nonzero(det[(n - 1) & 1]))

    def e2e_once():
        tm.barrier(casc)
        t0 = time.perf_counter()
        e2e_loop(K)
        return time.perf_counter() - t0

    e2e_loop(3)
    sampler = ClockSampler(device)
    sampler.start()
    e2e_s = tm.allmax([e2e_once()])[0]
    clocks_e2e = sampler.stop()
    clocks["e2e"] = {k: clocks_e2e[k] for k in ("sm_mhz", "reasons", "samples")}
    clocks["reasons"] = sorted(set(clocks["reasons"]) | set(clocks_e2e["reasons"]))
    tm.barrier(casc)
    t0 = time.perf_counter()                             # the same with one blocking call per step (nothing in flight across calls)
    for i in range(K):
        casc.exec_host(pin[i & 1].array, pin_res[i & 1].array)
    e2e_sync_s = time.perf_counter() - t0
    # what the host link delivers when every rank copies at once: the ceiling of any end-to-end number on this box
    L = nb.capi.lib()
    tm.barrier(casc)
    link_s = []
    for _ in range(3):                                   # four copies back to back per timing: the sustained rate, as the e2e loop sees it
        tm.barrier(casc)
        t0 = time.perf_counter()
        for i in range(4):
            nb.capi.check(L.nnsp_b200_memcpy_h2d(device, dev_pcm[i & 1].ptr, pin[i & 1].ptr, pin[0].nbytes))
        link_s.append((time.perf_counter() - t0) / 4)
    link_gbs = -tm.allmax([-pin[0].nbytes / min(link_s) / 1e9])[0]       # the slowest rank's rate
    h2d_bytes, d2h_bytes = S * T * FRAME * 2, S * T * 12

    for x in pin + pin_res + dev_pcm:
        x.free()
    dev_res.free()
    casc.close()

    # ---- the single-model configurations of BASELINE.json, device-resident, in the same run ---------------------------
    side = []
    if not args.no_side_configs:
        for name, nn_id, acc32, streams, scaling in SIDE_CONFIGS:
            Sg = streams // world if scaling == "strong" else streams
            m = nb.Model.from_blob(os.path.join(nb.MODEL_DIR, MODEL_FILE[nn_id]), acc32=acc32)
            b = nb.NNSPBatch(m, Sg, device=device)
            pool = min(Sg, 2048)
            base = synth_pcm(pool, T, first_stream=rank * 100003 + 17)
            pcm = np.tile(base, ((Sg + pool - 1) // pool, 1))[:Sg]
            d = [nb.DeviceArray.from_host(pcm, device), nb.DeviceArray.from_host(np.roll(pcm, 7, axis=0), device)]
            res = nb.DeviceArray((Sg, T), nb.RESULT_DT, device)
            fn = lambda i: b.exec_device(d[i & 1], T * FRAME, T, res)
            tc0, kl0 = nb.tc5_launches(), nb.kernel_launches()
            ms = tm.run(b, fn, K, W)
            tc5_share = (nb.tc5_launches() - tc0, nb.kernel_launches() - kl0)
            kk = []
            for i in range(3):
                fn(i); b.sync(); kk.append(b.last_kernel_ms())
            f_ms, n_ms = float(np.mean([k[0] for k in kk])), float(np.mean([k[1] for k in kk]))
            peak, _ = measured_peaks()
            ach = ALGO_BYTES[name] * Sg * T / (f_ms * 1e-3) / 1e9
            side.append({"config": "%s x %d streams%s%s" % (name.upper(), streams, " (ACC32BIT_OPT)" if acc32 else "",
                                                          " in total over the GPUs" if scaling == "strong" else " per GPU"),
                         "scaling": scaling, "streams_per_gpu": Sg,
                         "value": world * Sg * T * AUDIO_S_PER_FRAME * K / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms / K,
                         "kernel_ms": {"feat_kernel": f_ms, "network_kernels": n_ms},
                         "tcgen05_launches": "%d of %d launches (layer 0, seg0_tc5_kernel)" % tc5_share,
                         "roofline_hbm": {"kernel": "feat_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                          "algorithmic_bytes_per_stream_frame": ALGO_BYTES[name]}})
            for x in d:
                x.free()
            res.free()
            b.close()

    if rank == 0:
        audio_s = world * S * T * AUDIO_S_PER_FRAME * K
        value = audio_s / (ms_total * 1e-3)
        peak, peak_src = measured_peaks()
        frames = S * T
        ach = ALGO_BYTES["cascade"] * frames / (feat_ms * 1e-3) / 1e9
        cap = capture("feat_kernel", "cascade")
        sm_mhz = clocks.get("sm_mhz") or 1965
        issue_peak = 4.0 * 148 * sm_mhz * 1e6 / 1e9           # one warp instruction per clock per SM sub-partition, Ginst/s
        hbm_line = {"achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": ALGO_BYTES["cascade"] * frames,
                    "note": "SURVEY.md 8(d) whole-path algorithmic bytes per stream-frame (%d B, cascade) x %d frames per launch / "
                            "feat_kernel launch time; the kernel's own traffic is `traffic` (its 320 B of PCM in and its 160 B "
                            "log-mel row out per frame)" % (ALGO_BYTES["cascade"], frames)}
        if cap and cap.get("warp_instructions_per_frame"):
            winst = cap["warp_instructions_per_frame"] * frames
            roofline = {"bound": "issue", "kernel": "feat_kernel", "achieved": winst / (feat_ms * 1e-3) / 1e9, "peak": issue_peak,
                        "unit": "Ginst/s (warp instructions)", "frac": winst / (feat_ms * 1e-3) / 1e9 / issue_peak,
                        "traffic": cap.get("dram_bytes_per_frame", 0) * frames or None, "launch_ms": feat_ms,
                        "warp_instructions_per_launch": winst, "pipe_fmaheavy_pct": cap.get("pipe_fmaheavy_pct"),
                        "pipe_alu_pct": cap.get("pipe_alu_pct"), "capture": cap.get("source"),
                        "capture_is_current": cap["capture_is_current"],
                        "note": "integer kernel: the binding resource is the issue slots / the FMA-heavy pipe (IMAD.WIDE = 4 cycles), "
                                "not HBM and not the tensor pipe. peak = 4 schedulers x 148 SMs x the SM clock sampled in this run; "
                                "instruction and DRAM counts per frame from the committed ncu capture, the duration measured live",
                        "hbm": hbm_line}
        else:
            roofline = dict(hbm_line, bound="hbm", kernel="feat_kernel", traffic=None, launch_ms=feat_ms,
                            note=hbm_line["note"] + "; no current ncu capture of this workload is committed, so the issue-slot line is omitted")
        ipk = nb.int_peak(device)
        line = {
            "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic", "config": workload_config(world),
            "timing": {"timed_steps": K, "timed_region_s": ms_total * 1e-3,
                       "rule": "`warmup` steps, then exactly `steps` steps between CUDA events, barrier + synchronize on both "
                               "sides, MAX over ranks"},
            "bit_exact_frame_pct": bit_exact["pct"] if bit_exact else None, "bit_exact": bit_exact,
            "stage_frames_last_step": {"s2i": stage[0], "vad": stage[1], "kws": stage[2]},
            "e2e": {"value": audio_s / e2e_s, "unit": "audio-s/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": 1e3 * e2e_s / K, "timed_region_s": e2e_s,
                    "call": "nnsp_b200_cascade_exec_host_async + _wait_host, two pinned buffer pairs, results of every step read on the host",
                    "blocking_call_value": (audio_s / world) / e2e_sync_s if world == 1 else None,
                    "link_gbs": link_gbs, "link_frac": (h2d_bytes * K / e2e_s / 1e9) / link_gbs,
                    "link_note": "link_gbs = sustained pinned H2D rate (4 x 262 MB back to back, best of 3) of the slowest rank with all %d ranks copying at once; link_frac = "
                                 "this run's H2D rate / that: the host link, not a kernel, bounds the end-to-end number" % world},
            "gpu_launches": gpu_launches,
            "clocks": clocks,
            "roofline": roofline,
            "int_alu": {"peak_gops_imad": ipk["imad"], "peak_gops_mixed": ipk["mixed"], "peak_gops_imad_wide": ipk["imad_wide"],
                        "peak_gops_idp2a": ipk["idp2a"],
                        "peak_source": "self-measured nnsp_b200_int_peak (register-resident dependent chains), giga lane-instructions/s"},
            "kernel_ms": {"feat_kernel": feat_ms, "controller_and_network_kernels": nn_ms,
                          "path": "feat_kernel (log-mel of every raw frame) -> per round: stage-sorted seg/scan/seg kernels per model + "
                                  "controller walk -> sequential kernel for what is left"},
            "host": {"bound_cpus": len(bound)},
            "configs": side,
        }
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
