#!/usr/bin/env python
"""Ragged cascade calls against uniform ones: the shipped VAD -> KWS -> S2I cascade over 8 192 streams in 100-frame device
calls (two PCM buffers used alternately, as bench.py's headline cascade does), four arms on handles of their own:
  uniform     nnsp_b200_cascade_exec
  full        nnsp_b200_cascade_exec_ragged, every count 100
  jitter      ragged, seeded counts in [95, 100]
  idle25      ragged, 25 % of the streams idle (count 0), the rest uniform in [1, 100]
Each arm: 5 warm-up calls, then 20 timed calls between two CUDA events with a synchronise on both sides; the arms take turns
(--rounds times) so that drift on the shared host hits all of them alike. Prints the card name and power limit, then one
JSON line per arm: median ms per call over the rounds and audio-seconds per second counted on the frames the streams
actually advanced. usage: python tools/ragged_calls.py [--streams 8192] [--frames 100] [--rounds 3]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import nnsp_b200 as nb  # noqa: E402

FILES = ("s2i.nnspm", "vad.nnspm", "kws_galaxy.nnspm")


def card(device):
    """name and power limit of the card, read through nvidia-smi by PCI bus id"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", nb.device_pci_bus_id(device), "--query-gpu=name,power.limit",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = (x.strip() for x in out.split(","))
        return name, power
    except Exception as e:                  # the timing itself still needs the GPU and fails without one
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=8192)
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--device", type=int, default=0)
    a = ap.parse_args()
    S, T, dev = a.streams, a.frames, a.device
    name, power = card(dev)
    print(json.dumps({"card": name, "power_limit": power, "streams": S, "frames_per_call": T, "warmup": a.warmup,
                      "steps": a.steps, "rounds": a.rounds}), flush=True)
    rng = np.random.default_rng(0x72616767)
    counts = {"uniform": None, "full": [np.full(S, T, np.int32)],
              "jitter": [rng.integers(T - 5, T + 1, S).astype(np.int32) for _ in range(8)],
              "idle25": [np.where(rng.random(S) < 0.25, 0, rng.integers(1, T + 1, S)).astype(np.int32) for _ in range(8)]}
    models = [nb.Model.from_blob(os.path.join(nb.MODEL_DIR, f)) for f in FILES]
    pcm = [nb.DeviceArray.from_host(nb.synth_pcm(S, T, first_stream=k * 1000003), dev) for k in range(2)]
    res = nb.DeviceArray((S, T), nb.CASCADE_RESULT_DT, dev)
    arms = {}
    for arm, cs in counts.items():
        h = nb.Cascade(models, S, device=dev)
        d_counts = [nb.DeviceArray.from_host(c, dev) for c in cs] if cs is not None else None

        def step(i, h=h, d_counts=d_counts):
            if d_counts is None:
                h.exec_device(pcm[i & 1], T * 160, T, res)
            else:
                h.exec_ragged_device(pcm[i & 1], T * 160, T, d_counts[i % len(d_counts)], res)
        frames = [T * S] if cs is None else [int(c.sum()) for c in cs]
        arms[arm] = dict(h=h, step=step, frames=frames, ms=[], keep=d_counts)
    ev0, ev1 = nb.Event(dev), nb.Event(dev)
    for _ in range(a.rounds):
        for arm, x in arms.items():
            h, step = x["h"], x["step"]
            for i in range(a.warmup):
                step(i)
            h.sync()
            ev0.record(h.stream)
            for i in range(a.steps):
                step(i)
            h.sync()
            ev1.record(h.stream)
            h.sync()
            x["ms"].append(ev0.elapsed_ms_to(ev1) / a.steps)
    for arm, x in arms.items():
        ms = float(np.median(x["ms"]))
        frames = np.mean([x["frames"][i % len(x["frames"])] for i in range(a.steps)])
        print(json.dumps({"arm": arm, "ms_per_call": round(ms, 4), "ms_each_round": [round(v, 4) for v in x["ms"]],
                          "frames_advanced_per_call": int(frames), "audio_s_per_s": round(frames * 0.01 / (ms * 1e-3), 1)}),
              flush=True)
        x["h"].close()


if __name__ == "__main__":
    main()
