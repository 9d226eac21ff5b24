#!/usr/bin/env python
"""Cost of per-stream resets (nnsp_b200_cascade_reset_streams) on back-to-back device calls: the shipped VAD -> KWS -> S2I
cascade over 8 192 streams in 100-frame device calls (two PCM buffers used alternately, as bench.py's headline cascade
does), three arms on handles of their own:
  none        no resets
  fresh1pct   1 % of the streams rounded up (82 of 8 192), a different seeded set each call, reset FRESH before every call
  all         every stream reset FRESH before every call
Each arm: 5 warm-up calls, then 20 timed calls between two CUDA events with a synchronise on both sides; the arms take turns
(--rounds times) so that drift on the shared host hits all of them alike. After each timed window the handle's timeline
(nnsp_b200_cascade_timeline, last 8 calls) gives how long the front end of call k + 1 ran while the controller / network
chain of call k was still running. Prints the card name and power limit, then one JSON line per arm: median ms per call
over the rounds and the median overlap per call pair. usage: python tools/reset_calls.py [--streams 8192] [--rounds 5]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import nnsp_b200 as nb  # noqa: E402
from ragged_calls import FILES, card  # noqa: E402


def overlap_ms(tl):
    """mean over consecutive calls of the time call k + 1's front end ran inside call k's chain"""
    ov = [max(0.0, min(tl[k + 1][1], tl[k][3]) - max(tl[k + 1][0], tl[k][2])) for k in range(len(tl) - 1)]
    return float(np.mean(ov)) if ov else 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=8192)
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--device", type=int, default=0)
    a = ap.parse_args()
    S, T, dev = a.streams, a.frames, a.device
    name, power = card(dev)
    print(json.dumps({"card": name, "power_limit": power, "streams": S, "frames_per_call": T, "warmup": a.warmup,
                      "steps": a.steps, "rounds": a.rounds}), flush=True)
    rng = np.random.default_rng(0x72657365)
    lists = {"none": None,
             "fresh1pct": [np.sort(rng.choice(S, -(-S // 100), replace=False)).astype(np.int32) for _ in range(8)],
             "all": [np.arange(S, dtype=np.int32)]}
    models = [nb.Model.from_blob(os.path.join(nb.MODEL_DIR, f)) for f in FILES]
    pcm = [nb.DeviceArray.from_host(nb.synth_pcm(S, T, first_stream=k * 1000003), dev) for k in range(2)]
    res = nb.DeviceArray((S, T), nb.CASCADE_RESULT_DT, dev)
    arms = {}
    for arm, ls in lists.items():
        h = nb.Cascade(models, S, device=dev)

        def step(i, h=h, ls=ls):
            if ls is not None:
                h.reset_streams(ls[i % len(ls)], fresh=True)
            h.exec_device(pcm[i & 1], T * 160, T, res)
        arms[arm] = dict(h=h, step=step, ms=[], overlap=[])
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
            x["overlap"].append(overlap_ms(h.timeline()))
    for arm, x in arms.items():
        n = 0 if lists[arm] is None else len(lists[arm][0])
        print(json.dumps({"arm": arm, "streams_reset_per_call": n, "ms_per_call": round(float(np.median(x["ms"])), 4),
                          "ms_each_round": [round(v, 4) for v in x["ms"]],
                          "overlap_ms_per_call": round(float(np.median(x["overlap"])), 4),
                          "overlap_each_round": [round(v, 4) for v in x["overlap"]]}), flush=True)
        x["h"].close()


if __name__ == "__main__":
    main()
