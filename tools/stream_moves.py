#!/usr/bin/env python
"""Cost of moving sessions (nnsp_b200_cascade_export_streams / _import_streams) on back-to-back device calls: the shipped
VAD -> KWS -> S2I cascade over 8 192 streams in 100-frame device calls (two PCM buffers used alternately, as bench.py's
headline cascade does), five arms on handles of their own:
  none         no exports or imports
  import82     1 % of the streams rounded up (82 of 8 192), a different seeded set each call, imported before every call
  export82     82 streams exported after every call (synchronous: the next call starts on an idle device)
  import_all   every stream imported before one call: that call, from the import to its synchronise
  export_all   an export of every stream from an idle handle
The first three: 5 warm-up calls, then 20 timed calls between two CUDA events with a synchronise on both sides, and after
each timed window the timeline overlap (nnsp_b200_cascade_timeline, last 8 calls: how long the front end of call k + 1 ran
while the chain of call k still ran). The last two: host clock around one operation that ends in a synchronise. The arms
take turns (--rounds times) so that drift on the shared host hits all of them alike. Prints the card name and power
limit, then one JSON line per arm with medians over the rounds. usage: python tools/stream_moves.py [--streams 8192]"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import nnsp_b200 as nb  # noqa: E402
from ragged_calls import FILES, card  # noqa: E402
from reset_calls import overlap_ms  # noqa: E402


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
    rng = np.random.default_rng(0x6d6f7665)
    few = [np.sort(rng.choice(S, -(-S // 100), replace=False)).astype(np.int32) for _ in range(8)]
    every = np.arange(S, dtype=np.int32)
    models = [nb.Model.from_blob(os.path.join(nb.MODEL_DIR, f)) for f in FILES]
    pcm = [nb.DeviceArray.from_host(nb.synth_pcm(S, T, first_stream=k * 1000003), dev) for k in range(2)]
    res = nb.DeviceArray((S, T), nb.CASCADE_RESULT_DT, dev)
    src = nb.Cascade(models, S, device=dev)                # records of live streams: two calls in
    for i in range(2):
        src.exec_device(pcm[i], T * 160, T, res)
    recs_all = src.export_streams(every)
    rb = src.stream_state_bytes()
    src.close()
    recs_few = [b"".join(recs_all[s * rb:(s + 1) * rb] for s in ls) for ls in few]
    piped = {}
    for arm in ("none", "import82", "export82"):
        h = nb.Cascade(models, S, device=dev)

        def step(i, h=h, arm=arm):
            if arm == "import82":
                h.import_streams(few[i % len(few)], recs_few[i % len(few)])
            h.exec_device(pcm[i & 1], T * 160, T, res)
            if arm == "export82":
                h.export_streams(few[i % len(few)])
        piped[arm] = dict(h=h, step=step, ms=[], overlap=[])
    whole = {arm: dict(h=nb.Cascade(models, S, device=dev), ms=[]) for arm in ("import_all", "export_all")}
    ev0, ev1 = nb.Event(dev), nb.Event(dev)
    for _ in range(a.rounds):
        for arm, x in piped.items():
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
        for arm, x in whole.items():
            h = x["h"]
            for i in range(2):
                h.exec_device(pcm[i], T * 160, T, res)
            h.sync()
            t0 = time.perf_counter()
            if arm == "import_all":
                h.import_streams(every, recs_all)
                h.exec_device(pcm[0], T * 160, T, res)
                h.sync()
            else:
                h.export_streams(every)
            x["ms"].append((time.perf_counter() - t0) * 1e3)
    for arm, x in piped.items():
        print(json.dumps({"arm": arm, "streams_per_call": 0 if arm == "none" else len(few[0]),
                          "ms_per_call": round(float(np.median(x["ms"])), 4), "ms_each_round": [round(v, 4) for v in x["ms"]],
                          "overlap_ms_per_call": round(float(np.median(x["overlap"])), 4),
                          "overlap_each_round": [round(v, 4) for v in x["overlap"]]}), flush=True)
        x["h"].close()
    for arm, x in whole.items():
        print(json.dumps({"arm": arm, "streams": S, "record_bytes": rb, "ms": round(float(np.median(x["ms"])), 3),
                          "ms_each_round": [round(v, 3) for v in x["ms"]]}), flush=True)
        x["h"].close()


if __name__ == "__main__":
    main()
