#!/usr/bin/env python
"""Layer-0 kernel time per staged row: seg_kernel<2> of every cascade round (log-mel rows standardised while staging) next
to seg_kernel<1> of the batched S2I configuration (standardised int16 rows), from a torch.profiler trace.

Launches are serialised (CUDA_LAUNCH_BLOCKING=1, set here before CUDA starts), so a launch's duration is its own and not
shared with the group kernels of the other models or the next call's front end. Rows are (stream, inference) pairs: in
round k a stream whose k-th stage of the call starts at frame t runs (T - t + 1) // 2 inferences to the end of the call,
read off the stage_id of the call's result records.
usage: python tools/seg_stage_times.py [streams] [frames] [calls]   (defaults: bench.py's cascade shape, 8 192 x 100, 5 calls)"""
import collections
import json
import os
import sys
import tempfile

os.environ["CUDA_LAUNCH_BLOCKING"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402
import nnsp_b200 as nb  # noqa: E402

S = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
T = int(sys.argv[2]) if len(sys.argv) > 2 else 100
CALLS = int(sys.argv[3]) if len(sys.argv) > 3 else 5
S2I_STREAMS = 32768                                   # bench.py's S2I configuration on one GPU
SEQ = ("vad", "kws", "s2i")                           # group launch order of a round: the controller's sequence
ROUNDS = 3                                            # NNSP_B200_CASCADE_ROUNDS default


def kernels(prof, tag):
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "trace.json")
        prof.export_chrome_trace(p)
        ev = json.load(open(p))["traceEvents"]
    ks = [e for e in ev if e.get("cat") == "kernel" and tag in e.get("name", "")]
    return sorted(ks, key=lambda e: e["args"]["correlation"])


def round_rows(res):
    """rows[k][model] of one call from its result records (stage_id per frame)"""
    rows = collections.defaultdict(lambda: collections.Counter())
    st = res["stage_id"].astype(int)
    for s in range(st.shape[0]):
        starts = [0] + [int(t) for t in np.nonzero(np.diff(st[s]))[0] + 1]
        for k, t in enumerate(starts[:ROUNDS]):
            rows[k][int(st[s, t])] += (T - t + 1) // 2
    return rows


pool = min(S, 2048)
base = nb.synth_pcm(pool, T)
pcm = np.tile(base, ((S + pool - 1) // pool, 1))[:S]
d = [nb.DeviceArray.from_host(pcm), nb.DeviceArray.from_host(np.roll(pcm, 7, axis=0))]
models = [nb.Model.from_blob(os.path.join(nb.MODEL_DIR, f)) for f in ("s2i.nnspm", "vad.nnspm", "kws_galaxy.nnspm")]
h = nb.Cascade(models, S)
res = nb.DeviceArray((S, T), nb.CASCADE_RESULT_DT)
for i in range(20):
    h.exec_device(d[i & 1], T * 160, T, res)
h.sync()
rows = []
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for i in range(CALLS):
        h.exec_device(d[i & 1], T * 160, T, res)
        h.sync()
        rows.append(round_rows(res.to_host()))
seg2 = kernels(prof, "seg_kernel<2>")
per_call = len(seg2) // CALLS
assert per_call == ROUNDS * len(SEQ), "expected %d seg_kernel<2> launches per call, got %d" % (ROUNDS * len(SEQ), per_call)
h.close()

print("# %s, lib %s; cascade x %d streams x %d frames, %d calls, launches serialised" % (
    torch.cuda.get_device_name(0), os.path.basename(os.environ.get("NNSP_B200_LIB", "product")), S, T, CALLS))
print("# kernel           round  model  launches   us/launch   rows/launch   ns/row")
ids = {"s2i": 0, "vad": 1, "kws": 2}
for r in range(ROUNDS):
    for k, name in enumerate(SEQ):
        us = [seg2[c * per_call + r * len(SEQ) + k]["dur"] for c in range(CALLS)]
        n = [rows[c][r][ids[name]] for c in range(CALLS)]
        nspr = 1e3 * sum(us) / sum(n) if sum(n) else float("nan")
        print("  seg_kernel<2>    %d      %-5s  %8d  %10.1f  %12.0f  %7.3f" % (r, name, CALLS, np.mean(us), np.mean(n), nspr))

# the batched S2I configuration with layer 0 on seg_kernel<1> (NNSP_B200_TC5=0: not the tcgen05 kernel)
os.environ["NNSP_B200_TC5"] = "0"
m = nb.Model.from_blob(os.path.join(nb.MODEL_DIR, "s2i.nnspm"))
b = nb.NNSPBatch(m, S2I_STREAMS)
base = nb.synth_pcm(pool, T, first_stream=17)
pcm = np.tile(base, ((S2I_STREAMS + pool - 1) // pool, 1))[:S2I_STREAMS]
dp = nb.DeviceArray.from_host(pcm)
rb = nb.DeviceArray((S2I_STREAMS, T), nb.RESULT_DT)
for i in range(5):
    b.exec_device(dp, T * 160, T, rb)
b.sync()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for i in range(CALLS):
        b.exec_device(dp, T * 160, T, rb)
        b.sync()
seg1 = kernels(prof, "seg_kernel<1>")
n1 = S2I_STREAMS * (T // 2)
us = np.mean([e["dur"] for e in seg1])
print("  seg_kernel<1>    -      s2i    %8d  %10.1f  %12d  %7.3f   (batched S2I x %d)" % (len(seg1), us, n1, 1e3 * us / n1, S2I_STREAMS))
b.close()
