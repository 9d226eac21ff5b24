"""Ragged cascade calls: every stream advances by its own number of frames per call (nnsp_b200_cascade_exec_ragged,
nnsp_b200_cascade_exec_host_ragged_async), as if nnCntrlClass_exec ran n[s] times on instance s.

The oracle of stream s is Oracle.cascade_run over the concatenation of the frames s received across the calls. The GPU
records at (call c, frame t < n_c[s]) equal the oracle's records of those frames field for field; frames t >= n_c[s] hold
the "no frame" record (stage_id -1, every other field 0) and zero tap rows.

  every tap         : tapped ragged calls on the sequential kernel, the shipped trio and a wide trio, both accumulator
                      modes; counts 0 .. 3, odd and even, below and above the look-back (80) and the 82-frame PCM ring, 100;
  stage-sorted path : untapped ragged calls on the default configuration, 1, 2 and 4 rounds, the replay on the sequential
                      kernel, the tcgen05 first round, pipelined device calls and the sequential path; a tapped uniform
                      call then reads the state the ragged prefix left (the cut probe of test_gpu_product_state.py);
  idle streams      : runs of 0-count calls with a time-out counter running, then resumed;
  full counts       : every count = max_frames is the uniform call, byte for byte and launch for launch;
  unread PCM        : junk past each stream's count changes nothing;
  host calls        : 4100 streams (8 slices), asynchronous, two tickets in flight, PCM16 and AUDADC words; out-of-range
                      counts are refused before anything is queued.
nnsp_b200_cascade_kernel_launches says which per-stream network kernel ran in every call."""
from collections import Counter

import numpy as np
import pytest

from common import NET_CASCADE_EDGES, NET_CASES, cascade_events, net_case_blob

S2I, VAD, KWS = 0, 1, 2
MODEL_FILE = {S2I: "s2i.nnspm", VAD: "vad.nnspm", KWS: "kws_galaxy.nnspm"}
STACKS = {c[0]: c for c in NET_CASES + NET_CASCADE_EDGES}
# short time-outs, detections after one frame over a low threshold (a stage change every ~10 frames), the reference's
# 80-frame look-back for both KWS and S2I: the PCM ring holds 82 frames, the log-mel history 80 rows
PARAMS = dict(thresh_timeout_kws=40, thresh_timeout_s2i=30, frs_vbufBk_kws=80, frs_vbufBk_s2i=80, thresh_cnts_vad=1,
              thresh_prob_vad=100, thresh_prob_kws=100, thresh_cnts_kws=1)
# name, stacks in the S2I / VAD / KWS slots (None: the shipped models), narrow shape, parameters
TRIOS = {
    "shipped": (None, True, dict(PARAMS, thresh_cnts_kws=0)),   # the shipped KWS model needs a count threshold of 0 here
    "wide_rows81": (("s2i_wide_rows81", "lstm_last_fc_sigmoid", "odd_widths"), False, PARAMS),
}
S, MAXF, NCALLS, FIRST = 37, 100, 6, 5
FRAMES = NCALLS * MAXF + 2
FIELDS = ("stage_id", "pos_after", "detected", "outputs", "cnt_timeout")
CASC_TAPS = (("logmel", "logmel"), ("feat", "feat"), ("hstate", "h"), ("cstate", "c"), ("post", "post"))
SWITCHES = ("NNSP_B200_CASCADE_WIDE", "NNSP_B200_REPLAY_COOP", "NNSP_B200_CASCADE_ROUNDS", "NNSP_B200_TC5")
COUNTS = (0, 1, 2, 3, 4, 7, 8, 50, 51, 79, 80, 81, 82, 83, 99, 100)
IDLE = (4, 13, 22, 31)                 # idle for calls 1, 2 and 3, resumed in call 4
FULL = 36                              # always a full call


def schedule():
    """counts [NCALLS][S]: every value of COUNTS in every call, each stream through a spread of them"""
    n = np.array([[COUNTS[(7 * s + 3 * c) % len(COUNTS)] for s in range(S)] for c in range(NCALLS)])
    n[1:4, list(IDLE)] = 0
    n[0, list(IDLE)] = 89                # paused inside KWS / S2I with a time-out counter running
    n[:, FULL] = MAXF
    return n


def positions(counts):
    """frame of each stream's own audio at which each call starts: [NCALLS + 1][S]"""
    return np.concatenate([np.zeros((1, counts.shape[1]), int), np.cumsum(counts, axis=0)])


def no_frame_record():
    r = np.zeros((), np.dtype([("stage_id", "i1"), ("pos_after", "i1"), ("detected", "<i2"), ("outputs", "<i2", (3,)),
                               ("cnt_timeout", "<u2")]))
    r["stage_id"] = -1
    return r


def _params(oracle, nb, params):
    p = oracle.default_params()
    names = [n for n, _ in nb.capi.CascadeParams._fields_]
    for k, v in params.items():
        p[names.index(k)] = v
    return p


_RUNS = {}


def oracle_run(nb, oracle, name, acc32, n_streams=S, frames=FRAMES, streams=None, pcm=None):
    """(pcm, records, taps, valid) of the oracle over each stream's own audio"""
    key = (name, acc32, n_streams, frames, streams, None if pcm is None else id(pcm))
    if key not in _RUNS:
        stacks, _, params = TRIOS[name]
        if pcm is None:
            pcm = nb.synth_pcm(n_streams, frames, first_stream=FIRST)
        if stacks is None:
            om, own = [oracle.model(i, acc32) for i in range(3)], False
        else:
            om, own = [oracle.load_model(net_case_blob(STACKS[n], acc32), acc32) for n in stacks], True
        par = _params(oracle, nb, params)
        want, wtap, valid = [], {g: [] for g, _ in CASC_TAPS}, []
        for s in (range(n_streams) if streams is None else streams):
            r, tp, v = oracle.cascade_run(om, pcm[s], params=par)
            want.append(r)
            valid.append(v)
            for g, o in CASC_TAPS:
                wtap[g].append(getattr(tp, o))
        if own:
            for m in om:
                oracle.lib.nnsp_b200_model_free(m)
        _RUNS[key] = (pcm, np.stack(want), {g: np.stack(v) for g, v in wtap.items()}, np.stack(valid))
    return _RUNS[key]


def gpu_models(nb, name, acc32):
    stacks = TRIOS[name][0]
    if stacks is None:
        return [nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[i], acc32=acc32) for i in range(3)]
    return [nb.Model.from_blob(net_case_blob(STACKS[n], acc32), acc32=acc32) for n in stacks]


def call_pcm(pcm, pos, counts, maxf, junk):
    """the PCM of one ragged call: stream s's next counts[s] frames, junk behind them (None: zeros)"""
    n_streams = len(counts)
    buf = np.zeros((n_streams, maxf * 160), np.int16) if junk is None else \
        junk.integers(-32768, 32768, (n_streams, maxf * 160), dtype=np.int16)
    for s in range(n_streams):
        n = int(counts[s])
        buf[s, :n * 160] = pcm[s, pos[s] * 160:(pos[s] + n) * 160]
    return buf


def check(got, taps, want, wtap, pos, counts, how):
    """records got [S][T] (and taps, None: not taken) of one ragged call against the oracle's frames pos[s] .. pos[s] + n[s]"""
    T = got.shape[1]
    t = np.arange(T)[None, :]
    live = t < np.asarray(counts)[:, None]
    idx = np.minimum(np.asarray(pos)[:, None] + t, want.shape[1] - 1)
    for f in FIELDS:
        w = np.take_along_axis(want[f], idx.reshape(idx.shape + (1,) * (want[f].ndim - 2)), axis=1) if want[f].ndim > 2 \
            else np.take_along_axis(want[f], idx, axis=1)
        bad = (got[f] != w).reshape(len(got), T, -1).any(axis=2) & live
        if bad.any():
            s, tt = (int(x[0]) for x in np.nonzero(bad))
            raise AssertionError("%s: stream %d frame %d of %d (own frame %d) field %s: gpu %s oracle %s" %
                                 (how, s, tt, counts[s], pos[s] + tt, f, got[f][s, tt], w[s, tt]))
    nf = no_frame_record()
    tail = got.view(np.uint8).reshape(len(got), T, -1) != np.frombuffer(nf.tobytes(), np.uint8)
    bad = tail.any(axis=2) & ~live
    if bad.any():
        s, tt = (int(x[0]) for x in np.nonzero(bad))
        raise AssertionError("%s: stream %d frame %d >= %d is not the no-frame record: %s" % (how, s, tt, counts[s], got[s, tt]))
    for g, _ in CASC_TAPS if taps is not None else ():
        a, o = taps[g].reshape(len(got), T, -1), wtap[g].reshape(wtap[g].shape[0], wtap[g].shape[1], -1)
        w = np.take_along_axis(o, idx[:, :, None], axis=1)
        bad = np.where(live[:, :, None], a != w, a != 0).any(axis=2)
        if bad.any():
            s, tt = (int(x[0]) for x in np.nonzero(bad))
            raise AssertionError("%s: stream %d frame %d of %d tap %s: gpu %s oracle %s" %
                                 (how, s, tt, counts[s], g, a[s, tt][:6], w[s, tt][:6] if tt < counts[s] else 0))


def launched(nb, before):
    now = nb.cascade_kernel_launches()
    return Counter({k: now[k] - before[k] for k in now if now[k] != before[k]})


@pytest.fixture(autouse=True)
def _library_defaults(monkeypatch):
    for e in SWITCHES:
        monkeypatch.delenv(e, raising=False)


# ---------------------------------------------------------------------------------------------------------------------
# the workload (oracle only)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(TRIOS))
def test_schedule_cuts_at_events_and_idles_with_counters_running(nb, oracle, name):
    counts, pos = schedule(), positions(schedule())
    assert pos[-1].max() + 2 <= FRAMES and set(COUNTS) <= set(counts.ravel().tolist())
    for acc32 in (False, True):
        _, want, _, valid = oracle_run(nb, oracle, name, acc32)
        assert set(np.unique(want["stage_id"]).tolist()) == {S2I, VAD, KWS}
        new, det, timeout = cascade_events(want, valid)
        # the last frame of a call (t = n[s] - 1) and the first frame of the next one hold every kind of event
        for shift in (1, 0):
            sel = [(s, pos[c + 1][s] - shift) for c in range(NCALLS - 1) for s in range(S) if counts[c][s] > 0]
            ss, tt = np.array(sel).T
            for ev, what in ((new, "stage change"), (det, "detection"), (timeout, "time-out")):
                assert ev[ss, tt].any(), (acc32, what, shift)
        # some idle stream pauses inside KWS or S2I with its time-out counter running
        paused = pos[1][list(IDLE)]
        assert ((want["cnt_timeout"][list(IDLE), paused - 1] > 0) & (want["stage_id"][list(IDLE), paused - 1] != VAD)).any(), acc32


# ---------------------------------------------------------------------------------------------------------------------
# every tap: the sequential kernel
# ---------------------------------------------------------------------------------------------------------------------
TAP_CASES = [(n, a) for n in TRIOS for a in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,acc32", TAP_CASES, ids=["%s-%s" % (n, "acc32" if a else "acc64") for n, a in TAP_CASES])
def test_tapped_ragged_calls_every_tap(nb, oracle, name, acc32):
    pcm, want, wtap, valid = oracle_run(nb, oracle, name, acc32)
    counts, pos = schedule(), positions(schedule())
    c = nb.Cascade(gpu_models(nb, name, acc32), S, params=TRIOS[name][2])
    junk = np.random.default_rng(11)
    n0 = nb.cascade_kernel_launches()
    for k in range(NCALLS):
        res, taps = c.exec_ragged(call_pcm(pcm, pos[k], counts[k], MAXF, junk), counts[k], taps=True)
        check(res, taps, want, wtap, pos[k], counts[k], "tapped call %d" % k)
    ran = launched(nb, n0)
    c.close()
    assert ran == Counter({"narrow" if TRIOS[name][1] else "wide": NCALLS})


# ---------------------------------------------------------------------------------------------------------------------
# stage-sorted path: ragged prefix, then a tapped uniform call reads the state it left
# ---------------------------------------------------------------------------------------------------------------------
ARMS = {
    "default": {},
    "rounds1": {"NNSP_B200_CASCADE_ROUNDS": "1"},
    "rounds2": {"NNSP_B200_CASCADE_ROUNDS": "2"},
    "rounds4": {"NNSP_B200_CASCADE_ROUNDS": "4"},
    "replay_on_sequential": {"NNSP_B200_REPLAY_COOP": "0"},
    "tc5_first_round": {"NNSP_B200_TC5": "2"},
    "pipelined": {},
    "sequential": {},
}
PROBES = [("shipped", a) for a in ARMS] + [("wide_rows81", a) for a in ("default", "pipelined", "sequential")]


def replay_queued(valid, pos, counts, rounds):
    """streams the replay behind `rounds` stage-sorted rounds gets in one call: those that leave `rounds` instances before
    their own last frame of the call (valid == 0 marks the frames whose instance was reset)"""
    n = 0
    for s in range(len(counts)):
        if counts[s] > 1:
            n += int((valid[s, pos[s]:pos[s] + counts[s] - 1] == 0).sum() >= rounds)
    return n


@pytest.mark.gpu
@pytest.mark.parametrize("name,arm", PROBES, ids=["%s-%s" % p for p in PROBES])
def test_sorted_path_ragged_prefix_then_state(nb, oracle, monkeypatch, name, arm):
    env = ARMS[arm]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    narrow = TRIOS[name][1]
    seq_kind = "narrow" if narrow else "wide"
    if arm == "sequential":
        kind = seq_kind
    else:
        kind = "replay" if narrow and "NNSP_B200_REPLAY_COOP" not in env else seq_kind
    pcm, want, wtap, valid = oracle_run(nb, oracle, name, False)
    counts, pos = schedule(), positions(schedule())
    c = nb.Cascade(gpu_models(nb, name, False), S, params=TRIOS[name][2])
    if arm == "sequential":
        c.set_path("sequential")
    junk = np.random.default_rng(23)
    n0, tc0 = nb.cascade_kernel_launches(), nb.tc5_launches()
    bufs = [call_pcm(pcm, pos[k], counts[k], MAXF, junk) for k in range(NCALLS)]
    if arm == "pipelined":                  # back to back without a sync: overlapped front end, double-buffered rows
        d = [(nb.DeviceArray.from_host(b), nb.DeviceArray.from_host(counts[k].astype(np.int32)),
              nb.DeviceArray((S, MAXF), nb.CASCADE_RESULT_DT)) for k, b in enumerate(bufs)]
        for dp, dn, dr in d:
            c.exec_ragged_device(dp, MAXF * 160, MAXF, dn, dr)
        c.sync()
        parts = [dr.to_host() for _, _, dr in d]
        for x in d:
            for a in x:
                a.free()
    else:
        parts = [c.exec_ragged(b, counts[k]) for k, b in enumerate(bufs)]
    for k, got in enumerate(parts):
        check(got, None, want, wtap, pos[k], counts[k], "%s call %d" % (arm, k))
    # the state the prefix left, through every tap of a uniform 2-frame call
    end = pos[-1]
    probe = np.stack([pcm[s, end[s] * 160:(end[s] + 2) * 160] for s in range(S)])
    res, taps = c.exec(probe, taps=True)
    ran = launched(nb, n0)
    c.close()
    check(res, taps, want, wtap, end, np.full(S, 2), "%s after the prefix" % arm)
    assert ran == Counter({kind: NCALLS}) + Counter({seq_kind: 1})
    if arm != "sequential":
        rounds = int(env.get("NNSP_B200_CASCADE_ROUNDS", 3))
        assert max(replay_queued(valid, pos[k], counts[k], rounds) for k in range(NCALLS)) > 0, "no streams for the replay"
    if "NNSP_B200_TC5" in env:
        assert nb.tc5_launches() > tc0


# ---------------------------------------------------------------------------------------------------------------------
# every count = max_frames is the uniform call; the PCM past the counts is never read
# ---------------------------------------------------------------------------------------------------------------------
UNIFORM_LENS = (100, 37, 1, 62, 2)


def _run_uniform(nb, h, pcm, ragged, mode):
    """records (and taps) of the calls UNIFORM_LENS on handle h -- uniform calls, or ragged ones with every count full --
    and the launches they made: (all kernels, per-stream network kernels by kind)"""
    l0, k0 = nb.kernel_launches(), nb.cascade_kernel_launches()
    out, t = [], 0
    if mode == "pipelined":                 # issued back to back, one sync at the end
        bufs = []
        for n in UNIFORM_LENS:
            dp = nb.DeviceArray.from_host(pcm[:, t * 160:(t + n) * 160])
            dn = nb.DeviceArray.from_host(np.full(S, n, np.int32))
            dr = nb.DeviceArray((S, n), nb.CASCADE_RESULT_DT)
            if ragged:
                h.exec_ragged_device(dp, n * 160, n, dn, dr)
            else:
                h.exec_device(dp, n * 160, n, dr)
            bufs.append((dp, dn, dr))
            t += n
        h.sync()
        out = [(dr.to_host(), None) for _, _, dr in bufs]
        for x in bufs:
            for a in x:
                a.free()
    else:
        for n in UNIFORM_LENS:
            x = pcm[:, t * 160:(t + n) * 160]
            r = h.exec_ragged(x, np.full(S, n), taps=mode == "tapped") if ragged else h.exec(x, taps=mode == "tapped")
            out.append(r if mode == "tapped" else (r, None))
            t += n
    return out, nb.kernel_launches() - l0, launched(nb, k0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRIOS))
@pytest.mark.parametrize("mode", ["sorted", "tapped", "pipelined"])
def test_full_counts_are_the_uniform_call(nb, mode, name):
    models = gpu_models(nb, name, False)
    pcm = nb.synth_pcm(S, sum(UNIFORM_LENS), first_stream=FIRST)
    runs = []
    for ragged in (False, True):
        h = nb.Cascade(models, S, params=TRIOS[name][2])
        runs.append(_run_uniform(nb, h, pcm, ragged, mode))
        h.close()
    (ua, la, ka), (ub, lb, kb) = runs
    for k, ((ra, ta), (rb, tb)) in enumerate(zip(ua, ub)):
        assert ra.tobytes() == rb.tobytes(), (mode, k)
        for g in ta or ():
            assert ta[g].tobytes() == tb[g].tobytes(), (mode, k, g)
    assert la == lb and ka == kb, (la, lb, ka, kb)
    assert sum(ka.values()) == len(UNIFORM_LENS)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["auto", "sequential"])
def test_pcm_past_the_counts_is_not_read(nb, path):
    models = gpu_models(nb, "shipped", False)
    counts, pos = schedule(), positions(schedule())
    pcm = nb.synth_pcm(S, FRAMES, first_stream=FIRST)
    runs = []
    for seed in (None, 1, 2):
        junk = None if seed is None else np.random.default_rng(seed)
        c = nb.Cascade(models, S, params=TRIOS["shipped"][2])
        c.set_path(path)
        out = [c.exec_ragged(call_pcm(pcm, pos[k], counts[k], MAXF, junk), counts[k], taps=(path == "sequential"))
               for k in range(NCALLS)]
        c.close()
        runs.append(out)
    for other in runs[1:]:
        for x, y in zip(runs[0], other):
            if path == "sequential":
                assert x[0].tobytes() == y[0].tobytes()
                for g in x[1]:
                    assert x[1][g].tobytes() == y[1][g].tobytes(), g
            else:
                assert x.tobytes() == y.tobytes()


# ---------------------------------------------------------------------------------------------------------------------
# asynchronous host calls
# ---------------------------------------------------------------------------------------------------------------------
HOST_LENS = (37, 100, 2, 61, 40)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["pcm16", "audadc"])
def test_host_ragged_async(nb, oracle, fmt):
    """4100 streams (8 slices over the 3 pipeline streams), uneven calls of uneven counts, two tickets in flight, against
    ragged device calls over the same audio and, at the slice edges, the oracle; out-of-range counts queue nothing"""
    n_streams, name = 4100, "shipped"
    frames = sum(HOST_LENS) + 2
    sample = (0, 511, 512, 2047, 2048, 3583, 3584, 4099)
    rng = np.random.default_rng(5)
    pcm = nb.synth_pcm(n_streams, frames, first_stream=FIRST)
    if fmt == "audadc":                     # raw words: the PCM in the low half, junk above; conditioned on the device
        raw = pcm.view(np.uint16).astype(np.uint32) | (rng.integers(0, 1 << 16, pcm.shape, dtype=np.uint32) << 16)
        pcm = nb.ingest_audadc(raw)
    lens = np.array(HOST_LENS)
    counts = np.stack([rng.integers(0, n + 1, n_streams) for n in lens])
    counts[:, :16] = lens[:, None]                                     # a full tile
    counts[1:3, 16:40] = 0                                             # idle for two calls
    pos = positions(counts)
    _, want, _, _ = oracle_run(nb, oracle, name, False, n_streams, frames, sample, pcm=pcm)
    models = gpu_models(nb, name, False)
    ref = nb.Cascade(models, n_streams, params=TRIOS[name][2])
    c = nb.Cascade(models, n_streams, params=TRIOS[name][2])
    if fmt == "audadc":
        c.set_host_format("audadc")
    expect, pin, pres, tickets = [], [], [], []
    for k, n in enumerate(lens):
        buf = call_pcm(pcm, pos[k], counts[k], n, np.random.default_rng(100 + k))
        expect.append(ref.exec_ragged(buf, counts[k]))
        if fmt == "audadc":
            hb = np.random.default_rng(200 + k).integers(0, 1 << 32, (n_streams, n * 160), dtype=np.uint32)
            for s in range(n_streams):
                m = int(counts[k][s])
                hb[s, :m * 160] = raw[s, pos[k][s] * 160:(pos[k][s] + m) * 160]
        else:
            hb = buf
        pin.append(nb.PinnedArray(hb.shape, hb.dtype))
        pin[-1].array[...] = hb
        pres.append(nb.PinnedArray((n_streams, n), nb.CASCADE_RESULT_DT))
        if k == 2:                          # refused before anything is queued: the state stays where it is
            for bad in (n + 1, -1):
                wrong = counts[k].astype(np.int32)
                wrong[n_streams // 2] = bad
                with pytest.raises(nb.NnspError):
                    c.exec_host_ragged_async(pin[-1].array, wrong, pres[-1].array)
        tickets.append(c.exec_host_ragged_async(pin[-1].array, counts[k], pres[-1].array))
        if len(tickets) > 1:
            c.wait_host(tickets[-2])
    c.wait_host(tickets[-1])
    got = [p.array.copy() for p in pres]
    for x in pin + pres:
        x.free()
    ref.close(); c.close()
    for k in range(len(lens)):
        assert got[k].tobytes() == expect[k].tobytes(), (fmt, k)
        check(expect[k][list(sample)], None, want, None, pos[k][list(sample)], counts[k][list(sample)], "%s call %d" % (fmt, k))
