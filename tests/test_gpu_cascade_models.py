"""The cascade on model trios the shipped blobs never select: synthetic stacks in the S2I, VAD and KWS slots, on both sides
of the rule that picks the sequential kernel's shape (narrow: every layer at most 80 wide, LSTM state at most 80, at most
48 outputs; otherwise wide), against the oracle's cascade (nnsp_oracle_cascade_run, generic in the models; its network
code is pinned on these stacks by tests/golden/golden_nets_v1.npz) on every record and every tap.

  sequential kernel : every trio, both accumulator modes, one tapped call over every frame, in the shape the rule picks;
  stage-sorted pass : the cut probe of test_gpu_product_state.py -- a fresh handle runs frames [0, k) untapped in calls
                      of at most 100 frames, then a tapped 2-frame call reads what they stored -- with the round count 1 to
                      4, the replay on the sequential kernel (NNSP_B200_REPLAY_COOP=0), the tcgen05 first round
                      (NNSP_B200_TC5=2), pipelined prefixes, and the shipped models on the wide kernel;
  no scan-split form: the automatic path runs the sequential kernel, "sorted" is refused;
  sliced host calls : 4100 streams (8 slices) of a wide trio, asynchronous calls of uneven lengths.

nnsp_b200_cascade_kernel_launches says which of the three per-stream network kernels ran; the oracle's events say whether
the replay behind the rounds had streams to take (the kernel is launched in every call and returns at once without).

The narrow sequential kernel is the replay only when NNSP_B200_REPLAY_COOP=0 asks for it: both kernels stage the same
weight images behind their shared-memory structs and the replay kernel's is the smaller (a static_assert in
nnsp_cascade.cu), so no trio that fits the narrow kernel misses the replay kernel."""
import ctypes as C
from collections import Counter

import numpy as np
import pytest

from common import NET_CASCADE_EDGES, NET_CASES, NET_CRAFTED, NET_LIMITS, NET_TC5_SATURATING, cascade_events, chunks, net_case_blob, net_case_dims

S2I, VAD, KWS = 0, 1, 2
MODEL_FILE = {S2I: "s2i.nnspm", VAD: "vad.nnspm", KWS: "kws_galaxy.nnspm"}
STACKS = {c[0]: c for c in NET_CASES + NET_CRAFTED + NET_TC5_SATURATING + NET_CASCADE_EDGES + NET_LIMITS}
# short time-outs and look-backs, detections after one frame over a low threshold: a stage change every ~10 frames
PARAMS = dict(thresh_timeout_kws=40, thresh_timeout_s2i=30, frs_vbufBk_kws=20, frs_vbufBk_s2i=3, thresh_cnts_vad=1,
              thresh_prob_vad=100, thresh_prob_kws=100, thresh_cnts_kws=1)
S, T, FIRST = 37, 400, 5                       # two full 16-stream tiles and a partial one
CASC_TAPS = (("logmel", "logmel"), ("feat", "feat"), ("hstate", "h"), ("cstate", "c"), ("post", "post"))
FIELDS = ("stage_id", "pos_after", "detected", "outputs", "cnt_timeout")
PIPE_LENS = [50, 50, 3, 47, 100, 50, 1, 49, 50, 100]
SWITCHES = ("NNSP_B200_CASCADE_WIDE", "NNSP_B200_REPLAY_COOP", "NNSP_B200_CASCADE_ROUNDS", "NNSP_B200_TC5")

# name, stacks in the S2I / VAD / KWS slots (None: the shipped models), narrow shape, scan-split form, a layer 0 the
# tcgen05 kernel takes (tanh fc 240 -> <= 80, exact 32-bit finish, an LSTM behind it), accumulator modes, events the
# workload holds besides detections and fresh instances, parameters
EV = ("timeout",)
TRIOS = [
    ("narrow_edge", ("s2i_narrow_edge", "fc_only", "two_lstm"), True, True, True, (False, True), EV, PARAMS),
    ("wide_rows81", ("s2i_wide_rows81", "lstm_last_fc_sigmoid", "odd_widths"), False, True, True, (False, True), EV, PARAMS),
    ("wide_out49", ("s2i_wide_out49", "fc_only", "all_m128"), False, True, True, (False, True), EV, PARAMS),
    ("wide_h81", ("all_m128_q0", "sat_feat_random", "kws_wide_h81"), False, True, True, (False, True), (), PARAMS),   # S2I and KWS always fire in time
    ("wide_lstm100", ("lstm_wide", "sat_feat_random", "sat_feat_p127"), False, True, True, (False, True), EV, PARAMS),
    ("no_split_wide", ("lstm_requant", "fc_only", "two_lstm"), False, False, False, (False, True), EV, PARAMS),
    ("no_split_narrow", ("all_m128_q0", "bias_shift_18", "two_lstm"), True, False, False, (False,), (), PARAMS),   # acc32: VAD never fires
    # a second KWS LSTM at state offset 6 / 41 (not a multiple of 4): no scan-split form, the sequential kernel in each shape
    ("off6_narrow", ("s2i_narrow_edge", "fc_only", "lstm_off6"), True, False, False, (False, True), EV, PARAMS),
    ("off41_wide", ("lstm_wide", "ten_layers", "lstm_off41"), False, False, False, (False, True), EV, PARAMS),
    # the shipped KWS model stays under any probability threshold on this audio: a count threshold of 0 lets it through
    ("shipped", None, True, True, True, (False, True), EV, dict(PARAMS, thresh_cnts_kws=0)),
]
TRIO = {t[0]: t for t in TRIOS}
SYNTH = [t for t in TRIOS if t[1] is not None]


def narrow_limits_crossed(case):
    """the limits of the narrow shape (nnsp_b200_cascade_create) a stack crosses: a layer wider than 80 (rows, or inputs
    padded to 4 past layer 0), LSTM state beyond 80, more than 48 outputs"""
    sizes = case[2]
    _, h_stride, n_out = net_case_dims(case)
    out = []
    if max(sizes[1:]) > 80 or any(((n + 3) & ~3) > 80 for n in sizes[1:-1]):
        out.append("width")
    if h_stride > 80:
        out.append("h_stride")
    if n_out > 48:
        out.append("n_out")
    return out


def replay_queued(valid, lens, rounds, t0=0):
    """per call of `lens` (from frame t0 on): how many streams the replay behind `rounds` stage-sorted rounds gets. The
    controller walk cuts a stream at every instance it leaves and queues it for the next round while the call has frames
    left (exit frame + 1 < call length): a stream takes one round per instance exit, so it is left for the replay when it
    leaves `rounds` instances before the call's last frame. valid == 0 marks the frames whose instance was reset."""
    out, t = [], t0
    for n in lens:
        out.append(int(((valid[:, t:t + n - 1] == 0).sum(axis=1) >= rounds).sum()))
        t += n
    return out


def _params(oracle, nb, params):
    p = oracle.default_params()
    names = [n for n, _ in nb.capi.CascadeParams._fields_]
    for k, v in params.items():
        p[names.index(k)] = v
    return p


_RUNS = {}


def oracle_run(nb, oracle, trio, acc32, n_streams=S, frames=T, streams=None):
    """(pcm, records, taps, valid) of the oracle over `streams` (default all) of synth_pcm(n_streams, frames)"""
    key = (trio[0], acc32, n_streams, frames, streams)
    if key not in _RUNS:
        pcm = nb.synth_pcm(n_streams, frames, first_stream=FIRST)
        if trio[1] is None:
            om, own = [oracle.model(i, acc32) for i in range(3)], False
        else:
            om, own = [oracle.load_model(net_case_blob(STACKS[n], acc32), acc32) for n in trio[1]], True
        par = _params(oracle, nb, trio[7])
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


def gpu_models(nb, trio, acc32):
    if trio[1] is None:
        return [nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[i], acc32=acc32) for i in range(3)]
    return [nb.Model.from_blob(net_case_blob(STACKS[n], acc32), acc32=acc32) for n in trio[1]]


def launched(nb, before):
    now = nb.cascade_kernel_launches()
    return Counter({k: now[k] - before[k] for k in now if now[k] != before[k]})


def _first_diff(a, b):
    bad = (a != b).reshape(a.shape[0], a.shape[1], -1).any(axis=2)
    s, t = (int(x[0]) for x in np.nonzero(bad))
    return s, t


def check(got, taps, want, wtap, valid, t0, how):
    """records got [S][n] and taps (None: not taken) against the oracle's frames t0 .. t0 + n"""
    n = got.shape[1]
    for f in FIELDS:
        w = want[f][:, t0:t0 + n]
        if not (got[f] == w).all():
            s, t = _first_diff(got[f], w)
            raise AssertionError("%s: stream %d frame %d field %s: gpu %s oracle %s (stage %d)" %
                                 (how, s, t0 + t, f, got[f][s, t], w[s, t], want["stage_id"][s, t0 + t]))
    for g, _ in CASC_TAPS if taps is not None else ():
        a, o = taps[g], wtap[g][:, t0:t0 + n]
        if not (a == o).all():
            s, t = _first_diff(a, o)
            raise AssertionError("%s: stream %d frame %d tap %s (stage %d valid %d): gpu %s oracle %s" %
                                 (how, s, t0 + t, g, want["stage_id"][s, t0 + t], valid[s, t0 + t], a[s, t][:6], o[s, t][:6]))


@pytest.fixture(autouse=True)
def _library_defaults(monkeypatch):
    for e in SWITCHES:
        monkeypatch.delenv(e, raising=False)


# ---------------------------------------------------------------------------------------------------------------------
# the workload (oracle only)
# ---------------------------------------------------------------------------------------------------------------------
def test_edge_stacks_straddle_the_narrow_rule():
    e = {c[0]: c for c in NET_CASCADE_EDGES}
    assert narrow_limits_crossed(e["s2i_narrow_edge"]) == []
    assert net_case_dims(e["s2i_narrow_edge"])[1:] == (80, 48) and max(e["s2i_narrow_edge"][2][1:]) == 80
    assert narrow_limits_crossed(e["s2i_wide_rows81"]) == ["width"]
    assert narrow_limits_crossed(e["s2i_wide_out49"]) == ["n_out"]
    assert narrow_limits_crossed(e["kws_wide_h81"]) == ["h_stride"]
    for name, stacks, narrow, *_ in SYNTH:
        assert [STACKS[n][1] for n in stacks] == [S2I, VAD, KWS], name
        assert all(not narrow_limits_crossed(STACKS[n]) for n in stacks) == narrow, name
    wide = [t for t in SYNTH if not t[2]]
    crossed = set().union(*(narrow_limits_crossed(STACKS[n]) for t in wide for n in t[1]))
    assert crossed == {"width", "h_stride", "n_out"}
    for narrow in (True, False):               # time-outs on both shapes, with and without the stage-sorted pass
        assert any("timeout" in t[6] for t in SYNTH if t[2] == narrow and t[3])
    assert any("timeout" in t[6] for t in SYNTH if not t[3])


@pytest.mark.parametrize("trio", TRIOS, ids=[t[0] for t in TRIOS])
def test_trio_workload_reaches_every_stage_and_event(nb, oracle, trio):
    """all three stages live; cuts right after detections, time-outs and on the first two frames of a new instance; for
    every round count, prefix calls that leave streams to the replay"""
    for acc32 in trio[5]:
        _, want, _, valid = oracle_run(nb, oracle, trio, acc32)
        assert set(np.unique(want["stage_id"]).tolist()) == {S2I, VAD, KWS}, acc32
        new, det, timeout = cascade_events(want, valid)
        cuts = np.arange(1, T)
        assert sum((new[:, k - 1] | new[:, k]).any() for k in cuts) > 100
        assert det[:, cuts - 1].any()
        assert timeout[:, cuts - 1].any() == ("timeout" in trio[6])
        if trio[3]:
            for rounds in (1, 2, 3, 4):
                assert max(replay_queued(valid, chunks(T), rounds)) > 0, (acc32, rounds)


# ---------------------------------------------------------------------------------------------------------------------
# sequential kernel
# ---------------------------------------------------------------------------------------------------------------------
SEQ_CASES = [(t, a) for t in TRIOS for a in t[5]]


@pytest.mark.gpu
@pytest.mark.parametrize("trio,acc32", SEQ_CASES, ids=["%s-%s" % (t[0], "acc32" if a else "acc64") for t, a in SEQ_CASES])
def test_sequential_kernel_every_frame_every_tap(nb, oracle, trio, acc32):
    pcm, want, wtap, valid = oracle_run(nb, oracle, trio, acc32)
    c = nb.Cascade(gpu_models(nb, trio, acc32), S, params=trio[7])
    c.set_path("sequential")
    n0 = nb.cascade_kernel_launches()
    res, taps = c.exec(pcm, taps=True)
    ran = launched(nb, n0)
    c.close()
    assert ran == Counter({"narrow" if trio[2] else "wide": 1})
    check(res, taps, want, wtap, valid, 0, "sequential")


# ---------------------------------------------------------------------------------------------------------------------
# stage-sorted pass and replay: cut probe
# ---------------------------------------------------------------------------------------------------------------------
# arm: switches, accumulator mode, every cut (else every 7th, from an offset of its own), pipelined prefixes as well
ARMS = {
    "default": ({}, False, True, True),
    "default_acc32": ({}, True, False, False),
    "rounds1": ({"NNSP_B200_CASCADE_ROUNDS": "1"}, False, False, False),
    "rounds2": ({"NNSP_B200_CASCADE_ROUNDS": "2"}, False, False, False),
    "rounds4": ({"NNSP_B200_CASCADE_ROUNDS": "4"}, False, False, False),
    "replay_on_sequential": ({"NNSP_B200_REPLAY_COOP": "0"}, False, False, False),
    "tc5_first_round": ({"NNSP_B200_TC5": "2"}, False, False, True),
    "wide_kernel": ({"NNSP_B200_CASCADE_WIDE": "1"}, False, False, True),
}
EVERY_CUT = ("narrow_edge", "wide_rows81")
PROBES = ([(t[0], a) for t in SYNTH if t[3] for a in ARMS if a != "wide_kernel"] +
          [("shipped", "wide_kernel"), ("shipped", "replay_on_sequential")])


@pytest.mark.gpu
@pytest.mark.parametrize("trio_name,arm", PROBES, ids=["%s-%s" % p for p in PROBES])
def test_sorted_pass_state_at_cuts(nb, oracle, monkeypatch, trio_name, arm):
    trio = TRIO[trio_name]
    env, acc32, every, piped = ARMS[arm]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rounds = int(env.get("NNSP_B200_CASCADE_ROUNDS", 3))
    narrow = trio[2] and "NNSP_B200_CASCADE_WIDE" not in env
    seq_kind = "narrow" if narrow else "wide"
    replay_kind = "replay" if narrow and "NNSP_B200_REPLAY_COOP" not in env else seq_kind
    pcm, want, wtap, valid = oracle_run(nb, oracle, trio, acc32)
    models = gpu_models(nb, trio, acc32)
    cuts = np.arange(1, T - 1)                         # a 2-frame tapped call at every cut
    if not (every and trio_name in EVERY_CUT):
        cuts = cuts[list(ARMS).index(arm) % 7::7]

    n0, tc0, want_ran, queued = nb.cascade_kernel_launches(), nb.tc5_launches(), Counter(), []
    for k in cuts:
        c = nb.Cascade(models, S, params=trio[7])
        parts, t = [], 0
        for n in chunks(k):
            parts.append(c.exec(pcm[:, t * 160:(t + n) * 160]))
            t += n
        res2, taps = c.exec(pcm[:, k * 160:(k + 2) * 160], taps=True)
        c.close()
        check(np.concatenate(parts, axis=1), None, want, wtap, valid, 0, "%s cut %d" % (arm, k))
        check(res2, taps, want, wtap, valid, k, "%s cut %d" % (arm, k))
        want_ran[replay_kind] += len(parts)
        want_ran[seq_kind] += 1
        queued += replay_queued(valid, chunks(k), rounds)
    assert launched(nb, n0) == want_ran
    assert max(queued) > 0, "no prefix call left streams to the replay"
    if "NNSP_B200_TC5" in env:
        assert trio[4] and nb.tc5_launches() > tc0

    if not piped:
        return
    # pipelined: the prefix issued back to back without a sync (overlapped front end, double-buffered log-mel rows)
    d_pcm = nb.DeviceArray.from_host(pcm)
    row = pcm.shape[1]
    n0, want_ran, queued = nb.cascade_kernel_launches(), Counter(), []
    for k in np.arange(1, T - 1)[3::7]:
        c = nb.Cascade(models, S, params=trio[7])
        lens, t = chunks(k, PIPE_LENS), 0
        outs = [nb.DeviceArray((S, n), nb.CASCADE_RESULT_DT) for n in lens]
        for n, o in zip(lens, outs):
            c.exec_device(C.c_void_p(d_pcm.ptr.value + 2 * t * 160), row, n, o)
            t += n
        res2, taps = c.exec(pcm[:, k * 160:(k + 2) * 160], taps=True)
        parts = [o.to_host() for o in outs]
        for o in outs:
            o.free()
        c.close()
        check(np.concatenate(parts, axis=1), None, want, wtap, valid, 0, "pipelined %s cut %d" % (arm, k))
        check(res2, taps, want, wtap, valid, k, "pipelined %s cut %d" % (arm, k))
        want_ran[replay_kind] += len(lens)
        want_ran[seq_kind] += 1
        queued += replay_queued(valid, lens, rounds)
    d_pcm.free()
    assert launched(nb, n0) == want_ran
    assert max(queued) > 0


# ---------------------------------------------------------------------------------------------------------------------
# models without a scan-split form
# ---------------------------------------------------------------------------------------------------------------------
NO_SPLIT = [t for t in SYNTH if not t[3]]


@pytest.mark.gpu
@pytest.mark.parametrize("trio", NO_SPLIT, ids=[t[0] for t in NO_SPLIT])
def test_no_scan_split_form_takes_the_sequential_kernel(nb, oracle, trio):
    for acc32 in trio[5]:
        pcm, want, wtap, valid = oracle_run(nb, oracle, trio, acc32)
        c = nb.Cascade(gpu_models(nb, trio, acc32), S, params=trio[7])
        with pytest.raises(nb.NnspError):
            c.set_path("sorted")
        lens = chunks(T, (100, 37, 1, 62))
        n0, parts, t = nb.cascade_kernel_launches(), [], 0
        for n in lens:
            parts.append(c.exec(pcm[:, t * 160:(t + n) * 160]))
            t += n
        ran = launched(nb, n0)
        c.close()
        assert ran == Counter({"narrow" if trio[2] else "wide": len(lens)}), acc32
        check(np.concatenate(parts, axis=1), None, want, wtap, valid, 0, "auto, acc32=%d" % acc32)


# ---------------------------------------------------------------------------------------------------------------------
# sliced host calls
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sliced_async_host_calls_of_a_wide_trio(nb, oracle):
    """4100 streams: 8 slices over the 3 pipeline streams, stage-sorted pass and replay on the wide kernel per slice;
    asynchronous host calls of uneven lengths (the per-call scratch changes layout with every length) against one
    sequential call over the same audio, and streams at the slice edges against the oracle"""
    trio, n_streams, lens = TRIO["wide_rows81"], 4100, [37, 100, 2, 61, 40]
    frames = sum(lens)
    sample = (0, 511, 512, 2047, 2048, 3583, 3584, 4099)
    pcm, want, _, _ = oracle_run(nb, oracle, trio, False, n_streams, frames, sample)
    models = gpu_models(nb, trio, False)
    ref = nb.Cascade(models, n_streams, params=trio[7])
    ref.set_path("sequential")
    full = ref.exec(pcm)
    ref.close()
    for f in FIELDS:
        assert (full[list(sample)][f] == want[f]).all(), f
    c = nb.Cascade(models, n_streams, params=trio[7])
    c.set_path("sorted")
    pin, pres, tickets, t = [], [], [], 0
    n0 = nb.cascade_kernel_launches()
    for n in lens:
        pin.append(nb.PinnedArray((n_streams, n * 160), np.int16))
        pres.append(nb.PinnedArray((n_streams, n), nb.CASCADE_RESULT_DT))
        pin[-1].array[...] = pcm[:, t * 160:(t + n) * 160]
        tickets.append(c.exec_host_async(pin[-1].array, pres[-1].array))
        t += n
        if len(tickets) > 1:
            c.wait_host(tickets[-2])
    c.wait_host(tickets[-1])
    got = np.concatenate([p.array.copy() for p in pres], axis=1)
    ran = launched(nb, n0)
    for x in pin + pres:
        x.free()
    c.close()
    assert ran == Counter({"wide": 8 * len(lens)})
    for f in FIELDS:
        if not (got[f] == full[f]).all():
            s, tt = _first_diff(got[f], full[f])
            raise AssertionError("field %s stream %d frame %d: sorted %s sequential %s" % (f, s, tt, got[f][s, tt], full[f][s, tt]))
