"""Per-stream resets of a live cascade handle (nnsp_b200_cascade_reset_streams, nnsp_b200_group_reset_streams): the listed
streams start the next call from nnCntrlClass_reset of their controller (INSTANCE) or from the state a new handle starts
from (FRESH); no other stream notices.

The oracle of stream s is Oracle.cascade_run over its own audio, cut at its reset points: reset=2 (nnCntrlClass_reset of
the live controller) or a new state (init + reset). Resets before the same audio position compose to FRESH if any of them
is FRESH.

  every frame      : 6 pipelined device calls of 37 streams whose stages change every ~10 frames, a different subset reset
                     in each mode before each call (mid-S2I with a time-out counter running, mid-KWS in ragged calls,
                     look-back history full, some streams in consecutive calls), then resets before a tapped 2-frame call that reads the
                     state they left; default path with 1 and 4 rounds, sequential path, tcgen05 first round, ragged calls
                     (reset streams with count 0 stay reset), the shipped trio and a wide one, both accumulator modes;
  equivalences     : every stream INSTANCE is nnsp_b200_cascade_reset; FRESH is a new handle; unlisted streams are a handle
                     that never saw a reset -- byte for byte;
  no cost unused   : calls without pending resets make the launches and bytes of a handle that never saw the function;
  host calls       : 4100 streams, 8 slices, PCM16 and AUDADC words, a reset between two asynchronous tickets;
  group            : a cascade group with the device named twice, resets across the member boundary; a batch group refuses;
  arguments        : refused lists record nothing; duplicates with mixed modes give FRESH; a pending reset followed by
                     nnsp_b200_cascade_reset; per-stream parameters survive both modes."""
import ctypes as C

import numpy as np
import pytest

import test_gpu_cascade_ragged as R

S2I, VAD, KWS = 0, 1, 2
S, MAXF, NCALLS = R.S, R.MAXF, R.NCALLS
INSTANCE, FRESH = 0, 1                 # NNSP_B200_RESET_INSTANCE, NNSP_B200_RESET_FRESH
ERR_ARG = -1                           # NNSP_B200_ERR_ARG
FRAMES = NCALLS * MAXF + 2


@pytest.fixture(autouse=True)
def _library_defaults(monkeypatch):
    for e in R.SWITCHES:
        monkeypatch.delenv(e, raising=False)


def reset_plan():
    """{call k: [(stream, mode), ...]} for the calls 1 .. NCALLS (NCALLS: the tapped probe): different subsets in both
    modes, stream 3 INSTANCE and stream 8 FRESH before every call, stream 11 listed in both modes before call 2"""
    plan = {}
    for k in range(1, NCALLS + 1):
        lst = [(s, INSTANCE) for s in range(S) if (7 * s + 3 * k) % 6 == 0]
        lst += [(s, FRESH) for s in range(S) if (5 * s + k) % 7 == 0]
        lst += [(3, INSTANCE), (8, FRESH)]
        if k == 2:
            lst += [(11, INSTANCE), (11, FRESH), (11, INSTANCE)]
        plan[k] = lst
    return plan


def ragged_schedule(nb, oracle, name, acc32):
    """R.schedule(), but streams 3 and 8 end call 0 on their first KWS frame: the reset before call 1 falls mid-KWS"""
    counts = R.schedule().copy()
    _, want, _, _ = R.oracle_run(nb, oracle, name, acc32)
    for s in (3, 8):
        f = np.nonzero(want["stage_id"][s, :MAXF] == KWS)[0]
        assert len(f), s
        counts[0][s] = f[0] + 1
    return counts


def apply(handle, lst):
    for mode in (INSTANCE, FRESH):
        ids = [s for s, m in lst if m == mode]
        if ids:
            handle.reset_streams(ids, fresh=mode == FRESH)


def cuts_of(plan, pos):
    """per stream: {audio position: composed mode}"""
    cuts = [dict() for _ in range(S)]
    for k, lst in plan.items():
        for s, m in lst:
            p = int(pos[k][s])
            cuts[s][p] = max(cuts[s].get(p, INSTANCE), m)
    return cuts


def oracle_cut(nb, oracle, om, par, pcm, cuts, frames):
    """records and taps of one stream's audio [0, frames), cut at `cuts` {position: mode}"""
    st = oracle.lib.nnsp_oracle_cascade_new()
    bounds = sorted(p for p in cuts if 0 < p < frames)
    recs, taps = [], {g: [] for g, _ in R.CASC_TAPS}
    start = 0
    for end in bounds + [frames]:
        if start == 0:
            mode = True
        else:
            mode = 2 if cuts[start] == INSTANCE else True
        r, tp, _ = oracle.cascade_run(om, pcm[start * 160:end * 160], params=par, state=st, reset=mode)
        recs.append(r)
        for g, o in R.CASC_TAPS:
            taps[g].append(getattr(tp, o))
        start = end
    oracle.lib.nnsp_oracle_cascade_free(st)
    return np.concatenate(recs), {g: np.concatenate(v) for g, v in taps.items()}


def oracle_models(nb, oracle, name, acc32):
    stacks = R.TRIOS[name][0]
    if stacks is None:
        return [oracle.model(i, acc32) for i in range(3)], False
    return [oracle.load_model(R.net_case_blob(R.STACKS[n], acc32), acc32) for n in stacks], True


def oracle_streams(nb, oracle, name, acc32, pcm, cuts, frames):
    om, own = oracle_models(nb, oracle, name, acc32)
    par = R._params(oracle, nb, R.TRIOS[name][2])
    want, wtap = [], {g: [] for g, _ in R.CASC_TAPS}
    for s in range(len(cuts)):
        r, tp = oracle_cut(nb, oracle, om, par, pcm[s], cuts[s], frames)
        want.append(r)
        for g in wtap:
            wtap[g].append(tp[g])
    if own:
        for m in om:
            oracle.lib.nnsp_b200_model_free(m)
    return np.stack(want), {g: np.stack(v) for g, v in wtap.items()}


# ---------------------------------------------------------------------------------------------------------------------
# every frame against the oracle
# ---------------------------------------------------------------------------------------------------------------------
ARMS = {
    "rounds1": {"NNSP_B200_CASCADE_ROUNDS": "1"},
    "rounds4": {"NNSP_B200_CASCADE_ROUNDS": "4"},
    "default": {},
    "sequential": {},
    "tc5_first_round": {"NNSP_B200_TC5": "2"},
    "ragged": {},
}
CASES = [("shipped", False, a) for a in ARMS] + [("shipped", True, "default"), ("shipped", True, "ragged"),
                                                 ("wide_rows81", False, "default"), ("wide_rows81", True, "default"),
                                                 ("wide_rows81", False, "sequential")]


def test_reset_plan_hits_every_kind_of_state(nb, oracle):
    """the cuts fall in KWS, in S2I with its time-out counter running, with the look-back history full, in consecutive
    calls, and on ragged streams that then idle or resume (oracle only)"""
    pos = R.positions(np.full((NCALLS, S), MAXF))
    plan = reset_plan()
    pcm = nb.synth_pcm(S, FRAMES, first_stream=R.FIRST)
    want, _ = oracle_streams(nb, oracle, "shipped", False, pcm, cuts_of(plan, pos), FRAMES)
    before = np.concatenate([want[[s for s, _ in plan[k]], pos[k][[s for s, _ in plan[k]]] - 1] for k in range(1, NCALLS)])
    # with these parameters KWS decides on its first inference, so its counter never runs; S2I's does. The uniform
    # calls never end in KWS; the ragged arm cuts streams 3 and 8 there
    assert ((before["stage_id"] == S2I) & (before["cnt_timeout"] > 0)).sum() >= 3
    for acc32 in (False, True):
        rpos = R.positions(ragged_schedule(nb, oracle, "shipped", acc32))
        _, want, _, _ = R.oracle_run(nb, oracle, "shipped", acc32)
        assert (want["stage_id"][[3, 8], rpos[1][[3, 8]] - 1] == KWS).all()
    assert pos[1].min() >= 82                                          # ring and log-mel history full at every cut
    consecutive = set.intersection(*[{s for s, _ in plan[k]} for k in plan])
    assert {3, 8} <= consecutive
    counts = ragged_schedule(nb, oracle, "shipped", False)
    assert any(counts[k][s] == 0 for k in range(1, NCALLS) for s, _ in plan[k]), "no reset stream idles"
    assert any(counts[k - 1][s] == 0 and counts[k][s] > 0 for k in range(2, NCALLS) for s, _ in plan[k - 1]), \
        "no reset stream resumes after idling"


@pytest.mark.gpu
@pytest.mark.parametrize("name,acc32,arm", CASES, ids=["%s-%s-%s" % (n, "acc32" if a else "acc64", m) for n, a, m in CASES])
def test_every_frame_against_the_oracle(nb, oracle, monkeypatch, name, acc32, arm):
    for k, v in ARMS[arm].items():
        monkeypatch.setenv(k, v)
    ragged = arm == "ragged"
    counts = ragged_schedule(nb, oracle, name, acc32) if ragged else np.full((NCALLS, S), MAXF)
    pos = R.positions(counts)
    pcm = nb.synth_pcm(S, FRAMES, first_stream=R.FIRST)
    plan = reset_plan()
    want, wtap = oracle_streams(nb, oracle, name, acc32, pcm, cuts_of(plan, pos), FRAMES)
    c = nb.Cascade(R.gpu_models(nb, name, acc32), S, params=R.TRIOS[name][2])
    if arm == "sequential":
        c.set_path("sequential")
    tc0 = nb.tc5_launches()
    junk = np.random.default_rng(31)
    bufs = [R.call_pcm(pcm, pos[k], counts[k], MAXF, junk) for k in range(NCALLS)]
    d = [(nb.DeviceArray.from_host(b), nb.DeviceArray.from_host(counts[k].astype(np.int32)),
          nb.DeviceArray((S, MAXF), nb.CASCADE_RESULT_DT)) for k, b in enumerate(bufs)]
    for k, (dp, dn, dr) in enumerate(d):                   # back to back: resets between pipelined calls
        if k:
            apply(c, plan[k])
        if ragged:
            c.exec_ragged_device(dp, MAXF * 160, MAXF, dn, dr)
        else:
            c.exec_device(dp, MAXF * 160, MAXF, dr)
    c.sync()
    parts = [dr.to_host() for _, _, dr in d]
    for x in d:
        for a in x:
            a.free()
    for k, got in enumerate(parts):
        R.check(got, None, want, wtap, pos[k], counts[k], "%s call %d" % (arm, k))
    # resets before a tapped call: every tap of its two frames reads the state they left
    end = pos[-1]
    apply(c, plan[NCALLS])
    probe = np.stack([pcm[s, end[s] * 160:(end[s] + 2) * 160] for s in range(S)])
    res, taps = c.exec(probe, taps=True)
    c.close()
    R.check(res, taps, want, wtap, end, np.full(S, 2), "%s tapped call after resets" % arm)
    if "NNSP_B200_TC5" in ARMS[arm]:
        assert nb.tc5_launches() > tc0


# ---------------------------------------------------------------------------------------------------------------------
# equivalences, byte for byte
# ---------------------------------------------------------------------------------------------------------------------
LISTED = [0, 5, 15, 16, 17, 30, 36]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["auto", "sequential"])
def test_equivalences(nb, path):
    models = R.gpu_models(nb, "shipped", False)
    params = R.TRIOS["shipped"][2]
    pcm = nb.synth_pcm(S, 3 * MAXF, first_stream=R.FIRST)
    calls = [pcm[:, k * MAXF * 160:(k + 1) * MAXF * 160] for k in range(3)]

    def handle():
        h = nb.Cascade(models, S, params=params)
        h.set_path(path)
        return h

    def run(before_last):
        h = handle()
        out = [h.exec(calls[0]), h.exec(calls[1])]
        before_last(h)
        out.append(h.exec(calls[2]))
        h.close()
        return out

    plain = run(lambda h: None)
    every = run(lambda h: h.reset_streams(np.arange(S), fresh=False))
    whole = run(lambda h: h.reset())
    assert [x.tobytes() for x in every] == [x.tobytes() for x in whole]
    assert every[2].tobytes() != plain[2].tobytes()
    fresh = run(lambda h: h.reset_streams(LISTED, fresh=True))
    new = handle()
    first = new.exec(calls[2])
    new.close()
    unlisted = [s for s in range(S) if s not in LISTED]
    assert fresh[2][LISTED].tobytes() == first[LISTED].tobytes()
    assert fresh[2][unlisted].tobytes() == plain[2][unlisted].tobytes()
    assert fresh[2][LISTED].tobytes() != plain[2][LISTED].tobytes()


# ---------------------------------------------------------------------------------------------------------------------
# no cost when unused
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", ["auto", "sequential"])
def test_no_cost_without_pending_resets(nb, path):
    models = R.gpu_models(nb, "shipped", False)
    pcm = nb.synth_pcm(S, 4 * MAXF, first_stream=R.FIRST)
    calls = [pcm[:, k * MAXF * 160:(k + 1) * MAXF * 160] for k in range(4)]
    runs = []
    for uses in (False, True):
        h = nb.Cascade(models, S, params=R.TRIOS["shipped"][2])
        h.set_path(path)
        out, deltas = [], []
        for x in calls:
            if uses:
                h.reset_streams([], fresh=True)           # n == 0: nothing pending
            l0 = nb.kernel_launches()
            out.append(h.exec(x))
            deltas.append(nb.kernel_launches() - l0)
        # one call with pending resets: one reset launch more, two on the pipelined path (front end and chain)
        if uses:
            h.reset_streams([1, 2])
        l0 = nb.kernel_launches()
        h.exec(calls[0])
        deltas.append(nb.kernel_launches() - l0)
        h.close()
        runs.append((out, deltas))
    (a, la), (b, lb) = runs
    assert [x.tobytes() for x in a] == [x.tobytes() for x in b]
    assert la[:-1] == lb[:-1], (la, lb)
    assert lb[-1] - la[-1] == (1 if path == "sequential" else 2), (la, lb)


# ---------------------------------------------------------------------------------------------------------------------
# asynchronous host calls
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["pcm16", "audadc"])
def test_host_async_reset_between_tickets(nb, oracle, fmt):
    n_streams, T = 4100, MAXF
    edges = [0, 15, 16, 511, 512, 1023, 1024, 2047, 2048, 3583, 3584, 4099]
    fresh_ids, inst_ids = edges[::2], edges[1::2] + [700, 3000]
    rng = np.random.default_rng(7)
    pcm = nb.synth_pcm(n_streams, 2 * T, first_stream=R.FIRST)
    if fmt == "audadc":
        raw = pcm.view(np.uint16).astype(np.uint32) | (rng.integers(0, 1 << 16, pcm.shape, dtype=np.uint32) << 16)
        pcm = nb.ingest_audadc(raw)
        host = raw
    else:
        host = pcm
    models = R.gpu_models(nb, "shipped", False)
    params = R.TRIOS["shipped"][2]
    ref = nb.Cascade(models, n_streams, params=params)      # device calls, no reset, then with the same resets
    want1 = ref.exec(pcm[:, :T * 160])
    ref.reset_streams(fresh_ids, fresh=True)
    ref.reset_streams(inst_ids)
    want2 = ref.exec(pcm[:, T * 160:])
    ref.close()
    c = nb.Cascade(models, n_streams, params=params)
    if fmt == "audadc":
        c.set_host_format("audadc")
    pin = [nb.PinnedArray((n_streams, T * 160), host.dtype) for _ in range(2)]
    pres = [nb.PinnedArray((n_streams, T), nb.CASCADE_RESULT_DT) for _ in range(2)]
    pin[0].array[...] = host[:, :T * 160]
    pin[1].array[...] = host[:, T * 160:]
    t1 = c.exec_host_async(pin[0].array, pres[0].array) if fmt == "pcm16" else \
        c.exec_host_ragged_async(pin[0].array, np.full(n_streams, T), pres[0].array)
    c.reset_streams(fresh_ids, fresh=True)
    c.reset_streams(inst_ids)
    t2 = c.exec_host_async(pin[1].array, pres[1].array) if fmt == "pcm16" else \
        c.exec_host_ragged_async(pin[1].array, np.full(n_streams, T), pres[1].array)
    c.wait_host(t2)
    got = [p.array.copy() for p in pres]
    for x in pin + pres:
        x.free()
    c.close()
    assert t1 < t2
    assert got[0].tobytes() == want1.tobytes()
    assert got[1].tobytes() == want2.tobytes()
    # and the oracle, for the reset streams and some that were not
    om = [oracle.model(i, False) for i in range(3)]
    par = R._params(oracle, nb, params)
    sample = sorted(set(edges + [1, 17, 700, 3000, 3001]))
    want = []
    for s in sample:
        mode = FRESH if s in fresh_ids else (INSTANCE if s in inst_ids else None)
        want.append(oracle_cut(nb, oracle, om, par, pcm[s], {} if mode is None else {T: mode}, 2 * T)[0])
    want = np.stack(want)
    n = len(sample)
    R.check(got[0][sample], None, want, None, np.zeros(n, int), np.full(n, T), "%s ticket 1" % fmt)
    R.check(got[1][sample], None, want, None, np.full(n, T), np.full(n, T), "%s ticket 2" % fmt)


# ---------------------------------------------------------------------------------------------------------------------
# group
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_group_resets_across_members(nb, oracle):
    name = "shipped"
    g = nb.Group(R.gpu_models(nb, name, False), S, [0, 0], params=R.TRIOS[name][2])
    edge = g.ranges()[1][1]
    assert 0 < edge < S
    plan = {k: [(edge - 2, INSTANCE), (edge - 1, FRESH), (edge, FRESH), (edge + 1, INSTANCE), (3 * k, INSTANCE),
                (S - 1 - 2 * k, FRESH)] for k in range(1, NCALLS + 1)}
    counts = np.full((NCALLS + 1, S), MAXF)
    pos = R.positions(counts)
    pcm = nb.synth_pcm(S, (NCALLS + 1) * MAXF, first_stream=R.FIRST)
    want, wtap = oracle_streams(nb, oracle, name, False, pcm, cuts_of(plan, pos), (NCALLS + 1) * MAXF)
    bufs = [np.ascontiguousarray(pcm[:, k * MAXF * 160:(k + 1) * MAXF * 160]) for k in range(NCALLS + 1)]
    res = [np.empty((S, MAXF), nb.CASCADE_RESULT_DT) for _ in bufs]
    tickets = []
    for k, b in enumerate(bufs):                           # asynchronous, resets queued between the calls
        if k:
            apply(g, plan[k])
        tickets.append(g.exec_host_async(b, res[k]))
    g.wait(tickets[-1])
    # a reset with no call behind it is complete once recorded: what waits for the group's commands returns
    g.reset_streams([edge])
    g.set_stream_params(0, R._params(oracle, nb, R.TRIOS[name][2])[None])
    g.close()
    for k in range(NCALLS + 1):
        R.check(res[k], None, want, wtap, pos[k], counts[k], "group call %d" % k)


@pytest.mark.gpu
def test_batch_group_refuses(nb):
    m = nb.Model.from_blob(nb.MODEL_DIR + "/vad.nnspm")
    g = nb.Group(m, 64, [0, 0])
    with pytest.raises(nb.NnspError):
        g.reset_streams([1, 2])
    g.close()


# ---------------------------------------------------------------------------------------------------------------------
# arguments and composition
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_arguments_and_composition(nb):
    from nnsp_b200 import capi
    L = capi.lib()
    models = R.gpu_models(nb, "shipped", False)
    params = R.TRIOS["shipped"][2]
    pcm = nb.synth_pcm(S, 2 * MAXF, first_stream=R.FIRST)
    x0, x1 = pcm[:, :MAXF * 160], pcm[:, MAXF * 160:]
    ps = [4, 9, 20]                                        # streams with parameters of their own

    def handle():
        h = nb.Cascade(models, S, params=params)
        p = np.tile(h.params_array(), (len(ps), 1))
        p[:, [n for n, _ in capi.CascadeParams._fields_].index("thresh_timeout_kws")] = [17, 23, 29]
        for i, s in enumerate(ps):
            h.set_stream_params(s, p[i:i + 1])
        return h

    def two_calls(between):
        h = handle()
        h.exec(x0)
        between(h)
        out = h.exec(x1)
        h.close()
        return out

    plain = two_calls(lambda h: None)

    def refused(h):                                        # NNSP_B200_ERR_ARG, and nothing recorded
        for ids, mode in (([0, S], 0), ([-1, 1], 1), ([1, 2], 2), ([1], -1)):
            a = np.asarray(ids, np.int32)
            assert L.nnsp_b200_cascade_reset_streams(h.h, a.ctypes.data_as(C.c_void_p), len(a), mode) == ERR_ARG, (ids, mode)
        assert L.nnsp_b200_cascade_reset_streams(h.h, None, -1, 0) == ERR_ARG
        assert L.nnsp_b200_cascade_reset_streams(h.h, None, 0, 0) == 0

    assert two_calls(refused).tobytes() == plain.tobytes()
    fresh = two_calls(lambda h: h.reset_streams([5, 9, 30], fresh=True))
    for order in ((False, True), (True, False)):
        def mixed(h, order=order):
            h.reset_streams([5, 9, 30], fresh=order[0])
            h.reset_streams([30, 9, 5, 9], fresh=order[1])
        assert two_calls(mixed).tobytes() == fresh.tobytes(), order
    # fresh: the records of a new handle with the same per-stream parameters; instance: those of a whole-handle reset
    new = handle()
    first = new.exec(x1)
    new.close()
    assert fresh[[5, 9, 30]].tobytes() == first[[5, 9, 30]].tobytes()
    whole = two_calls(lambda h: h.reset())
    inst = two_calls(lambda h: h.reset_streams(ps + [5]))
    assert inst[ps + [5]].tobytes() == whole[ps + [5]].tobytes()
    # pending FRESH, then the whole-handle reset: fresh-listed streams fresh, the rest reset as by nnsp_b200_cascade_reset
    both = two_calls(lambda h: (h.reset_streams([5, 9, 30], fresh=True), h.reset()))
    others = [s for s in range(S) if s not in (5, 9, 30)]
    assert both[[5, 9, 30]].tobytes() == first[[5, 9, 30]].tobytes()
    assert both[others].tobytes() == whole[others].tobytes()
