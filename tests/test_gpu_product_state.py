"""The state the shipped network paths store, checked against the oracle at every frame of a call, not only through the
result records (a one-LSB error in a layer-0 row or an LSTM cell rarely flips an argmax or a threshold flag).

Cut probe: for each cut frame k a fresh handle runs frames [0, k) on the product path without taps, as calls of at most
100 frames (the bench shape and its call boundaries), then one tapped call over [k, k + 2) -- the sequential kernel for
the cascade, the tcgen05 or mma.sync layer 0 for the batch, as the library selects. Those two frames (one inference, one
non-inference frame) read what the untapped calls stored, and their taps are compared with the same frames of one oracle
run over the whole sequence. Every cut is run, so every inference slot of every call length is the last one stored at
some cut and is compared while a fault in it is still fresh:
  cascade (stage-sorted pass): per-row start frames, the fix rows of a fresh instance's first two frames, look-back rows
    from lmhist, the stale-row hand-over at a stage change, and the counters of the closed-form controller walk
    (counts, argmax_last, slides, the time-out counter); also with the first round on the tcgen05 kernel
    (NNSP_B200_TC5=2) and, for a subset of cuts, with the prefix issued back to back without a sync (pipelined front end,
    double-buffered log-mel rows);
  batch: what scan_kernel, post_kernel and ctx_kernel store at the end of every call length, through two 62-inference
    tcgen05 chunks and a remainder."""
import ctypes as C

import numpy as np
import pytest

from common import cascade_events, chunks

pytestmark = pytest.mark.gpu
MODEL_FILE = {0: "s2i.nnspm", 1: "vad.nnspm", 2: "kws_galaxy.nnspm"}
S2I, VAD, KWS = 0, 1, 2
CASC_TAPS = (("logmel", "logmel"), ("feat", "feat"), ("hstate", "h"), ("cstate", "c"), ("post", "post"))
BATCH_TAPS = CASC_TAPS + (("act", "act"), ("logits", "logits"))
PIPE_LENS = [50, 50, 3, 47, 100, 50, 1, 49, 50, 100]     # prefix calls of the pipelined arm (cycled, cut to length)

# (seq, params, acc32, per-stream parameters, frames, stages the workload reaches, events it must contain): the sets of
# test_cascade_stage_sorted_pass and one with per-stream ParamCntrlClass rows drawn as in
# test_per_stream_params_changed_at_run_time. A fresh VAD -> KWS -> S2I cascade first reaches S2I at frame 338 of this
# audio, so the default set runs 400 frames; the other sets keep S2I out of reach (KWS look-back 99 and the drawn rows) or
# run it behind VAD or alone within 260.
CASC_SETS = [
    ((VAD, KWS, S2I), None, False, False, 400, {VAD, KWS, S2I}, ("fix", "detection")),
    ((VAD, KWS, S2I), dict(frs_vbufBk_kws=99, frs_vbufBk_s2i=1, thresh_timeout_kws=45, thresh_timeout_s2i=30, thresh_prob_kws=100, thresh_cnts_kws=2),
     False, False, 260, {VAD, KWS}, ("fix", "detection", "timeout")),
    ((VAD, S2I), dict(frs_vbufBk_s2i=5, thresh_timeout_s2i=60, thresh_cnts_vad=2), True, False, 260, {VAD, S2I}, ("fix", "detection", "timeout")),
    ((S2I,), dict(frs_vbufBk_s2i=0, thresh_timeout_s2i=37, thresh_cnts_s2i=1), False, False, 260, {S2I}, ("detection", "timeout")),
    ((VAD, KWS, S2I), None, False, True, 260, {VAD, KWS}, ("fix", "detection", "timeout")),
]
CASC_IDS = ["default", "kws_lookback99", "vad_s2i_acc32", "s2i_only", "per_stream"]


def test_cascade_sets_cover_every_stage_and_event():
    assert set().union(*(c[5] for c in CASC_SETS)) == {VAD, KWS, S2I}
    assert all(any(e in c[6] for c in CASC_SETS) for e in ("fix", "detection", "timeout"))


def _first_diff(a, b):
    bad = (a != b).reshape(a.shape[0], a.shape[1], -1).any(axis=2)
    s, t = (int(x[0]) for x in np.nonzero(bad))
    return s, t


def _stream_params(nb, c):
    """per-stream rows drawn as in test_per_stream_params_changed_at_run_time"""
    rng = np.random.default_rng(11)
    base = c.params_array()
    names = [n for n, _ in nb.capi.CascadeParams._fields_]
    rows = []
    for _ in range(c.S):
        p = base.copy()
        for n, lo, hi in [("thresh_timeout_kws", 20, 120), ("thresh_timeout_s2i", 15, 90), ("thresh_cnts_vad", 1, 6), ("thresh_cnts_kws", 1, 5),
                          ("thresh_cnts_s2i", 1, 5), ("thresh_prob_vad", 2000, 30000), ("thresh_prob_kws", 100, 30000), ("thresh_prob_s2i", 100, 30000)]:
            p[names.index(n)] = rng.integers(lo, hi + 1)
        rows.append(p)
    return np.stack(rows)


@pytest.fixture(scope="module")
def cascade_models(nb):
    return {acc32: [nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[i], acc32=acc32) for i in range(3)] for acc32 in (False, True)}


@pytest.mark.parametrize("tc5", ["default", "tc5_first_round"])
@pytest.mark.parametrize("cset", CASC_SETS, ids=CASC_IDS)
def test_cascade_sorted_pass_state_at_every_cut(nb, oracle, cascade_models, monkeypatch, cset, tc5):
    seq, params, acc32, per_stream, T, live, events = cset
    if tc5 == "default":
        monkeypatch.delenv("NNSP_B200_TC5", raising=False)
    else:
        monkeypatch.setenv("NNSP_B200_TC5", "2")
    S = 75                                             # four full tiles and a partial one, spread over the groups
    pcm = nb.synth_pcm(S, 600, first_stream=17)[:, :(T + 1) * 160]      # (the audio depends on the length asked for)
    models = cascade_models[acc32]

    def make():
        c = nb.Cascade(models, S, seq=seq, params=params)
        if per_stream:
            c.set_stream_params(0, par)
        return c

    c = nb.Cascade(models, S, seq=seq, params=params)
    par = _stream_params(nb, c) if per_stream else c.params_array()
    c.close()
    om = [oracle.model(i, acc32) for i in range(3)]
    want, wtap, valid = [], {g: [] for g, _ in CASC_TAPS}, []
    for s in range(S):
        r, tp, v = oracle.cascade_run(om, pcm[s], seq=seq, params=par[s] if per_stream else par)
        want.append(r)
        valid.append(v)
        for g, o in CASC_TAPS:
            wtap[g].append(getattr(tp, o))
    want, valid = np.stack(want), np.stack(valid)
    wtap = {g: np.stack(v) for g, v in wtap.items()}

    # the workload means something: the stages are live, cuts fall right after instance changes (fix rows, stale-row
    # hand-over), after detections and after time-outs
    new, det, timeout = cascade_events(want, valid)
    cuts = np.arange(1, T)
    assert set(np.unique(want["stage_id"][:, :T]).tolist()) == live
    n_fix = int(sum((new[:, k - 1] | new[:, k]).any() for k in cuts))
    assert "fix" not in events or n_fix > 20, "only %d cuts fall on the first or second frame of a new instance" % n_fix
    assert "detection" not in events or det[:, cuts - 1].any(), "no cut follows a detection"
    assert "timeout" not in events or timeout[:, cuts - 1].any(), "no cut follows a time-out"

    def check(k, parts, res2, taps, how):
        got = np.concatenate(parts + [res2], axis=1)
        for f in ("stage_id", "pos_after", "detected", "outputs", "cnt_timeout"):
            if not (got[f] == want[f][:, :k + 2]).all():
                s, t = _first_diff(got[f], want[f][:, :k + 2])
                raise AssertionError("%s cut %d: stream %d frame %d field %s: gpu %s oracle %s (stage %d)" %
                                     (how, k, s, t, f, got[f][s, t], want[f][s, t], want["stage_id"][s, t]))
        for g, _ in CASC_TAPS:
            a, o = taps[g], wtap[g][:, k:k + 2]
            if not (a == o).all():
                s, t = _first_diff(a, o)
                raise AssertionError("%s cut %d: stream %d frame %d tap %s (stage %d valid %d, new instance at %s): gpu %s oracle %s" %
                                     (how, k, s, k + t, g, want["stage_id"][s, k + t], valid[s, k + t],
                                      np.nonzero(new[s, :k + 2])[0][-2:].tolist(), a[s, t][:6], o[s, t][:6]))

    for k in cuts:
        c = make()
        parts, t = [], 0
        for n in chunks(k):
            parts.append(c.exec(pcm[:, t * 160:(t + n) * 160]))
            t += n
        res2, taps = c.exec(pcm[:, k * 160:(k + 2) * 160], taps=True)
        c.close()
        check(k, parts, res2, taps, "sorted")

    # pipelined: the prefix issued back to back without a sync (overlapped front end, double-buffered log-mel rows)
    d_pcm = nb.DeviceArray.from_host(pcm)
    row = pcm.shape[1]
    for k in cuts[::7]:
        c = make()
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
        check(k, parts, res2, taps, "pipelined")
    d_pcm.free()


@pytest.mark.parametrize("arm", ["library_rule", "tc5_forced"])
@pytest.mark.parametrize("nn_id,acc32", [(0, False), (1, False), (2, True)])
def test_batch_state_at_every_cut(nb, oracle, monkeypatch, nn_id, acc32, arm):
    """cuts 1 .. 140: two 62-inference tcgen05 chunks and a remainder; under the library's rule prefix calls of >= 29
    inferences take the tcgen05 kernel and shorter ones seg_kernel<feat>"""
    if arm == "library_rule":
        monkeypatch.delenv("NNSP_B200_TC5", raising=False)
    else:
        monkeypatch.setenv("NNSP_B200_TC5", "2")
    S, K = 35, 140
    pcm = nb.synth_pcm(S, K + 2, first_stream=250 + nn_id)
    m = nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[nn_id], acc32=acc32)
    m_or = oracle.model(nn_id, acc32)
    want, wtap = [], {g: [] for g, _ in BATCH_TAPS}
    for s in range(S):
        r, tp = oracle.nnsp_run(m_or, pcm[s])
        want.append(r)
        for g, o in BATCH_TAPS:
            wtap[g].append(getattr(tp, o))
    want = np.stack(want)
    wtap = {g: np.stack(v) for g, v in wtap.items()}
    tc5_calls = 0
    for k in range(1, K + 1):
        b = nb.NNSPBatch(m, S)
        assert b.nn_path == "split"
        parts, t = [], 0
        n0 = nb.tc5_launches()
        for n in chunks(k):
            parts.append(b.exec(pcm[:, t * 160:(t + n) * 160]))
            t += n
        tc5_calls += nb.tc5_launches() - n0
        res2, taps = b.exec(pcm[:, k * 160:(k + 2) * 160], taps=True)
        b.close()
        got = np.concatenate(parts + [res2], axis=1)
        if not (got == want[:, :k + 2]).all():
            s, t = _first_diff(got.view(np.int16).reshape(S, k + 2, -1), want[:, :k + 2].view(np.int16).reshape(S, k + 2, -1))
            raise AssertionError("cut %d: results differ on stream %d frame %d" % (k, s, t))
        for g, _ in BATCH_TAPS:
            a, o = taps[g], wtap[g][:, k:k + 2]
            if not (a == o).all():
                s, t = _first_diff(a, o)
                raise AssertionError("cut %d: stream %d frame %d tap %s: gpu %s oracle %s" % (k, s, k + t, g, a[s, t][:6], o[s, t][:6]))
    # prefix calls with an inference: k = 1 .. 140 hold 140 of them plus one per cut past 100; the library's rule takes the
    # tcgen05 kernel for the calls of >= 29 inferences only
    with_inf = sum(len(chunks(k)) for k in range(1, K + 1))
    if arm == "tc5_forced":
        assert tc5_calls == with_inf
    else:
        assert 0 < tc5_calls < with_inf
