"""The kernels whose grid is capped at the SM count, past their first pass. Each walks the streams in a loop: a warp (the
IMMA kernel: a CTA of 16 streams, the replay kernel: a two-warp group) takes stream si, then si + pass, then si + 2 pass,
in the same shared-memory scratch, so whatever one stream leaves there meets the next. At the bench's 8 192 streams per
GPU that loop runs on every call; here each kernel runs at least three passes, the last one partial, with the pass sizes
read from the device's SM count (pass_sizes restates each cap next to its launch line). The batch kernels take 1 to 4
CTAs per SM, by the model's shared memory, and do not say how many: their cases are sized for 4, and the layout and the
partial last pass hold for every count.

  layout     : 200 base streams of five kinds -- full-scale noise, quiet (digital silence, DC levels), square waves, pure
               tones, speech-like (synth_pcm) -- replicated in blocks of one grid's worth of warps so that stream si and
               si - k blocks (k = 1 .. 4), the stream its warp ran before it, are of different kinds, and every base sits
               in passes 0, 1 and 2;
  batch      : the dp2a (nn_kernel) and IMMA (nn_mma_kernel) time loops, the shipped models in both accumulator modes and
               a NET_LIMITS stack whose automatic path is that kernel, 2.5 passes of streams, calls of 33 and 31 frames (the
               stride-2 phase flips between them), every record and every tap;
  net_eval   : the same two kernels on adversarial (input, LSTM state) rows tiled to 2.5 passes;
  sequential : cascade_kernel<CsNarrow> (the shipped trio) and cascade_kernel<CsWide> (wide_rows81), 2.5 passes of streams,
               pipelined device calls of 100, 57 and 1 frames, a ragged call (counts 0 .. 40 by base: idle streams in every
               pass), a tapped call from each stream's own position; a stage change every ~10 frames (PARAMS);
  replay     : the default path with 1 and 3 stage-sorted rounds at 8 192 streams: cascade_replay_kernel hands out more
               than two streams per group, and the one-CTA kernels (cascade_regroup_kernel, cascade_sort_replay_kernel)
               take more than two streams per thread; the records equal a sequential-path run over the same audio.

Every stream is checked against the oracle run of its base, every frame, every record field and every tap the call took:
so every copy of a base is equal wherever it sits, and the copies in each pass equal the oracle. These tests pin the
per-stream reload of the warp scratch (context, h and c, the scalars, logits[] as the log-mel scratch row), the borrowed
front-end scratch slots of the narrow kernel, the ragged zero-fill and early exit of later streams, the replay group's
hand-out and the loop indices. Each fails, for example, when cascade_kernel reloads h / c only for a warp's first stream,
when nn_kernel keeps the scalars of the warp's previous stream, or when a replay group takes only one stream."""
import ctypes as C
from collections import Counter

import numpy as np
import pytest

from common import NET_LIMITS, adversarial_net_inputs, adversarial_states, net_case_blob, net_case_dims
from test_gpu_cascade_models import CASC_TAPS, FIELDS, STACKS, SWITCHES, TRIO, _params, gpu_models, launched, replay_queued

MODEL_FILE = {0: "s2i.nnspm", 1: "vad.nnspm", 2: "kws_galaxy.nnspm"}
KINDS = ("noise", "quiet", "square", "tone", "speech")
PER_KIND = 40
N_BASE = len(KINDS) * PER_KIND                 # base b is of kind b // PER_KIND
FIRST = 11
CHUNK = 2048                                   # streams per device-to-host copy of a tap
LIMITS = {c[0]: c for c in NET_LIMITS}
SORT_THREADS = 1024


def pass_sizes(sms):
    """streams each capped grid takes per pass on `sms` SMs"""
    return {
        # nnsp_cascade.cu:1394-1397, :1405 -- min(ceil(ns / 16), SMs) CTAs of CsNarrow::WARPS = 16 warps, a stream per warp
        "narrow": sms * 16,
        # nnsp_cascade.cu:1394-1397, :1406 -- the same with CsWide::WARPS = 8
        "wide": sms * 8,
        # nnsp_cascade.cu:1401-1403 -- min(ceil(ns / CR_GROUPS), SMs) CTAs of CR_GROUPS = 8 groups, a stream per group
        "replay": sms * 8,
        # nnsp_cascade.cu:1340, :1389 -- cascade_regroup_kernel, cascade_sort_replay_kernel: one CTA of CSORT_THREADS
        "one_cta": SORT_THREADS,
        # nnsp_engine.cu:771-774 (batch), :1193-1196 (net_eval) -- SMs * nn_ctas_per_sm CTAs of NN_WARPS = 16 warps;
        # nn_ctas_per_sm (1 .. 4) is not exposed: the cap of 4
        "dp2a": sms * 4 * 16,
        # nnsp_mma.cu:396-404 -- SMs * per_sm CTAs of 16 streams; per_sm (1 .. 4) is not exposed: the cap of 4
        "imma": sms * 4 * 16,
    }


def pass_options(kind, sms):
    """the pass sizes `kind` may run with: the batch kernels take 1 .. 4 CTAs per SM, the others exactly their cap"""
    P = pass_sizes(sms)[kind if kind != "replay" else "narrow"]
    return [P * k // 4 for k in (1, 2, 3, 4)] if kind in ("dp2a", "imma") else [P]


def stream_count(kind, sms):
    """(streams, pass size at the cap, layout block) of the case that runs `kind`; 8 streams past 2.5 passes leave the
    last pass partial for every CTA count, and the last IMMA tile half full"""
    opts = pass_options(kind, sms)
    if kind == "replay":
        return 8192, opts[-1], opts[0]         # the bench's share of a GPU; passes of the sequential reference run
    return 5 * opts[-1] // 2 + 8, opts[-1], opts[0]


def assert_passes(S, opts, what):
    """at least three passes, the last one partial, at every pass size the kernel may run with"""
    for P in opts:
        assert S > 2 * P and S % P, "%s: %d streams at %d per pass is not three passes with a partial last one" % (what, S, P)


def layout(S, u):
    """base stream of each of S streams, in blocks of u streams (a pass at one CTA per SM): stream si and si - k u
    (k = 1 .. 4: the stream its warp ran before it, at 1 .. 4 CTAs per SM) are of different kinds -- the kind steps by k
    modulo 5 -- and every block of at least N_BASE streams holds every base"""
    si = np.arange(S)
    q, j = si // u, si % u
    kind = (j + q) % len(KINDS)
    member = (j // len(KINDS) + 7 * q) % PER_KIND
    return kind * PER_KIND + member


def base_pcm(nb, frames):
    """[N_BASE, frames * 160]: PER_KIND streams of each of KINDS"""
    n = frames * 160
    t = np.arange(n)
    out = np.empty((N_BASE, n), np.int16)
    for m in range(PER_KIND):
        rng = np.random.default_rng([0x70A55, m])
        out[m] = rng.integers(-32768, 32768, n)
        out[PER_KIND + m] = 0 if m == 0 else (m * 61) % 4001 - 2000 + rng.integers(-3, 4, n)
        out[2 * PER_KIND + m] = np.where((t // (4 + m % 13)) % 2 == 0, 1, -1) * (12000 + 500 * m)
        out[3 * PER_KIND + m] = np.round((2000 + 700 * m) * np.sin(2 * np.pi * (150 + 97 * m) * t / 16000))
    syn = nb.synth_pcm(64, frames, first_stream=FIRST)
    out[4 * PER_KIND:] = syn[[r for r in range(64) if (FIRST + r) % 16 >= 4][:PER_KIND]]     # no synth edge-case rows
    return out


def sms_of_device():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rows(nb, d, s0, s1):
    """streams [s0, s1) of a host array or a DeviceArray [S, ...]"""
    if isinstance(d, np.ndarray):
        return d[s0:s1]
    out = np.empty((s1 - s0,) + d.shape[1:], d.dtype)
    rb = d.nbytes // d.shape[0]
    rc = nb.capi.lib().nnsp_b200_memcpy_d2h(d.device, out.ctypes.data_as(C.c_void_p), C.c_void_p(d.ptr.value + s0 * rb), out.nbytes)
    assert rc == 0, rc
    return out


def expect_streams(nb, d, idx, want, u, what):
    """every stream s of d [S, ...] (host or device) equals want[idx[s]], the oracle's rows of its base; u: layout block"""
    S, bad = len(idx), []
    for s0 in range(0, S, CHUNK):
        s1 = min(S, s0 + CHUNK)
        got = _rows(nb, d, s0, s1)
        bad += (s0 + np.nonzero((got != want[idx[s0:s1]]).reshape(s1 - s0, -1).any(axis=1))[0]).tolist()
    if bad:
        s = bad[0]
        got, w = _rows(nb, d, s, s + 1)[0], want[idx[s]]
        k = int(np.nonzero((got != w).reshape(-1))[0][0])
        pos = np.unravel_index(k, got.shape)
        raise AssertionError("%s: %d streams differ from the oracle, by block of %d %s; first: stream %d (base %d, %s) at %s: "
                             "gpu %s oracle %s" % (what, len(bad), u, dict(Counter(b // u for b in bad)), s, idx[s],
                                                   KINDS[idx[s] // PER_KIND], pos, got[pos], w[pos]))


@pytest.fixture(scope="module")
def sms():
    return sms_of_device()


@pytest.fixture(autouse=True)
def _library_defaults(monkeypatch):
    for e in SWITCHES:
        monkeypatch.delenv(e, raising=False)


# ---------------------------------------------------------------------------------------------------------------------
# layout (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_sms", [132, 148, 160])
def test_layout_puts_a_different_kind_before_every_stream(n_sms):
    """at every pass size each kernel may run with: three passes or more, the last one partial; stream si and its
    predecessor si - pass of different kinds; every base in passes 0, 1 and 2"""
    for kind in ("dp2a", "imma", "narrow", "wide", "replay"):
        S, _, u = stream_count(kind, n_sms)
        opts = pass_options(kind, n_sms)
        assert_passes(S, opts, kind)
        idx = layout(S, u)
        assert idx.min() >= 0 and idx.max() < N_BASE
        k = idx // PER_KIND
        for P in opts:
            assert (k[P:] != k[:-P]).all(), (kind, P)                 # hence a different base too
            for p in (0, 1, 2):
                assert set(idx[p * P:(p + 1) * P].tolist()) == set(range(N_BASE)), (kind, P, p)
        pairs = set(zip(k[u:].tolist(), k[:-u].tolist()))
        assert (KINDS.index("quiet"), KINDS.index("noise")) in pairs and (KINDS.index("noise"), KINDS.index("speech")) in pairs
    assert stream_count("replay", n_sms)[0] > 2 * SORT_THREADS


# ---------------------------------------------------------------------------------------------------------------------
# batch handle: dp2a and IMMA time loops
# ---------------------------------------------------------------------------------------------------------------------
BATCH_TAPS = (("feat", "feat"), ("act", "act"), ("logits", "logits"), ("hstate", "h"), ("cstate", "c"), ("post", "post"))
LENS = (33, 31)
BATCH = ([("shipped_%s_%s" % (MODEL_FILE[i].split(".")[0], "acc32" if a else "acc64"), i, a, path)
          for path in ("dp2a", "imma") for i in (0, 1, 2) for a in (False, True)] +
         [("lstm_off41", None, False, "dp2a"), ("ten_layers_last_lstm", None, False, "imma")])


def _net_model(nb, oracle, name, nn_id, acc32):
    """(gpu model, oracle model, oracle model to free or None, h_stride)"""
    if nn_id is not None:
        m_or = oracle.model(nn_id, acc32)
        return nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[nn_id], acc32=acc32), m_or, None, oracle.model_dims(m_or)[2][2]
    raw = net_case_blob(LIMITS[name], acc32)
    m_or = oracle.load_model(raw, acc32)
    return nb.Model.from_blob(raw, acc32=acc32), m_or, m_or, net_case_dims(LIMITS[name])[1]


@pytest.mark.gpu
@pytest.mark.parametrize("case", BATCH, ids=["%s-%s" % (c[3], c[0]) for c in BATCH])
def test_batch_kernel_past_three_passes(nb, oracle, sms, case):
    from nnsp_b200.api import _make_taps
    name, nn_id, acc32, path = case
    S, _, u = stream_count(path, sms)
    assert_passes(S, pass_options(path, sms), path)
    m, m_or, own, _ = _net_model(nb, oracle, name, nn_id, acc32)
    b = nb.NNSPBatch(m, S, nn_path=path if nn_id is not None else "auto")
    assert b.nn_path == path
    idx = layout(S, u)
    base = base_pcm(nb, sum(LENS))
    want = [oracle.nnsp_run(m_or, base[k], h_stride=max(b.h_stride, 1)) for k in range(N_BASE)]
    if own:
        oracle.lib.nnsp_b200_model_free(own)
    wrec = np.stack([r for r, _ in want])
    wtap = {g: np.stack([getattr(tp, o) for _, tp in want]) for g, o in BATCH_TAPS}
    t = 0
    for n in LENS:
        d_pcm = nb.DeviceArray.from_host(base[idx, t * 160:(t + n) * 160])
        d_res = nb.DeviceArray((S, n), nb.RESULT_DT)
        tp, arrs = _make_taps(S, n, b.act_stride, b.h_stride, b.n_out, 0)
        b.exec_device(d_pcm, n * 160, n, d_res, tp)
        b.sync()
        d_pcm.free()
        how = "%s %s frames %d..%d" % (path, name, t, t + n)
        expect_streams(nb, d_res.to_host(), idx, wrec[:, t:t + n], u, how + " records")
        for g, _ in BATCH_TAPS:
            expect_streams(nb, arrs[g], idx, wtap[g][:, t:t + n], u, how + " tap " + g)
        for a in [d_res] + list(arrs.values()):
            a.free()
        t += n
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", BATCH, ids=["%s-%s" % (c[3], c[0]) for c in BATCH])
def test_net_eval_past_three_passes(nb, oracle, sms, case):
    name, nn_id, acc32, path = case
    S, _, u = stream_count(path, sms)
    assert_passes(S, pass_options(path, sms), path)
    m, m_or, own, hs = _net_model(nb, oracle, name, nn_id, acc32)
    rng = np.random.default_rng(N_BASE + len(name))
    x = adversarial_net_inputs(rng)
    x = np.concatenate([x, rng.integers(-32768, 32768, (N_BASE - len(x), x.shape[1])).astype(np.int16)])
    h0, c0 = adversarial_states(rng, N_BASE, hs)
    want = [oracle.net_eval(m_or, x[k], h0[k], c0[k]) for k in range(N_BASE)]
    if own:
        oracle.lib.nnsp_b200_model_free(own)
    idx = layout(S, u)
    got = nb.net_eval(m, x[idx], h0[idx], c0[idx], nn_path=path)
    for i, what in enumerate(("act", "logits", "h1", "c1")):
        expect_streams(nb, got[i], idx, np.stack([w[i] for w in want]), u, "net_eval %s %s %s" % (path, name, what))


# ---------------------------------------------------------------------------------------------------------------------
# cascade: sequential kernel
# ---------------------------------------------------------------------------------------------------------------------
PIPE, TR, TT = (100, 57, 1), 40, 30            # pipelined calls, the ragged call, the tapped call
SEQ = [("narrow", "shipped", {}), ("wide", "wide_rows81", {"NNSP_B200_CASCADE_WIDE": "1"})]


def _oracle_models(nb, oracle, trio):
    if trio[1] is None:
        return [oracle.model(i, False) for i in range(3)], False
    return [oracle.load_model(net_case_blob(STACKS[n], False), False) for n in trio[1]], True


def _no_frame(nb, n):
    r = np.zeros(n, nb.CASCADE_RESULT_DT)
    r["stage_id"] = -1
    return r


def sequential_want(nb, oracle, trio, base, cnt):
    """per base: the records of the whole call sequence (the ragged call's frames past the count hold the "no frame"
    record), the taps of the tapped call, and the oracle records of the frames the base ran"""
    om, own = _oracle_models(nb, oracle, trio)
    par = _params(oracle, nb, trio[7])
    F0 = sum(PIPE)
    rec, taps, ran = [], {g: [] for g, _ in CASC_TAPS}, []
    for b in range(N_BASE):
        n = F0 + cnt[b] + TT
        r, tp, _ = oracle.cascade_run(om, base[b, :n * 160], params=par)
        rec.append(np.concatenate([r[:F0 + cnt[b]], _no_frame(nb, TR - cnt[b]), r[F0 + cnt[b]:]]))
        for g, o in CASC_TAPS:
            taps[g].append(getattr(tp, o)[F0 + cnt[b]:])
        ran.append(r)
    if own:
        for m in om:
            oracle.lib.nnsp_b200_model_free(m)
    return np.stack(rec), {g: np.stack(v) for g, v in taps.items()}, ran


@pytest.mark.gpu
@pytest.mark.parametrize("kind,trio_name,env", SEQ, ids=[s[0] for s in SEQ])
def test_sequential_kernel_past_three_passes(nb, oracle, monkeypatch, sms, kind, trio_name, env):
    from nnsp_b200.api import _make_taps
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    trio = TRIO[trio_name]
    S, P, _ = stream_count(kind, sms)
    assert_passes(S, [P], kind)
    idx = layout(S, P)
    F0 = sum(PIPE)
    base = base_pcm(nb, F0 + TR + TT)
    cnt = np.arange(N_BASE) % (TR + 1)                 # 0 .. TR; bases of count 0 sit in every pass
    wrec, wtap, ran = sequential_want(nb, oracle, trio, base, cnt)
    # the placement meets stage differences: at a call boundary, a stream whose predecessor in its warp sits in S2I with
    # a running time-out while it sits in VAD, and the other way round
    for t in np.cumsum(PIPE) - 1:
        st, to = wrec["stage_id"][idx, t], wrec["cnt_timeout"][idx, t]
        assert ((st[:-P] == 0) & (to[:-P] > 0) & (st[P:] == 1)).any(), t
        assert ((st[:-P] == 1) & (st[P:] == 0) & (to[P:] > 0)).any(), t
    assert len(set(np.concatenate([r["stage_id"] for r in ran]).tolist())) == 3

    c = nb.Cascade(gpu_models(nb, trio, False), S, params=trio[7])
    c.set_path("sequential")
    n0 = nb.cascade_kernel_launches()
    d_pcm = nb.DeviceArray.from_host(base[idx, :F0 * 160])
    outs, t = [], 0
    for n in PIPE:                                      # back to back, no sync
        outs.append(nb.DeviceArray((S, n), nb.CASCADE_RESULT_DT))
        c.exec_device(C.c_void_p(d_pcm.ptr.value + 2 * t * 160), F0 * 160, n, outs[-1])
        t += n
    rag = c.exec_ragged(base[idx, F0 * 160:(F0 + TR) * 160], cnt[idx])
    d_pcm.free()
    own = np.stack([base[b, (F0 + cnt[b]) * 160:(F0 + cnt[b] + TT) * 160] for b in range(N_BASE)])
    d_tp = nb.DeviceArray.from_host(own[idx])           # each stream from its own position
    d_res = nb.DeviceArray((S, TT), nb.CASCADE_RESULT_DT)
    tp, arrs = _make_taps(S, TT, 1, 128, 1, 0)
    c.exec_device(d_tp, TT * 160, TT, d_res, tp)
    c.sync()
    assert launched(nb, n0) == Counter({kind: len(PIPE) + 2})
    got = np.concatenate([o.to_host() for o in outs] + [rag, d_res.to_host()], axis=1)
    for a in outs + [d_tp, d_res]:
        a.free()
    c.close()
    expect_streams(nb, got, idx, wrec, P, "%s records" % kind)
    for g, _ in CASC_TAPS:
        expect_streams(nb, arrs[g], idx, wtap[g], P, "%s tap %s" % (kind, g))
    for a in arrs.values():
        a.free()


# ---------------------------------------------------------------------------------------------------------------------
# cascade: replay and one-CTA kernels behind the stage-sorted rounds
# ---------------------------------------------------------------------------------------------------------------------
REPLAY_LENS = (100, 100)


@pytest.mark.gpu
@pytest.mark.parametrize("rounds", [1, 3])
def test_replay_and_one_cta_kernels_past_three_passes(nb, oracle, monkeypatch, sms, rounds):
    monkeypatch.setenv("NNSP_B200_CASCADE_ROUNDS", str(rounds))
    trio = TRIO["shipped"]
    S, P, _ = stream_count("replay", sms)
    assert_passes(S, [P], "narrow")
    idx = layout(S, P)
    base = base_pcm(nb, sum(REPLAY_LENS))
    om = [oracle.model(i, False) for i in range(3)]
    par = _params(oracle, nb, trio[7])
    want, valid = [], []
    for b in range(N_BASE):
        r, _, v = oracle.cascade_run(om, base[b], params=par, taps=False)
        want.append(r)
        valid.append(v)
    want, valid = np.stack(want), np.stack(valid)
    # the replay list of some call holds more than two streams per group, and some one-CTA kernel (the regroup of round
    # r >= 1, or the sort of the replay list) more than two per thread
    queued = {r: replay_queued(valid[idx], REPLAY_LENS, r) for r in range(1, rounds + 1)}
    assert max(queued[rounds]) > 2 * pass_sizes(sms)["replay"], queued
    assert max(max(q) for q in queued.values()) > 2 * SORT_THREADS, queued

    models = gpu_models(nb, trio, False)
    c = nb.Cascade(models, S, params=trio[7])
    ref = nb.Cascade(models, S, params=trio[7])
    ref.set_path("sequential")
    parts, seq, ran, ran_seq, t = [], [], Counter(), Counter(), 0
    for n in REPLAY_LENS:
        pcm = base[idx, t * 160:(t + n) * 160]
        n0 = nb.cascade_kernel_launches()
        parts.append(c.exec(pcm))
        ran += launched(nb, n0)
        n0 = nb.cascade_kernel_launches()
        seq.append(ref.exec(pcm))
        ran_seq += launched(nb, n0)
        t += n
    c.close()
    ref.close()
    assert ran == Counter({"replay": len(REPLAY_LENS)}) and ran_seq == Counter({"narrow": len(REPLAY_LENS)})
    got, full = np.concatenate(parts, axis=1), np.concatenate(seq, axis=1)
    for f in FIELDS:
        bad = np.nonzero((got[f] != full[f]).reshape(S, -1).any(axis=1))[0]
        assert len(bad) == 0, "field %s: %d streams differ from the sequential path, first %d (base %d)" % (f, len(bad), bad[0], idx[bad[0]])
    expect_streams(nb, got, idx, want, P, "rounds %d records" % rounds)
