"""GPU parity of the tcgen05 layer-0 kernel (nnsp_b200/csrc/nnsp_tc5.cuh) of the batched scan-split path: first fc layer of
NeuralNetClass_exe (neural_nets.c:44-168, affine.c:409-490, activation.c:31-69) for all (stream, inference) rows of a call on
the 5th-generation tensor cores. A tapped call takes the same layer-0 kernel as an untapped one (tc5_tap_kernel reads its
outputs back), so every call below is tapped and every tap of every frame is checked against the oracle: the layer-0
activations at each inference slot of each 64-slot tile and 62-inference chunk, and what the LSTM, head and post-processing
make of them."""
import numpy as np
import pytest

from common import NET_CASES, NET_TC5_SATURATING, make_blob, net_case_blob

pytestmark = pytest.mark.gpu
TAPS = ["feat", "act", "logits", "hstate", "cstate", "post"]
ORACLE_TAP = dict(feat="feat", act="act", logits="logits", hstate="h", cstate="c", post="post")
MODEL_FILE = {0: "s2i.nnspm", 1: "vad.nnspm", 2: "kws_galaxy.nnspm"}
# call lengths: one-frame calls (both phases of the stride-2 gate), a call with a single inference, 100 frames (the bench
# shape), 129 and 257 frames (65 / 129 inferences: two and three 62-inference chunks per stream pair); then calls of
# 61, 62, 63, 124 and 125 inferences (one slot short of / exactly / one past the 62-inference chunk, twice that) in both
# phases of the gate (first = 0 and first = 1)
LENS = [1, 1, 2, 7, 100, 129, 3, 257, 64, 121, 122, 124, 127, 124, 125, 248, 251, 248, 249, 9]
EDGE_INF = [61, 62, 63, 124, 125]


def _schedule(lens):
    """(frame offset, frames, first, inferences) of each call of a fresh stream (nn_speech.c:84,125: frame t infers when t is even)"""
    out, t = [], 0
    for n in lens:
        first = t & 1
        out.append((t, n, first, (n - first + 1) // 2))
        t += n
    return out


def test_call_lengths_reach_the_chunk_edges_in_both_phases():
    have = {(ni, first) for _, _, first, ni in _schedule(LENS)}
    assert all((ni, ph) in have for ni in EDGE_INF for ph in (0, 1)), sorted(have)


@pytest.fixture(autouse=True)
def _force_tc5(monkeypatch):
    """the library takes the kernel on its own only when the tiles are at least 45 % full (calls of >= 58 frames); the
    small shapes below are forced through it"""
    monkeypatch.setenv("NNSP_B200_TC5", "2")


def _compare(oracle, m_or, pcm, got, taps, t0, s_list, kw):
    """results and every tap of frames [t0, t0 + T) against one oracle run per stream from frame 0"""
    T = got.shape[1]
    for s in s_list:
        r, tp = oracle.nnsp_run(m_or, pcm[s], **kw)
        r = r[t0:t0 + T]
        if not (r == got[s]).all():
            raise AssertionError("results differ on stream %d: first frame %d" % (s, t0 + int(np.nonzero(r != got[s])[0][0])))
        for name in TAPS:
            a, o = taps[name][s], getattr(tp, ORACLE_TAP[name])[t0:t0 + T]
            assert a.shape == o.shape, (name, a.shape, o.shape)
            if not (a == o).all():
                t = int(np.nonzero((a != o).reshape(T, -1).any(axis=1))[0][0])
                u = int(np.nonzero(a[t] != o[t])[0][0])
                raise AssertionError("tap %s differs on stream %d frame %d (inference %d of its call) unit %d: gpu %d oracle %d" %
                                     (name, s, t0 + t, t // 2, u, a[t][u], o[t][u]))


def _run(nb, oracle, m, m_or, S, first_stream, h_stride=None):
    sched = _schedule(LENS)
    T = sum(LENS)
    pcm = nb.synth_pcm(S, T, first_stream=first_stream)
    b = nb.NNSPBatch(m, S)
    assert b.nn_path == "split"
    parts, tap_parts = [], []
    before = nb.tc5_launches()
    for t, n, first, ni in sched:
        r, tp = b.exec(pcm[:, t * 160:(t + n) * 160], taps=True)
        parts.append(r)
        tap_parts.append(tp)
    ran = nb.tc5_launches() - before
    assert ran == sum(1 for _, _, _, ni in sched if ni > 0), "the tcgen05 kernel did not run for every tapped call with an inference"
    b.close()
    got = np.concatenate(parts, axis=1)
    taps = {k: np.concatenate([tp[k] for tp in tap_parts], axis=1) for k in TAPS}
    kw = {} if h_stride is None else dict(h_stride=h_stride)
    _compare(oracle, m_or, pcm, got, taps, 0, range(S), kw)
    return taps


@pytest.mark.parametrize("S", [1, 2, 3, 17, 35])
@pytest.mark.parametrize("nn_id,acc32", [(0, False), (1, False), (2, True), (0, True), (1, True), (2, False)])
def test_shipped_models_every_tap_matches_oracle(nb, oracle, nn_id, acc32, S):
    """scan variants <9,2,3> (S2I), <4,4,1> (VAD), <8,2,2> (KWS); odd stream pairs and partial 16-stream tiles"""
    m = nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[nn_id], acc32=acc32)
    _run(nb, oracle, m, oracle.model(nn_id, acc32), S, first_stream=10 * nn_id + S)


ELIGIBLE = [c for c in NET_CASES if c[0] in ("two_lstm", "odd_widths", "big_shifts")]     # tanh layer 0 with the exact 32-bit finish, LSTM behind it


@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
@pytest.mark.parametrize("case", ELIGIBLE, ids=[c[0] for c in ELIGIBLE])
def test_synthetic_widths_and_shifts(nb, oracle, case, acc32):
    """units 24 (padded to 32), 7 (padded to 16: 9 zero-weight units), 16 with a finish shift far from the shipped ones;
    both accumulator modes"""
    name, nn_id, sizes, types, acts, qk, qi, qb = case
    raw = make_blob(nn_id, sizes, types, list(acts), list(qk), list(qi), list(qb), seed=len(name))
    h_stride = sum(sizes[i + 1] for i, t in enumerate(types) if t == 1) or 1
    _run(nb, oracle, nb.Model.from_blob(raw, acc32=acc32), oracle.load_model(raw, acc32), 21, first_stream=400, h_stride=h_stride)


@pytest.mark.parametrize("acc32", [False, True])
@pytest.mark.parametrize("case", NET_TC5_SATURATING, ids=[c[0] for c in NET_TC5_SATURATING])
def test_saturated_feature_rows(nb, oracle, case, acc32):
    """full-scale operands: feature rows at -32768 / 32767 (hi byte -128 / 127, lo byte 0 / 255) against weights of -128,
    +127 or random bytes, the largest magnitudes the s8 x s8 and u8 x s8 chains can reach"""
    raw = net_case_blob(case, acc32)
    sizes, types = case[2], case[3]
    h_stride = sum(sizes[i + 1] for i, t in enumerate(types) if t == 1)
    before = nb.tc5_launches()
    taps = _run(nb, oracle, nb.Model.from_blob(raw, acc32=acc32), oracle.load_model(raw, acc32), 5, first_stream=600, h_stride=h_stride)
    assert nb.tc5_launches() > before                    # the stack is eligible
    f = taps["feat"]
    both = ((f == 32767).any(axis=2) & (f == -32768).any(axis=2)).mean()
    assert both > 0.5, "only %.2f of the feature rows hold both full-scale values" % both


def test_tapped_calls_of_bench_shape(nb, oracle, monkeypatch):
    """100-frame calls on 600 streams (2 pipeline slices), the kernel chosen by the library's own rule, every tap checked"""
    monkeypatch.delenv("NNSP_B200_TC5")
    S, n, calls = 600, 100, 3
    pcm = nb.synth_pcm(S, n * calls, first_stream=1900)
    m = nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[0])
    b = nb.NNSPBatch(m, S)
    before, parts, tap_parts = nb.tc5_launches(), [], []
    for k in range(calls):
        r, tp = b.exec(pcm[:, k * n * 160:(k + 1) * n * 160], taps=True)
        parts.append(r)
        tap_parts.append(tp)
    assert nb.tc5_launches() - before == calls
    b.close()
    got = np.concatenate(parts, axis=1)
    taps = {k: np.concatenate([tp[k] for tp in tap_parts], axis=1) for k in TAPS}
    _compare(oracle, oracle.model(0, False), pcm, got, taps, 0, range(S), {})


def test_ineligible_layers_keep_the_mma_sync_kernel(nb, oracle):
    """relu6 / sigmoid first layers and stacks without an LSTM behind layer 0 are not taken by the tcgen05 kernel"""
    for case in NET_CASES:
        name, nn_id, sizes, types, acts, qk, qi, qb = case
        if name not in ("fc_only", "lstm_wide", "lstm_last_fc_sigmoid"):
            continue
        raw = make_blob(nn_id, sizes, types, list(acts), list(qk), list(qi), list(qb), seed=3)
        m = nb.Model.from_blob(raw)
        b = nb.NNSPBatch(m, 9)
        before = nb.tc5_launches()
        pcm = nb.synth_pcm(9, 30, first_stream=5)
        got = b.exec(pcm)
        assert nb.tc5_launches() == before, name
        m_or = oracle.load_model(raw, False)
        h_stride = sum(sizes[i + 1] for i, t in enumerate(types) if t == 1) or 1
        for s in range(9):
            r, _ = oracle.nnsp_run(m_or, pcm[s], h_stride=h_stride, taps=False)
            assert (r == got[s]).all(), (name, s)
        b.close()


def test_short_calls_keep_the_mma_sync_kernel(nb, monkeypatch):
    """the selection rule: tiles of 2 streams x 64 inference slots must be at least 45 % in use"""
    monkeypatch.delenv("NNSP_B200_TC5")
    m = nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[1])
    b = nb.NNSPBatch(m, 8)
    for frames, want in [(2, 0), (16, 0), (40, 0), (64, 1), (100, 1), (130, 1), (300, 1)]:
        before = nb.tc5_launches()
        b.exec(nb.synth_pcm(8, frames, first_stream=1))
        assert nb.tc5_launches() - before == want, frames
    b.close()


def test_async_host_calls_of_bench_shape(nb, oracle, monkeypatch):
    """the end-to-end loop of bench.py at 100 frames per call: the kernel is chosen by the library's own rule and runs on
    the pipeline slices of asynchronous host-buffer calls (600 streams = 2 slices; slice starts are multiples of 16)"""
    monkeypatch.delenv("NNSP_B200_TC5")
    S, n, calls = 600, 100, 3
    pcm = nb.synth_pcm(S, n * calls, first_stream=900)
    m = nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[2], acc32=True)
    b = nb.NNSPBatch(m, S)
    pin = [nb.PinnedArray((S, n * 160), np.int16) for _ in range(2)]
    pres = [nb.PinnedArray((S, n), nb.RESULT_DT) for _ in range(2)]
    before, got, prev = nb.tc5_launches(), [], None
    for k in range(calls):
        pin[k & 1].array[...] = pcm[:, k * n * 160:(k + 1) * n * 160]
        tk = b.exec_host_async(pin[k & 1].array, pres[k & 1].array)
        if prev is not None:
            b.wait_host(prev)
            got.append(pres[(k - 1) & 1].array.copy())
        prev = tk
    b.wait_host(prev)
    got.append(pres[(calls - 1) & 1].array.copy())
    assert nb.tc5_launches() - before >= calls
    got = np.concatenate(got, axis=1)
    m_or = oracle.model(2, True)
    for s in list(range(0, S, 41)) + [S - 1]:
        r, _ = oracle.nnsp_run(m_or, pcm[s], taps=False)
        assert (r == got[s]).all(), s
    for x in pin + pres:
        x.free()
    b.close()


def test_cascade_first_round_on_the_tcgen05_kernel(nb, oracle):
    """NNSP_B200_TC5=2 (the fixture) also sends layer 0 of the cascade's first round through vseq_kernel + the tcgen05 kernel
    (device-side stream lists, per-stream first inference frames, context / look-back / fresh-instance rows): every field of
    the result records against the oracle, over calls long enough for the kernel to be chosen and with stage changes inside."""
    S, n, calls = 48, 150, 5
    pcm = nb.synth_pcm(S, n * calls, first_stream=0)
    models = [nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[i]) for i in range(3)]
    c = nb.Cascade(models, S, params=dict(thresh_timeout_s2i=45))
    before = nb.tc5_launches()
    got = np.concatenate([c.exec(pcm[:, k * n * 160:(k + 1) * n * 160]) for k in range(calls)], axis=1)
    assert nb.tc5_launches() - before == 3 * calls          # one per model group of the first round
    par = c.params_array()
    c.close()
    om = [oracle.model(i) for i in range(3)]
    stages = np.zeros(3, np.int64)
    for s in range(S):
        r, _, _ = oracle.cascade_run(om, pcm[s], params=par, taps=False)
        for f in r.dtype.names:
            assert (got[s][f] == r[f]).all(), "stream %d field %s" % (s, f)
        stages += np.bincount(r["stage_id"], minlength=3)
    assert (stages > 0).all(), stages                        # all three models were live somewhere
