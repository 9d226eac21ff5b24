"""GPU parity: the CUDA engine (through the C ABI) against the CPU oracle, bit for bit.

Reference behaviour being matched: NNSPClass_exec (ns-nnsp/src/nn_speech.c:74-127) called once
per frame per stream; every intermediate the reference exposes is compared (log-mel, normalised
feature row, every layer output, LSTM h/c, logits, trigger/outputs/counters).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TAPS = ["logmel", "feat", "act", "logits", "hstate", "cstate", "post"]
ORACLE_TAP = dict(logmel="logmel", feat="feat", act="act", logits="logits", hstate="h", cstate="c", post="post")
MODEL_FILE = {0: "s2i.nnspm", 1: "vad.nnspm", 2: "kws_galaxy.nnspm"}


def _model(nb, nn_id, acc32):
    return nb.Model.from_blob(nb.MODEL_DIR + "/" + MODEL_FILE[nn_id], acc32=acc32)


def _compare_stream(oracle, m_or, pcm_row, res_row, taps, s, th=(16383, 4)):
    r, tp = oracle.nnsp_run(m_or, pcm_row, thresh_prob=th[0], th_count=th[1])
    assert (r == res_row).all(), "results differ on stream %d: first frame %d" % (s, int(np.nonzero(r != res_row)[0][0]))
    for name in TAPS:
        a, b = taps[name][s], getattr(tp, ORACLE_TAP[name])
        assert a.shape == b.shape, (name, a.shape, b.shape)
        if not (a == b).all():
            t = int(np.nonzero((a != b).any(axis=1))[0][0])
            raise AssertionError("tap %s differs on stream %d frame %d: gpu %s oracle %s" % (name, s, t, a[t][:8], b[t][:8]))


def test_feature_stages_bit_exact(nb, oracle):
    """fft_in / spectrum / power spectrum / mel / log10 of the front end, incl. full-scale input (H5 bound)."""
    wins = np.concatenate([nb.adversarial_windows(), nb.synth_pcm(40, 3).reshape(40, 480)])
    out = nb.feature_stages(wins)
    for i, w in enumerate(wins):
        ref = oracle.feature_stages(w)
        for k in ("fft_in", "spec", "pspec", "mel", "logmel"):
            assert (out[k][i] == ref[k]).all(), "stage %s differs for window %d" % (k, i)


@pytest.mark.parametrize("path", ["split", "split_tc5", "imma", "dp2a"])
@pytest.mark.parametrize("nn_id,acc32", [(1, False), (2, True), (0, False), (0, True), (1, True), (2, False)])
def test_batch_matches_oracle_every_tap(nb, oracle, monkeypatch, nn_id, acc32, path):
    """All network paths: scan-split (default) with layer 0 on the mma.sync kernel seg_kernel<feat> (NNSP_B200_TC5=0) and
    on the tcgen05 kernel (=2), tensor-core IMMA in the time loop, dp2a warp per stream."""
    S, T = 53, 64                      # 53: a partial 16-stream tile at the end
    if path.startswith("split"):
        monkeypatch.setenv("NNSP_B200_TC5", "2" if path == "split_tc5" else "0")
    pcm = nb.synth_pcm(S, T)
    m = _model(nb, nn_id, acc32)
    b = nb.NNSPBatch(m, S, nn_path=path.split("_")[0])
    n0 = nb.tc5_launches()
    res, taps = b.exec(pcm, taps=True)
    assert nb.tc5_launches() - n0 == (1 if path == "split_tc5" else 0)       # which layer-0 kernel ran
    m_or = oracle.model(nn_id, acc32)
    for s in range(S):
        _compare_stream(oracle, m_or, pcm[s], res[s], taps, s)
    b.close()


def test_chunked_exec_equals_one_shot(nb, oracle):
    """State (window history, context, LSTM, counters, slides) must carry across exec calls, any chunking."""
    S, T = 20, 61
    pcm = nb.synth_pcm(S, T, first_stream=100)
    m = _model(nb, 0, False)
    b = nb.NNSPBatch(m, S)
    full, full_taps = b.exec(pcm, taps=True)
    b.close()
    b = nb.NNSPBatch(m, S)
    parts, feats, t = [], [], 0
    for n in (1, 1, 2, 3, 1, 7, 16, 30):
        r, tp = b.exec(pcm[:, t * 160:(t + n) * 160], taps=True)
        parts.append(r)
        feats.append(tp["cstate"])
        t += n
    assert t == T
    assert (np.concatenate(parts, axis=1) == full).all()
    assert (np.concatenate(feats, axis=1) == full_taps["cstate"]).all()
    m_or = oracle.model(0, False)
    for s in range(S):
        r, _ = oracle.nnsp_run(m_or, pcm[s], taps=False)
        assert (r == full[s]).all()
    b.close()


def test_reset_keeps_stale_context_row_like_the_reference(nb, oracle):
    """NNSPClass_reset refills context rows 0..4 only (feature_module.c:39-42): row 5 of the previous
    activation survives and is seen by the first inferences after the reset. Bit-exact means that too."""
    S, T = 24, 30
    pcm = nb.synth_pcm(S, 2 * T, first_stream=48)
    m = _model(nb, 1, False)
    b = nb.NNSPBatch(m, S)
    b.exec(pcm[:, :T * 160])
    b.reset()
    res, taps = b.exec(pcm[:, T * 160:], taps=True)
    m_or = oracle.model(1, False)
    st = oracle.lib.nnsp_oracle_stream_new()
    differs_from_fresh = 0
    for s in range(S):
        oracle.nnsp_run(m_or, pcm[s, :T * 160], state=st, reset=1, taps=False)
        r, tp = oracle.nnsp_run(m_or, pcm[s, T * 160:], state=st, reset=2)
        assert (r == res[s]).all()
        assert (tp.act == taps["act"][s]).all() and (tp.c == taps["cstate"][s]).all()
        _, tf = oracle.nnsp_run(m_or, pcm[s, T * 160:], reset=1)
        differs_from_fresh += int((tf.act != tp.act).any())
    oracle.lib.nnsp_oracle_stream_free(st)
    assert differs_from_fresh > 0      # the quirk is observable, so the test means something
    b.close()


def test_exec_host_equals_exec_device(nb):
    S, T = 300, 20
    pcm = nb.synth_pcm(S, T, first_stream=7)
    m = _model(nb, 1, False)
    b = nb.NNSPBatch(m, S)
    dev = b.exec(pcm)
    b.close()
    b = nb.NNSPBatch(m, S)
    n0 = nb.kernel_launches()
    host = b.exec_host(pcm)
    assert nb.kernel_launches() > n0
    assert (dev == host).all()
    host2 = b.exec_host(pcm)           # second call continues the streams: state carried on the device
    b2 = nb.NNSPBatch(m, S)
    both = b2.exec(np.concatenate([pcm, pcm], axis=1))
    assert (both[:, T:] == host2).all()
    b.close(); b2.close()


def test_thresholds_are_honoured(nb, oracle):
    S, T = 16, 80
    pcm = nb.synth_pcm(S, T, first_stream=32)
    for nn_id, th in ((1, (30000, 2)), (0, (16383, 1)), (2, (100, 9))):
        m = _model(nb, nn_id, False)
        b = nb.NNSPBatch(m, S, thresh_prob=th[0], th_count=th[1])
        res = b.exec(pcm)
        m_or = oracle.model(nn_id, False)
        for s in range(S):
            r, _ = oracle.nnsp_run(m_or, pcm[s], thresh_prob=th[0], th_count=th[1], taps=False)
            assert (r == res[s]).all()
        b.close()


def test_network_paths_share_one_state(nb, oracle):
    """Switching the network path between calls must not disturb a stream: context, LSTM state, counters and
    the stride-2 phase are one canonical state whichever kernels advance it (odd chunk lengths flip the phase)."""
    S, T = 37, 45
    pcm = nb.synth_pcm(S, T, first_stream=5)
    m = _model(nb, 0, False)
    b = nb.NNSPBatch(m, S)
    parts, t = [], 0
    for n, path in ((7, "split"), (5, "imma"), (1, "split"), (9, "dp2a"), (23, "split")):
        b.set_nn_path(path)
        parts.append(b.exec(pcm[:, t * 160:(t + n) * 160]))
        t += n
    assert t == T
    got = np.concatenate(parts, axis=1)
    m_or = oracle.model(0, False)
    for s in range(S):
        r, _ = oracle.nnsp_run(m_or, pcm[s], taps=False)
        assert (r == got[s]).all(), "stream %d" % s
    b.close()


def test_ingest_conditioning_matches_the_application(nb, oracle):
    """evb/src/main_nnsp.cc:58-65: `raw & 0xFFF0` as int16 and the sample-3 glitch interpolation of every frame."""
    rng = np.random.default_rng(7)
    raw = rng.integers(0, 2**32, (37, 9 * 160), dtype=np.uint64).astype(np.uint32)
    raw[0, :160] = 0xFFFFFFFF
    raw[1, 2] = 0x00007FF0; raw[1, 4] = 0x00007FF0          # (32752 + 32752) >> 1 needs more than 16 bits
    raw[2, 2] = 0x00008000; raw[2, 4] = 0x00008000          # two negative neighbours
    got = nb.ingest_audadc(raw)
    want = oracle.ingest_audadc(raw)
    assert (got == want).all()
    ref = (raw & 0xFFF0).astype(np.uint16).view(np.int16).reshape(37, 9, 160).copy()
    ref[:, :, 3] = (ref[:, :, 2].astype(np.int32) + ref[:, :, 4]) >> 1
    assert (want.reshape(37, 9, 160) == ref).all()


def test_back_to_back_calls_are_pipelined_correctly(nb, oracle):
    """Device-buffer calls issued without a sync in between: the engine runs the front end of call N+1 while the network
    kernels of call N are still in flight (double-buffered features). Results of every call must still be exact."""
    S, n_calls = 100, 9
    lens = [10, 1, 7, 10, 3, 10, 2, 10, 11]
    T = sum(lens)
    pcm = nb.synth_pcm(S, T, first_stream=21)
    m = _model(nb, 0, False)
    b = nb.NNSPBatch(m, S)
    d_pcm, d_res, t = [], [], 0
    for n in lens:
        d_pcm.append(nb.DeviceArray.from_host(pcm[:, t * 160:(t + n) * 160]))
        d_res.append(nb.DeviceArray((S, n), nb.RESULT_DT))
        t += n
    for k, n in enumerate(lens):                       # no sync between the calls
        b.exec_device(d_pcm[k], n * 160, n, d_res[k])
    b.sync()
    got = np.concatenate([r.to_host() for r in d_res], axis=1)
    m_or = oracle.model(0, False)
    for s in range(S):
        r, _ = oracle.nnsp_run(m_or, pcm[s], taps=False)
        assert (r == got[s]).all(), "stream %d" % s
    for x in d_pcm + d_res:
        x.free()
    b.close()


def test_async_host_calls_double_buffered(nb, oracle):
    """nnsp_b200_batch_exec_host_async / _wait_host: a server loop with two pinned PCM/result buffer pairs, one call in
    flight while the previous one is consumed; odd call lengths flip the stride-2 inference gate between calls; a
    device-buffer call and a synchronous host call are mixed in behind the asynchronous ones, then 1-frame device-buffer
    and host calls interleaved (each keeps one frame of the 2-frame PCM history the call before it wrote)."""
    S, n = 600, 7                                      # 600 streams -> 2 pipeline slices; 7 frames per call
    calls = 9
    ones = (True, True, False, True, False, False)     # the 1-frame calls: device buffers (no sync between) or host
    T = n * (calls + 2) + len(ones)
    pcm = nb.synth_pcm(S, T, first_stream=5)
    for nn_id in (1, 0):
        b = nb.NNSPBatch(_model(nb, nn_id, False), S)
        pin = [nb.PinnedArray((S, n * 160), np.int16) for _ in range(2)]
        pres = [nb.PinnedArray((S, n), nb.RESULT_DT) for _ in range(2)]
        got, prev = [], None
        for k in range(calls):
            pin[k & 1].array[...] = pcm[:, k * n * 160:(k + 1) * n * 160]
            tk = b.exec_host_async(pin[k & 1].array, pres[k & 1].array)
            assert tk == k + 1
            if prev is not None:
                b.wait_host(prev)
                got.append(pres[(k - 1) & 1].array.copy())
            prev = tk
        b.wait_host(prev)
        b.wait_host(1)                                 # an old ticket: already complete, returns at once
        got.append(pres[(calls - 1) & 1].array.copy())
        got.append(b.exec(pcm[:, calls * n * 160:(calls + 1) * n * 160].copy()))          # device-buffer call
        got.append(b.exec_host(pcm[:, (calls + 1) * n * 160:(calls + 2) * n * 160].copy()))   # synchronous host call
        tail = []
        for j, dev in enumerate(ones):
            t = (calls + 2) * n + j
            part = pcm[:, t * 160:(t + 1) * 160].copy()
            if dev:
                tail.append((nb.DeviceArray.from_host(part), nb.DeviceArray((S, 1), nb.RESULT_DT)))
                b.exec_device(tail[-1][0], 160, 1, tail[-1][1])
            else:
                tail.append((None, b.exec_host(part)))
        b.sync()
        for dp, r in tail:
            got.append(r if dp is None else r.to_host())
            if dp is not None:
                dp.free(); r.free()
        got = np.concatenate(got, axis=1)
        m_or = oracle.model(nn_id, False)
        for s in list(range(0, S, 37)) + [S - 1]:
            r, _ = oracle.nnsp_run(m_or, pcm[s], taps=False)
            assert (r == got[s]).all(), "model %d stream %d" % (nn_id, s)
        with pytest.raises(Exception):
            b.wait_host(calls + 5)                     # a ticket that was never handed out
        for x in pin + pres:
            x.free()
        b.close()


@pytest.mark.parametrize("kind", ["batch", "cascade"])
def test_async_host_calls_of_varying_odd_lengths(nb, oracle, kind):
    """Asynchronous host-buffer calls whose lengths differ from call to call (odd ones flip the inference gate, so the
    inference count of a call changes even at equal length): consecutive calls run on different pipeline streams, and a
    stream slice must still own its scratch bytes exclusively. Repeated several times; every stream checked against one
    device-buffer call over the same audio (which the other tests pin to the oracle)."""
    lens = [7, 7, 5, 12, 1, 9, 9, 3, 20, 7, 6, 11]
    S, T = 4200, sum(lens)                           # 16 / 8 slices over the pipeline streams
    pcm = nb.synth_pcm(S, T, first_stream=3)
    if kind == "batch":
        make = lambda: nb.NNSPBatch(_model(nb, 1, False), S)
        res_dt = nb.RESULT_DT
    else:
        models = [nb.Model.from_blob(nb.MODEL_DIR + "/" + f) for f in ("s2i.nnspm", "vad.nnspm", "kws_galaxy.nnspm")]
        make = lambda: nb.Cascade(models, S, params=dict(thresh_timeout_kws=40, thresh_timeout_s2i=30))
        res_dt = nb.CASCADE_RESULT_DT
    ref = make()
    want = ref.exec(pcm)
    ref.close()
    nmax = max(lens)
    pin = [nb.PinnedArray((S, nmax * 160), np.int16) for _ in range(3)]
    pres = [nb.PinnedArray((S, nmax), res_dt) for _ in range(3)]
    for rep in range(3):
        h = make()
        got, tickets, t = [], [], 0
        for k, n in enumerate(lens):
            if k >= 3:                                  # the buffer pair about to be reused: its call must be over
                h.wait_host(tickets[k - 3])
                got.append(pres[k % 3].array.reshape(-1)[: S * lens[k - 3]].reshape(S, lens[k - 3]).copy())
            pv = pin[k % 3].array.reshape(-1)[: S * n * 160].reshape(S, n * 160)
            pv[...] = pcm[:, t * 160:(t + n) * 160]
            rv = pres[k % 3].array.reshape(-1)[: S * n].reshape(S, n)
            tickets.append(h.exec_host_async(pv, rv))
            t += n
        for k in range(len(lens) - 3, len(lens)):
            h.wait_host(tickets[k])
            got.append(pres[k % 3].array.reshape(-1)[: S * lens[k]].reshape(S, lens[k]).copy())
        h.close()
        got = np.concatenate(got, axis=1)
        for f in want.dtype.names:
            bad = np.nonzero((got[f] != want[f]).reshape(S, -1).any(axis=1))[0]
            assert len(bad) == 0, "%s rep %d: field %s differs on streams %s" % (kind, rep, f, bad[:8].tolist())
    for x in pin + pres:
        x.free()


def test_long_call_many_inference_rounds(nb, oracle):
    """One call of 301 frames (151 inferences): several 16-inference work items per tile in the fc kernels, several
    staging rounds in the post kernel, a long TMA ring in the scan."""
    S, T = 19, 301
    pcm = nb.synth_pcm(S, T, first_stream=77)
    for nn_id in (0, 2):
        m = _model(nb, nn_id, False)
        b = nb.NNSPBatch(m, S)
        assert b.nn_path == "split"
        res, taps = b.exec(pcm, taps=True)
        plain = nb.NNSPBatch(m, S).exec(pcm)
        m_or = oracle.model(nn_id, False)
        for s in range(S):
            _compare_stream(oracle, m_or, pcm[s], res[s], taps, s)
        assert (plain == res).all()
        b.close()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_many_pipelined_calls_equal_one_shot(nb, seed):
    """40 back-to-back calls of random lengths (no sync in between) on 1 000 streams must give exactly what one call
    over the same 200 frames gives: stresses the two-stream pipeline (buffer reuse, history roll, phase of the gate)."""
    rng = np.random.default_rng(seed)
    S, T = 1000, 200
    cuts = np.sort(rng.choice(np.arange(1, T), 39, replace=False))
    lens = np.diff(np.concatenate([[0], cuts, [T]])).tolist()
    pcm = nb.synth_pcm(S, T, first_stream=seed * 100)
    m = _model(nb, (0, 2, 1)[seed - 1], seed == 2)
    one = nb.NNSPBatch(m, S)
    want = one.exec(pcm)
    one.close()
    b = nb.NNSPBatch(m, S)
    d_pcm, d_res, t = [], [], 0
    for n in lens:
        d_pcm.append(nb.DeviceArray.from_host(pcm[:, t * 160:(t + n) * 160]))
        d_res.append(nb.DeviceArray((S, n), nb.RESULT_DT))
        t += n
    for k, n in enumerate(lens):
        b.exec_device(d_pcm[k], n * 160, n, d_res[k])
    b.sync()
    got = np.concatenate([r.to_host() for r in d_res], axis=1)
    assert (got == want).all()
    for x in d_pcm + d_res:
        x.free()
    b.close()


@pytest.mark.parametrize("S", [1, 15, 16, 17, 33])
def test_tile_boundaries_and_strided_input(nb, oracle, S):
    """Stream counts around the 16-stream tile size, PCM rows with padding between streams (stream_stride > n_frames*160),
    and one-frame calls (what a real-time caller issues)."""
    T = 21
    pcm = nb.synth_pcm(S, T, first_stream=300 + S)
    wide = np.zeros((S, T * 160 + 96), np.int16)             # 96 samples of padding after every stream's chunk
    wide[:, :T * 160] = pcm
    wide[:, T * 160:] = 12345
    m = _model(nb, 1, False)
    m_or = oracle.model(1, False)
    want = np.stack([oracle.nnsp_run(m_or, pcm[s], taps=False)[0] for s in range(S)])
    b = nb.NNSPBatch(m, S)
    d = nb.DeviceArray.from_host(wide)
    r = nb.DeviceArray((S, T), nb.RESULT_DT)
    b.exec_device(d, wide.shape[1], T, r)                     # strided device input
    b.sync()
    assert (r.to_host() == want).all()
    b.close()
    b = nb.NNSPBatch(m, S)                                    # (a fresh handle: NNSPClass_reset keeps context row 5)
    res = np.empty((S, T), nb.RESULT_DT)
    from nnsp_b200.capi import lib, check
    import ctypes as C
    check(lib().nnsp_b200_batch_exec_host(b.h, wide.ctypes.data_as(C.c_void_p), wide.shape[1], T, res.ctypes.data_as(C.c_void_p)))
    assert (res == want).all()                                # strided host input (2-D copy)
    b.close()
    b = nb.NNSPBatch(m, S)
    one = [b.exec(pcm[:, t * 160:(t + 1) * 160]) for t in range(T)]     # frame by frame
    assert (np.concatenate(one, axis=1) == want).all()
    b.close(); d.free(); r.free()
