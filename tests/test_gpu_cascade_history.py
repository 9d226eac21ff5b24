"""The cascade's PCM history on pipelined device calls: the front end of a call writes each stream's newest frames into
the next call's history buffer (feat_kernel), which also copies the frames of the old history that stay when a stream
has fewer frames in the call than the history holds, and three history buffers rotate so that the next call's front
end never writes one that a chain still in flight reads.

  call lengths : back-to-back calls without a host wait between them, 1, 2, 57, 81, 82, 83, 100 and 257 frames mixed,
                 against the oracle over each stream's whole audio, with the 80-frame look-back and with none (the
                 history is then the two frames the analysis window reaches back);
  records      : the same calls on the pipelined path and on the sequential path (in-place history update) leave
                 byte-identical stream records after every call, for uniform and for ragged calls (counts 0 .. 257);
  resets       : streams reset and imported between pipelined calls continue from their new history.
The log-mel history (the look-back rows of the delayed stages) goes the same way: feat_kernel writes the newest rows,
cascade_ctx_kernel copies the old rows that stay."""
import numpy as np
import pytest

import test_gpu_cascade_ragged as R

S = 37
LENGTHS = (100, 1, 2, 57, 81, 82, 83, 257, 100, 3, 100)
LOOKBACK = {"lookback80": {}, "lookback0": dict(frs_vbufBk_kws=0, frs_vbufBk_s2i=0)}


def _params(extra):
    return dict(R.TRIOS["shipped"][2], **extra)


def _handle(nb, path, extra):
    h = nb.Cascade(R.gpu_models(nb, "shipped", False), S, params=_params(extra))
    h.set_path(path)
    return h


def _pipelined(nb, h, pcm, lengths):
    """every call queued before any is waited for; the records of each call"""
    bufs, pos = [], 0
    for n in lengths:
        bufs.append((nb.DeviceArray.from_host(np.ascontiguousarray(pcm[:, pos * 160:(pos + n) * 160])),
                     nb.DeviceArray((S, n), nb.CASCADE_RESULT_DT)))
        pos += n
    for (dp, dr), n in zip(bufs, lengths):
        h.exec_device(dp, n * 160, n, dr)
    h.sync()
    out = [dr.to_host() for _, dr in bufs]
    for dp, dr in bufs:
        dp.free(); dr.free()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("lookback", sorted(LOOKBACK))
def test_pipelined_call_lengths_against_the_oracle(nb, oracle, lookback):
    frames = sum(LENGTHS)
    pcm = nb.synth_pcm(S, frames, first_stream=R.FIRST)
    h = _handle(nb, "auto", LOOKBACK[lookback])
    got = np.concatenate(_pipelined(nb, h, pcm, LENGTHS), axis=1)
    h.close()
    om = [oracle.model(i, False) for i in range(3)]
    par = R._params(oracle, nb, _params(LOOKBACK[lookback]))
    for s in range(S):
        want = oracle.cascade_run(om, pcm[s], params=par, taps=False)[0]
        for f in R.FIELDS:
            assert (got[s][f] == want[f]).all(), "field %s of stream %d differs from the oracle" % (f, s)


@pytest.mark.gpu
@pytest.mark.parametrize("lookback", sorted(LOOKBACK))
def test_records_match_the_sequential_path(nb, lookback):
    frames = sum(LENGTHS)
    pcm = nb.synth_pcm(S, frames, first_stream=R.FIRST)
    a, b = _handle(nb, "auto", LOOKBACK[lookback]), _handle(nb, "sequential", LOOKBACK[lookback])
    every = np.arange(S)
    pos = 0
    for n in LENGTHS:
        part = np.ascontiguousarray(pcm[:, pos * 160:(pos + n) * 160])
        ra = a.exec(part)
        rb = b.exec(part)
        assert ra.tobytes() == rb.tobytes(), "records of the %d-frame call differ" % n
        assert a.export_streams(every) == b.export_streams(every), "stream state after the %d-frame call differs" % n
        pos += n
    # ragged calls: every count of 0 .. 257 frames that straddles the 82-frame PCM history
    counts = (0, 1, 2, 3, 57, 80, 81, 82, 83, 99, 100, 257)
    rng = np.random.default_rng(5)
    for k in range(4):
        n = np.array([counts[(5 * s + 3 * k) % len(counts)] for s in range(S)], np.int32)
        T = int(n.max())
        part = rng.integers(-8000, 8000, (S, T * 160), dtype=np.int16)
        ra = a.exec_ragged(part, n)
        rb = b.exec_ragged(part, n)
        assert ra.tobytes() == rb.tobytes(), "records of ragged call %d differ" % k
        assert a.export_streams(every) == b.export_streams(every), "stream state after ragged call %d differs" % k
    a.close(); b.close()


@pytest.mark.gpu
def test_resets_and_imports_between_pipelined_calls(nb):
    frames = sum(LENGTHS)
    pcm = nb.synth_pcm(S, frames, first_stream=R.FIRST)
    donor = _handle(nb, "sequential", {})
    donor.exec(pcm[:, :150 * 160])
    recs = donor.export_streams([3, 11, 20])
    donor.close()
    handles = [_handle(nb, "auto", {}), _handle(nb, "sequential", {})]
    results = []
    for h in handles:
        pos, out = 0, []
        for k, n in enumerate(LENGTHS):
            if k == 3:
                h.reset_streams([0, 5, 30])
            if k == 5:
                h.reset_streams([7, 8], fresh=True)
                h.import_streams([12, 2, 33], recs)
            dp = nb.DeviceArray.from_host(np.ascontiguousarray(pcm[:, pos * 160:(pos + n) * 160]))
            dr = nb.DeviceArray((S, n), nb.CASCADE_RESULT_DT)
            h.exec_device(dp, n * 160, n, dr)
            out.append((dp, dr))
            pos += n
        h.sync()
        results.append(([dr.to_host().tobytes() for _, dr in out], h.export_streams(np.arange(S))))
        for dp, dr in out:
            dp.free(); dr.free()
        h.close()
    assert results[0][0] == results[1][0]
    assert results[0][1] == results[1][1]
