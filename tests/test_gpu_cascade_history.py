"""The cascade's PCM and log-mel histories: the front end of every call writes each stream's newest frames and log-mel
rows into the next call's history buffers (feat_kernel), and copies what stays of the old histories when a stream has
fewer frames in the call than a history holds. The three buffers of each history rotate once per call, whichever way
the call is issued, so that a pipelined call's front end never writes one that a chain still in flight reads, and all
slices of a host call read the same ones.

  call lengths : back-to-back calls of 1, 2, 57, 81, 82, 83, 100 and 257 frames mixed, issued as pipelined device
                 calls, on the sequential path, with taps, as asynchronous host tickets (256 streams: four slices on
                 three CUDA streams) and as one sequence that interleaves device, host and tapped calls; every stream's
                 records byte for byte against the pipelined device calls, and every 7th stream against the oracle over
                 its whole audio, with the 80-frame look-back and with none (the PCM history is then the two frames the
                 analysis window reaches back);
  records      : the same calls on the pipelined path and on the sequential path leave byte-identical stream records
                 after every call, for uniform and for ragged calls (counts 0 .. 257);
  resets       : streams reset and imported between pipelined device calls and between host tickets continue from
                 their new histories."""
import numpy as np
import pytest

import test_gpu_cascade_ragged as R

S = 256
LENGTHS = (100, 1, 2, 57, 81, 82, 83, 257, 100, 3, 100)
LOOKBACK = {"lookback80": {}, "lookback0": dict(frs_vbufBk_kws=0, frs_vbufBk_s2i=0)}
# how the calls of LENGTHS are issued, call k as issue[k % len(issue)]: "device" (exec_device, nothing waited for
# between the calls), "host" (exec_host_async tickets, nothing waited for between them) or "tapped" (exec with taps)
ISSUE = {"pipelined": ("device",), "sequential": ("device",), "tapped": ("tapped",), "host": ("host",),
         "mixed": ("device", "device", "host", "host", "tapped", "device", "host", "tapped", "tapped", "host", "device")}


def _params(extra):
    return dict(R.TRIOS["shipped"][2], **extra)


def _handle(nb, path, extra):
    h = nb.Cascade(R.gpu_models(nb, "shipped", False), S, params=_params(extra))
    h.set_path(path)
    return h


def _calls(nb, h, pcm, issue, before=None):
    """the calls of LENGTHS over pcm, issued as `issue` says, before(h, k) right before call k; the records of each"""
    how = [issue[k % len(issue)] for k in range(len(LENGTHS))]
    bufs, pos = [], 0
    for k, n in enumerate(LENGTHS):                  # every buffer first: the calls then go back to back
        part = np.ascontiguousarray(pcm[:, pos * 160:(pos + n) * 160])
        if how[k] == "device":
            bufs.append((nb.DeviceArray.from_host(part), nb.DeviceArray((S, n), nb.CASCADE_RESULT_DT)))
        elif how[k] == "host":
            bufs.append((nb.PinnedArray(part.shape, np.int16), nb.PinnedArray((S, n), nb.CASCADE_RESULT_DT)))
            bufs[-1][0].array[...] = part
        else:
            bufs.append((part, None))
        pos += n
    out = [None] * len(LENGTHS)
    for k, n in enumerate(LENGTHS):
        if before:
            before(h, k)
        p, r = bufs[k]
        if how[k] == "device":
            h.exec_device(p, n * 160, n, r)
        elif how[k] == "host":
            h.exec_host_async(p.array, r.array)
        else:
            out[k] = h.exec(p, taps=True)[0]
    h.sync()
    for k, (p, r) in enumerate(bufs):
        if how[k] != "tapped":
            out[k] = r.to_host() if how[k] == "device" else r.array.copy()
            p.free(); r.free()
    return out


CASES = [pytest.param(issue, lb, id=lb if issue == "pipelined" else issue + "-" + lb) for issue in ISSUE for lb in sorted(LOOKBACK)]


@pytest.mark.gpu
@pytest.mark.parametrize("issue,lookback", CASES)
def test_pipelined_call_lengths_against_the_oracle(nb, oracle, issue, lookback):
    pcm = nb.synth_pcm(S, sum(LENGTHS), first_stream=R.FIRST)
    h = _handle(nb, "sequential" if issue == "sequential" else "auto", LOOKBACK[lookback])
    got = _calls(nb, h, pcm, ISSUE[issue])
    h.close()
    if issue != "pipelined":
        ref = _handle(nb, "auto", LOOKBACK[lookback])
        want = _calls(nb, ref, pcm, ISSUE["pipelined"])
        ref.close()
        for k, n in enumerate(LENGTHS):
            assert got[k].tobytes() == want[k].tobytes(), "records of the %d-frame call %d differ from the pipelined device call's" % (n, k)
    got = np.concatenate(got, axis=1)
    om = [oracle.model(i, False) for i in range(3)]
    par = R._params(oracle, nb, _params(LOOKBACK[lookback]))
    for s in range(0, S, 7):
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


def _resets_and_imports(recs):
    def before(h, k):
        if k == 3:
            h.reset_streams([0, 5, 30, 100, 250])
        if k == 5:
            h.reset_streams([7, 8, 140], fresh=True)
            h.import_streams([12, 2, 33, 201], recs)
    return before


@pytest.mark.gpu
def test_resets_and_imports_between_pipelined_calls(nb):
    pcm = nb.synth_pcm(S, sum(LENGTHS), first_stream=R.FIRST)
    donor = _handle(nb, "sequential", {})
    donor.exec(pcm[:, :150 * 160])
    recs = donor.export_streams([3, 11, 20, 130])
    donor.close()
    results = []
    for path, issue in (("auto", "pipelined"), ("sequential", "sequential"), ("auto", "host")):
        h = _handle(nb, path, {})
        out = _calls(nb, h, pcm, ISSUE[issue], _resets_and_imports(recs))
        results.append(([r.tobytes() for r in out], h.export_streams(np.arange(S))))
        h.close()
    for issue, (records, state) in zip(("sequential", "host"), results[1:]):
        assert results[0][0] == records, "records of the %s calls differ from the pipelined ones" % issue
        assert results[0][1] == state, "stream state after the %s calls differs from the pipelined one" % issue
