"""Sessions of a live cascade handle (nnsp_b200_cascade_export_streams / _import_streams, nnsp_b200_group_export_streams
/ _import_streams): a stream's whole state leaves its slot as a record and continues in another slot, another handle or
another member of a group.

A moved stream is a session: its oracle is Oracle.cascade_run over its own uninterrupted audio (R.oracle_run), whichever
slot and handle it runs in.

  move and continue : pipelined calls of 37 sessions spread over two handles whose stages change every ~10 frames; before
                      each call a subset is exported from one handle and imported into a permuted set of free slots of
                      the other while that one's previous call may still run, and the vacated slots are reset FRESH. The
                      cuts fall in every live stage, with a time-out counter running, with the look-back history full, on
                      instances entered on the call's last frame or the one before (ages 0 and 1) -- a stage change left
                      on a call's last frame for the next call. Every record of every session against the oracle, and a
                      final tapped 2-frame call after one more move; default path with 1 and 4 rounds, sequential path,
                      tcgen05 first round, ragged calls with the moved sessions idle in the call after their move, tapped
                      calls; the shipped trio and a wide one (LSTM state at offsets not a multiple of 4), both
                      accumulator modes;
  round trip        : every stream into the same slots of a new handle continues byte for byte; an export right after an
                      import returns the imported bytes;
  composition       : import -> INSTANCE, import -> FRESH, FRESH -> import, import -> import, the whole-handle reset after
                      an import, and an export with operations pending, each against its sequential definition;
  stale pool slot   : imports after an import that a FRESH reset replaced, with a call between, each load their own record;
  no cost unused    : calls without pending imports make the launches, the copies (every memcpy and memset of a
                      torch.profiler trace) and the records of a handle that never saw the functions;
  host calls        : 4100 streams, 8 slices, PCM16 and AUDADC words, an import between two asynchronous tickets;
  group             : a cascade group with the device named twice, sessions moved across the member boundary; a batch
                      group refuses;
  refusals          : records of other models, accumulator mode, sequence and look-back depths; bad magic, version and
                      size; every range-checked field out of range; duplicate destinations; ids out of range -- all refused
                      on the host and nothing recorded. No test sends such a record to the device."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import test_gpu_cascade_ragged as R

S2I, VAD, KWS = 0, 1, 2
SEQ = (VAD, KWS, S2I)
S, MAXF, NCALLS = R.S, R.MAXF, R.NCALLS
ERR_ARG = -1                           # NNSP_B200_ERR_ARG
HEADER_FIELDS = {"magic": 0, "version": 4, "record_bytes": 8, "len_seq": 12, "seq": 16, "frs_vbufBk_kws": 28,
                 "frs_vbufBk_s2i": 30, "model_fnv1a": 32, "reserved": 56}
# body offsets the refusal test edits (DESIGN.md section 4.3): NNSPClass scalars, then the controller scalars
REC_SCAL, REC_CASC = 64, 96
SC_ARGMAX_LAST, SC_SLIDES = 12, 13
CS_POS, CS_CNT_KWS, CS_CNT_S2I, CS_AGE = 0, 1, 2, 3


@pytest.fixture(autouse=True)
def _library_defaults(monkeypatch):
    for e in R.SWITCHES:
        monkeypatch.delenv(e, raising=False)


# ---------------------------------------------------------------------------------------------------------------------
# the record header, without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_header_struct_layout(nb, tmp_path):
    """capi.StreamHeader is nnsp_b200_stream_header: 64 bytes, the documented offsets, as the C compiler lays it out"""
    H = nb.capi.StreamHeader
    assert C.sizeof(H) == 64
    assert {n: getattr(H, n).offset for n, _ in H._fields_} == HEADER_FIELDS
    cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
    assert cc, "no C compiler"
    src = tmp_path / "hdr.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "nnsp_b200.h"\nint main(void) {\n'
                   '  printf("size %zu\\n", sizeof(nnsp_b200_stream_header));\n' +
                   "".join('  printf("%s %%zu\\n", offsetof(nnsp_b200_stream_header, %s));\n' % (n, n) for n in HEADER_FIELDS) +
                   '  printf("MAGIC %u\\nVERSION %u\\n", (unsigned)NNSP_B200_STREAM_MAGIC, (unsigned)NNSP_B200_STREAM_VERSION);\n'
                   "  return 0;\n}\n")
    exe = tmp_path / "hdr"
    subprocess.run([cc, "-I", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got.pop("size")) == 64
    assert int(got.pop("MAGIC")) == nb.capi.STREAM_MAGIC and int(got.pop("VERSION")) == nb.capi.STREAM_VERSION
    assert {k: int(v) for k, v in got.items()} == HEADER_FIELDS


# ---------------------------------------------------------------------------------------------------------------------
# move and continue, every frame against the oracle
# ---------------------------------------------------------------------------------------------------------------------
KINDS = ("stage%d" % S2I, "stage%d" % VAD, "stage%d" % KWS, "counter", "history_full", "age0", "age1")


def kinds_of(want, s, p):
    """the kinds of state session s is in after its first p >= 3 frames (oracle records)"""
    pa = want["pos_after"][s]
    k = {"stage%d" % SEQ[pa[p - 1]]}
    if want["cnt_timeout"][s][p - 1] > 0:
        k.add("counter")
    if p >= 82:
        k.add("history_full")                          # 82 PCM frames and 80 log-mel rows of look-back
    if pa[p - 1] != pa[p - 2]:
        k.add("age0")                                  # entered on the call's last frame: the change is left for the next call
    elif pa[p - 2] != pa[p - 3]:
        k.add("age1")
    return k


def move_plan(want, ragged):
    """slots, moves and counts of the move test: (where [NCALLS + 2] of {session: (handle, slot)}, moves [NCALLS + 1] of
    [(session, from, to)], counts [NCALLS][S] per session, positions). Sessions 0 .. 18 start in handle 0, 19 .. 36 in
    handle 1; before call k >= 1 (and before the tapped probe) sessions move from handle k % 2 ... to free slots of the
    other, in reverse slot order; in ragged calls a moved session idles in the call after its move."""
    where = {s: (0, s) if s < 19 else (1, S - 1 - (s - 19)) for s in range(S)}
    counts = R.schedule().copy() if ragged else np.full((NCALLS, S), MAXF)
    plan_where, moves = [dict(where)], [[]]
    pos = np.zeros(S, int)
    for k in range(1, NCALLS + 1):
        pos = pos + counts[k - 1]
        src = (k + 1) % 2
        cand = [s for s in sorted(where, key=lambda s: where[s][1]) if where[s][0] == src and pos[s] >= 3]
        pick = [s for s in cand if (5 * s + k) % 3 == 0]
        for kind in KINDS:                             # the first two sessions of every kind of state
            pick += [s for s in cand if kind in kinds_of(want, s, pos[s])][:2]
        pick = sorted(set(pick), key=lambda s: where[s][1])
        used = {where[s][1] for s in where if where[s][0] == 1 - src}
        free = sorted(set(range(S)) - used, reverse=True)
        pick = pick[:len(free)]
        mv = [(s, where[s], (1 - src, free[i])) for i, s in enumerate(pick)]
        for s, _, to in mv:
            where[s] = to
        if ragged and k < NCALLS:
            counts[k][pick] = 0
        moves.append(mv)
        plan_where.append(dict(where))
    return plan_where, moves, counts


def plan_kinds(want, moves, counts):
    pos = R.positions(counts)
    got = set()
    for k in range(1, len(moves)):
        for s, _, _ in moves[k]:
            got |= kinds_of(want, s, pos[k][s])
    return got


ARMS = {
    "rounds1": {"NNSP_B200_CASCADE_ROUNDS": "1"},
    "rounds4": {"NNSP_B200_CASCADE_ROUNDS": "4"},
    "default": {},
    "sequential": {},
    "tc5_first_round": {"NNSP_B200_TC5": "2"},
    "ragged": {},
    "tapped": {},
}
CASES = [("shipped", False, a) for a in ARMS] + [("shipped", True, "default"), ("shipped", True, "ragged"),
                                                 ("wide_rows81", False, "ragged"), ("wide_rows81", True, "default"),
                                                 ("wide_rows81", True, "sequential"), ("wide_rows81", True, "ragged")]
# (the wide trio's acc64 sessions end no 100-frame call in KWS: that mode runs ragged calls, whose cuts fall there)


def occupants(where, handle):
    """(sessions, slots) of one handle, in slot order"""
    pairs = sorted((slot, s) for s, (h, slot) in where.items() if h == handle)
    return np.array([s for _, s in pairs], int), np.array([slot for slot, _ in pairs], int)


def move(handles, mv):
    """export the sessions of mv from their handle, import them into their new slots, reset the vacated slots FRESH"""
    if not mv:
        return
    src, dst = mv[0][1][0], mv[0][2][0]
    recs = handles[src].export_streams([f[1] for _, f, _ in mv])
    handles[dst].import_streams([t[1] for _, _, t in mv], recs)
    handles[src].reset_streams([f[1] for _, f, _ in mv], fresh=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name,acc32,arm", CASES, ids=["%s-%s-%s" % (n, "acc32" if a else "acc64", m) for n, a, m in CASES])
def test_move_and_continue_every_frame(nb, oracle, monkeypatch, name, acc32, arm):
    for k, v in ARMS[arm].items():
        monkeypatch.setenv(k, v)
    ragged, tapped = arm == "ragged", arm == "tapped"
    pcm, want, wtap, _ = R.oracle_run(nb, oracle, name, acc32)
    where, moves, counts = move_plan(want, ragged)
    assert plan_kinds(want, moves, counts) == set(KINDS)
    pos = R.positions(counts)
    handles = [nb.Cascade(R.gpu_models(nb, name, acc32), S, params=R.TRIOS[name][2]) for _ in range(2)]
    if arm == "sequential":
        for h in handles:
            h.set_path("sequential")
    tc0 = nb.tc5_launches()
    junk = np.random.default_rng(31)
    keep, out = [], []
    for k in range(NCALLS):
        move(handles, moves[k])
        calls = []
        for hi, h in enumerate(handles):
            sess, slots = occupants(where[k], hi)
            hp, hn = np.zeros((S, pcm.shape[1]), np.int16), np.full(S, MAXF)
            hp[slots] = pcm[sess]
            hn[slots] = counts[k][sess]
            hpos = np.zeros(S, int)
            hpos[slots] = pos[k][sess]
            buf = R.call_pcm(hp, hpos, hn, MAXF, junk)       # junk past the counts, vacant slots silent
            if tapped:
                res, taps = h.exec(buf, taps=True)
                calls.append((hi, sess, slots, res, taps))
                continue
            dp, dn, dr = nb.DeviceArray.from_host(buf), nb.DeviceArray.from_host(hn.astype(np.int32)), \
                nb.DeviceArray((S, MAXF), nb.CASCADE_RESULT_DT)
            keep.append((dp, dn, dr))
            if ragged:
                h.exec_ragged_device(dp, MAXF * 160, MAXF, dn, dr)
            else:
                h.exec_device(dp, MAXF * 160, MAXF, dr)
            calls.append((hi, sess, slots, dr, None))
        out.append(calls)
    for h in handles:
        h.sync()
    for k, calls in enumerate(out):
        for hi, sess, slots, r, taps in calls:
            got = r if isinstance(r, np.ndarray) else r.to_host()
            tp = None if taps is None else {g: taps[g][slots] for g, _ in R.CASC_TAPS}
            R.check(got[slots], tp, want[sess], {g: v[sess] for g, v in wtap.items()}, pos[k][sess], counts[k][sess],
                    "%s call %d handle %d" % (arm, k, hi))
    for x in keep:
        for a in x:
            a.free()
    # one more move, then a tapped call: every tap of its two frames reads the moved state
    move(handles, moves[NCALLS])
    end = pos[NCALLS]
    for hi, h in enumerate(handles):
        sess, slots = occupants(where[NCALLS], hi)
        probe = np.zeros((S, 2 * 160), np.int16)
        for s, slot in zip(sess, slots):
            probe[slot] = pcm[s, end[s] * 160:(end[s] + 2) * 160]
        res, taps = h.exec(probe, taps=True)
        R.check(res[slots], {g: taps[g][slots] for g, _ in R.CASC_TAPS}, want[sess], {g: v[sess] for g, v in wtap.items()},
                end[sess], np.full(len(sess), 2), "%s tapped call after the last move, handle %d" % (arm, hi))
        h.close()
    if "NNSP_B200_TC5" in ARMS[arm]:
        assert nb.tc5_launches() > tc0


# ---------------------------------------------------------------------------------------------------------------------
# round trip, byte for byte
# ---------------------------------------------------------------------------------------------------------------------
def _handle(nb, path="auto", name="shipped", acc32=False, **params):
    h = nb.Cascade(R.gpu_models(nb, name, acc32), S, params=dict(R.TRIOS[name][2], **params))
    h.set_path(path)
    return h


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["auto", "sequential"])
def test_round_trip_byte_for_byte(nb, path):
    pcm = nb.synth_pcm(S, 3 * MAXF, first_stream=R.FIRST)
    calls = [pcm[:, k * MAXF * 160:(k + 1) * MAXF * 160] for k in range(3)]
    a = _handle(nb, path)
    a.exec(calls[0])
    a.exec(calls[1])
    every = np.arange(S)
    recs = a.export_streams(every)
    rb = a.stream_state_bytes()
    assert len(recs) == S * rb
    b = _handle(nb, path)
    b.import_streams(every, recs)
    assert b.export_streams(every) == recs                 # right after the import: the imported bytes
    assert a.export_streams(every) == recs                 # exporting changes nothing
    assert a.exec(calls[2]).tobytes() == b.exec(calls[2]).tobytes()
    assert a.export_streams(every) == b.export_streams(every)
    # a stream listed twice; the record of a new handle differs from a live one's
    twice = a.export_streams([4, 4, 9])
    assert twice[:rb] == twice[rb:2 * rb]
    new = _handle(nb, path)
    assert new.export_streams([4]) != twice[:rb]
    for h in (a, b, new):
        h.close()


# ---------------------------------------------------------------------------------------------------------------------
# composition, against the sequential definition
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_composition(nb):
    pcm = nb.synth_pcm(S, 3 * MAXF, first_stream=R.FIRST)
    x0, x1, x2 = (pcm[:, k * MAXF * 160:(k + 1) * MAXF * 160] for k in range(3))
    src = _handle(nb)
    src.exec(x0)
    r1 = src.export_streams([3, 7, 30])
    src.exec(x1)
    r2 = src.export_streams([3, 7, 30])
    src.close()
    ids = [12, 0, 36]

    def run(ops):
        """ops on a live handle after one call, then a call; (its records, the state after it)"""
        h = _handle(nb)
        h.exec(x1)
        for op in ops:
            op(h)
        out = h.exec(x2)
        st = h.export_streams(np.arange(S))
        h.close()
        return out.tobytes(), st

    imp1, imp2 = (lambda h: h.import_streams(ids, r1)), (lambda h: h.import_streams(ids, r2))
    inst, fresh = (lambda h: h.reset_streams(ids)), (lambda h: h.reset_streams(ids, fresh=True))
    apply_now = lambda h: h.export_streams(ids)            # noqa: E731 -- applies what is pending, synchronously
    assert run([imp1, inst]) == run([imp1, apply_now, inst])
    assert run([imp1, inst]) != run([imp1])
    assert run([imp1, fresh]) == run([fresh])
    assert run([fresh, imp1]) == run([imp1])
    assert run([inst, imp1]) == run([imp1])
    assert run([imp1, imp2]) == run([imp2])
    assert run([imp1, inst, inst]) == run([imp1, inst])
    assert run([imp1, lambda h: h.reset()]) == run([imp1, apply_now, lambda h: h.reset()])
    # an export with operations pending applies them first
    h = _handle(nb)
    h.exec(x1)
    h.reset_streams([5], fresh=True)
    h.import_streams(ids, r1)
    got = h.export_streams([5] + ids)
    h.close()
    rb = len(r1) // 3
    new = _handle(nb)
    assert got[:rb] == new.export_streams([5])
    new.close()
    assert got[rb:] == r1


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["other_first", "same_first", "same_only"])
def test_imports_after_an_import_replaced_by_a_reset(nb, order):
    """import [5], FRESH reset [5], a call; then imports into [9] and [5] (or [5] alone): each slot continues its own
    record -- the first import's pending record leaves nothing behind that a later import reuses"""
    pcm = nb.synth_pcm(S, 3 * MAXF, first_stream=R.FIRST)
    x0, x1, x2 = (pcm[:, k * MAXF * 160:(k + 1) * MAXF * 160] for k in range(3))
    src = _handle(nb)
    src.exec(x0)
    r3, r20, r30 = (src.export_streams([s]) for s in (3, 20, 30))
    src.close()
    later = {"other_first": [(9, r20), (5, r30)], "same_first": [(5, r30), (9, r20)], "same_only": [(5, r30)]}[order]

    def run(first):
        h = _handle(nb)
        h.exec(x0)
        if first:
            h.import_streams([5], r3)
            h.reset_streams([5], fresh=True)
        h.exec(x1)
        for s, r in later:
            h.import_streams([s], r)
        ids = [s for s, _ in later]
        st = h.export_streams(ids)
        out = h.exec(x2)
        h.close()
        return st, out[ids].tobytes()

    st, got = run(True)
    assert st == b"".join(r for _, r in later)            # the state each slot's next call starts from
    assert (st, got) == run(False)


# ---------------------------------------------------------------------------------------------------------------------
# no cost when unused
# ---------------------------------------------------------------------------------------------------------------------
def _copies(prof):
    """(category, name, bytes) of every memcpy and memset of a torch.profiler run, in device order"""
    import json
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "trace.json")
        prof.export_chrome_trace(p)
        with open(p) as f:
            ev = json.load(f)["traceEvents"]
    cp = sorted((e for e in ev if e.get("cat") in ("gpu_memcpy", "gpu_memset")), key=lambda e: e["ts"])
    return [(e["cat"], e["name"], e.get("args", {}).get("bytes")) for e in cp]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["auto", "sequential"])
def test_no_cost_without_pending_imports(nb, path):
    from torch.profiler import ProfilerActivity, profile
    pcm = nb.synth_pcm(S, 4 * MAXF, first_stream=R.FIRST)
    calls = [pcm[:, k * MAXF * 160:(k + 1) * MAXF * 160] for k in range(4)]
    runs = []

    def call(h, x, out, deltas, copies):
        """one call (with the binding's upload of x and download of the records), its launches and its copies"""
        l0 = nb.kernel_launches()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out.append(h.exec(x))
            h.sync()
        deltas.append(nb.kernel_launches() - l0)
        copies.append(_copies(prof))

    for uses in (False, True):
        h = _handle(nb, path)
        out, deltas, copies = [], [], []
        for k, x in enumerate(calls):
            if uses:
                h.import_streams([], b"")                  # n == 0: nothing pending
                if k == 1:
                    h.export_streams([2, 3])
            call(h, x, out, deltas, copies)
        # one call with a pending import: one launch more, two on the pipelined path (front end and chain), and two
        # copies more (the list, the records)
        if uses:
            h.import_streams([1, 2], h.export_streams([2, 1]))
        call(h, calls[0], out, deltas, copies)
        rb = h.stream_state_bytes()
        h.close()
        runs.append((out, deltas, copies))
    (a, la, ca), (b, lb, cb) = runs
    assert [x.tobytes() for x in a[:-1]] == [x.tobytes() for x in b[:-1]]
    others = [s for s in range(S) if s not in (1, 2)]           # the last call: streams 1 and 2 swapped their states
    assert a[-1][others].tobytes() == b[-1][others].tobytes()
    assert la[:-1] == lb[:-1], (la, lb)
    assert lb[-1] - la[-1] == (1 if path == "sequential" else 2), (la, lb)
    assert all(len(c) >= 2 for c in ca), ca                # the profiler sees the binding's upload and download
    assert ca[:-1] == cb[:-1], (ca, cb)
    extra = list(cb[-1])
    for c in ca[-1]:
        extra.remove(c)
    assert sorted(e[2] for e in extra) == [2 * 4, 2 * rb], extra
    assert all(e[0] == "gpu_memcpy" and "HtoD" in e[1] for e in extra), extra


# ---------------------------------------------------------------------------------------------------------------------
# asynchronous host calls
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["pcm16", "audadc"])
def test_host_async_import_between_tickets(nb, oracle, fmt):
    n_streams, T = 4100, MAXF
    src_ids = [0, 15, 16, 511, 512, 1023, 1024, 2047, 2048, 3583, 3584, 4099, 700, 3000]
    dst_ids = src_ids[::-1][:7] + [1, 17, 1500, 2500, 3001, 4000, 4098]   # across the slices, permuted
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
    ref = nb.Cascade(models, n_streams, params=params)      # device calls with the same import
    want1 = ref.exec(pcm[:, :T * 160])
    recs = ref.export_streams(src_ids)
    ref.import_streams(dst_ids, recs)
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
    c.import_streams(dst_ids, recs)
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
    # the oracle: a slot that received stream p's state continues with its own audio
    om = [oracle.model(i, False) for i in range(3)]
    par = R._params(oracle, nb, params)
    for p, q in zip(src_ids, dst_ids):
        w, _, _ = oracle.cascade_run(om, np.concatenate([pcm[p, :T * 160], pcm[q, T * 160:]]), params=par, taps=False)
        R.check(got[1][[q]], None, w[None], None, np.array([T]), np.array([T]), "%s slot %d from stream %d" % (fmt, q, p))


# ---------------------------------------------------------------------------------------------------------------------
# group
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_group_moves_across_members(nb, oracle):
    name = "shipped"
    pcm, want, wtap, _ = R.oracle_run(nb, oracle, name, False)
    g = nb.Group(R.gpu_models(nb, name, False), S, [0, 0], params=R.TRIOS[name][2])
    edge = g.ranges()[1][1]
    assert 0 < edge < S
    assert g.stream_state_bytes() > 0
    vacant = {edge - 3, edge - 2, edge + 2, edge + 3, 0, S - 1}
    where = {s: s for s in range(S) if s not in vacant}         # session -> slot
    # before call k: two sessions next to the edge swap members into vacant slots, one moves inside a member
    plan = []
    for k in range(1, NCALLS):
        occ = sorted(where, key=lambda s: where[s])
        left = [s for s in occ if where[s] < edge][-1 - (k % 2)]
        right = [s for s in occ if where[s] >= edge][k % 2]
        free_r = sorted(set(range(edge, S)) - set(where.values()))
        free_l = sorted(set(range(edge)) - set(where.values()))
        mv = [(left, free_r[-1]), (right, free_l[0])]
        inner = [s for s in occ if where[s] < edge and s != left][k % 3]
        plan.append(mv + [(inner, free_l[-1])])
        for s, to in plan[-1]:
            where[s] = to
    where = {s: s for s in range(S) if s not in vacant}
    res, tickets, slots_of = [], [], []
    for k in range(NCALLS):
        if k:
            mv = plan[k - 1]
            recs = g.export_streams([where[s] for s, _ in mv])
            g.import_streams([to for _, to in mv], recs)
            g.reset_streams([where[s] for s, _ in mv], fresh=True)
            for s, to in mv:
                where[s] = to
        sess = np.array(sorted(where), int)
        slots = np.array([where[s] for s in sess], int)
        buf = np.zeros((S, MAXF * 160), np.int16)
        buf[slots] = pcm[sess, k * MAXF * 160:(k + 1) * MAXF * 160]
        res.append(np.empty((S, MAXF), nb.CASCADE_RESULT_DT))
        tickets.append(g.exec_host_async(buf, res[-1]))
        slots_of.append((sess, slots, buf))
    g.wait(tickets[-1])
    g.close()
    for k, (sess, slots, _) in enumerate(slots_of):
        R.check(res[k][slots], None, want[sess], None, np.full(len(sess), k * MAXF), np.full(len(sess), MAXF), "group call %d" % k)


@pytest.mark.gpu
def test_batch_group_refuses(nb):
    m = nb.Model.from_blob(nb.MODEL_DIR + "/vad.nnspm")
    g = nb.Group(m, 64, [0, 0])
    assert g.stream_state_bytes() == 0
    from nnsp_b200 import capi
    L = capi.lib()
    a = np.asarray([1, 2], np.int32)
    buf = np.zeros(4096, np.uint8)
    assert L.nnsp_b200_group_export_streams(g.h, a.ctypes.data_as(C.c_void_p), 2, buf.ctypes.data_as(C.c_void_p)) == ERR_ARG
    assert L.nnsp_b200_group_import_streams(g.h, a.ctypes.data_as(C.c_void_p), 2, buf.ctypes.data_as(C.c_void_p)) == ERR_ARG
    g.close()


# ---------------------------------------------------------------------------------------------------------------------
# refusals: on the host, nothing recorded
# ---------------------------------------------------------------------------------------------------------------------
def _edit(rec, off, fmt, value):
    r = bytearray(rec)
    r[off:off + np.dtype(fmt).itemsize] = np.array(value, fmt).tobytes()
    return bytes(r)


@pytest.mark.gpu
def test_refusals(nb):
    from nnsp_b200 import capi
    L = capi.lib()
    pcm = nb.synth_pcm(S, 2 * MAXF, first_stream=R.FIRST)
    x0, x1 = pcm[:, :MAXF * 160], pcm[:, MAXF * 160:]
    src = _handle(nb)
    src.exec(x0)
    good = src.export_streams([6])
    src.close()
    rb = len(good)
    plain = _handle(nb)
    plain.exec(x0)
    want = plain.exec(x1).tobytes()
    plain.close()

    def refused(h, ids, recs):
        a = np.asarray(ids, np.int32)
        b = np.frombuffer(recs, np.uint8) if len(recs) else np.zeros(1, np.uint8)
        assert L.nnsp_b200_cascade_import_streams(h.h, a.ctypes.data_as(C.c_void_p), len(a), b.ctypes.data_as(C.c_void_p)) == ERR_ARG
        assert nb.capi.lib().nnsp_b200_last_error()

    # records of another handle: other models, the other accumulator mode, another sequence, other look-back depths
    for other in (dict(name="wide_rows81"), dict(acc32=True), dict(seq=(VAD, S2I, KWS)), dict(frs_vbufBk_kws=40)):
        seq = other.pop("seq", SEQ)
        h = nb.Cascade(R.gpu_models(nb, other.pop("name", "shipped"), other.pop("acc32", False)), S,
                       seq=seq, params=dict(R.TRIOS["shipped"][2], **other))
        theirs = h.export_streams([6])
        assert theirs != good and len(theirs) == rb
        h.close()
        h = _handle(nb)
        h.exec(x0)
        refused(h, [6], theirs)
        assert h.exec(x1).tobytes() == want
        h.close()
    hdr = nb.capi.StreamHeader
    bad = [
        _edit(good, hdr.magic.offset, "<u4", 0x12345678),
        _edit(good, hdr.version.offset, "<u4", 2),
        _edit(good, hdr.record_bytes.offset, "<u4", rb + 8),
        _edit(good, REC_CASC + 2 * CS_POS, "<u2", 3),             # sequence position: len_seq = 3
        _edit(good, REC_CASC + 2 * CS_AGE, "<u2", 3),
        _edit(good, REC_CASC + 2 * CS_CNT_KWS, "<u2", 32767),
        _edit(good, REC_CASC + 2 * CS_CNT_S2I, "<u2", 65535),
        _edit(good, REC_SCAL + 2 * SC_SLIDES, "<i2", 2),
        _edit(good, REC_SCAL + 2 * SC_SLIDES, "<i2", -1),
        _edit(good, REC_SCAL + 2 * SC_ARGMAX_LAST, "<i2", 7),
        _edit(good, REC_SCAL + 2 * SC_ARGMAX_LAST, "<i2", -1),
    ]
    # the edges that are accepted, so the checks above are exactly at the limits
    ok = [_edit(good, REC_CASC + 2 * CS_POS, "<u2", 2), _edit(good, REC_CASC + 2 * CS_AGE, "<u2", 2),
          _edit(good, REC_CASC + 2 * CS_CNT_S2I, "<u2", 32766), _edit(good, REC_SCAL + 2 * SC_ARGMAX_LAST, "<i2", 6)]
    h = _handle(nb)
    h.exec(x0)
    for r in bad:
        refused(h, [6], r)
        refused(h, [1, 6], good + r)                      # one bad record refuses the whole call
    refused(h, [6, 6], good + good)                       # a slot listed twice
    refused(h, [S], good)
    refused(h, [-1], good)
    a = np.asarray([1], np.int32)
    assert L.nnsp_b200_cascade_import_streams(h.h, a.ctypes.data_as(C.c_void_p), -1, None) == ERR_ARG
    assert L.nnsp_b200_cascade_import_streams(h.h, a.ctypes.data_as(C.c_void_p), 1, None) == ERR_ARG
    for ids in ([S], [-1], [0, S]):
        b = np.zeros(rb * len(ids), np.uint8)
        a = np.asarray(ids, np.int32)
        assert L.nnsp_b200_cascade_export_streams(h.h, a.ctypes.data_as(C.c_void_p), len(a), b.ctypes.data_as(C.c_void_p)) == ERR_ARG
    assert h.exec(x1).tobytes() == want                   # nothing was recorded
    assert L.nnsp_b200_cascade_import_streams(h.h, None, 0, None) == 0
    for r in ok:
        h.import_streams([6], r)                          # accepted
    h.close()
    with pytest.raises(ValueError):
        _handle(nb).import_streams([1, 2], good)          # the binding checks the buffer length
