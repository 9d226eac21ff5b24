"""The nine legacy entry points (NNSPClass_*, FeatureClass_*, NeuralNetClass_*) on the GPU, driven by an application
compiled at test time: tests/dropin_driver.c, linked to the same libnnsp_b200.so the binding loaded, with model tables
written by Model.to_table_text and compiled with and without -DDEF_ACC32BIT_OPT. Nothing here needs the reference
sources. Every comparison is exact:
  * the shipped models against the reference's own recorded outputs (golden_v1.npz, golden_nets_v1.npz);
  * synthetic layer stacks, several live instances, threads and thresholds changed mid-stream against the oracle;
  * the per-table model cache: either call order, and one NeuralNetClass refilled with another table."""
import ctypes as C
import os
import subprocess
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from common import (GOLDEN_NETS, MODEL_NAME, NET_CASCADE_EDGES, NET_CASES, NET_CRAFTED, NET_LIMITS, NET_TC5_SATURATING, ROOT, golden,
                    net_case_blob, net_case_dims, res4, sha)
from oracle.pyoracle import RESULT_DT, Taps

pytestmark = pytest.mark.gpu
G = golden()
MODEL_FILE = {0: "s2i.nnspm", 1: "vad.nnspm", 2: "kws_galaxy.nnspm"}
ACC = {False: "acc64", True: "acc32"}
SYNTH = NET_CASES + NET_CRAFTED + NET_CASCADE_EDGES + NET_TC5_SATURATING + NET_LIMITS
WAVS = ("speech", "galaxy", "galaxy_s2i")


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Table:
    """One compiled def_nn*.c table: the addresses of net_<name>, feature_mean_<name>, feature_stdR_<name>."""

    def __init__(self, lib, name, nn_id, blob, acc32):
        self.name, self.nn_id, self.blob, self.acc32 = name, nn_id, blob, acc32
        self.net = C.addressof(C.c_char.in_dll(lib, "net_" + name))
        self.mean = C.addressof(C.c_char.in_dll(lib, "feature_mean_" + name))
        self.stdR = C.addressof(C.c_char.in_dll(lib, "feature_stdR_" + name))


class Dropin:
    def __init__(self, lib, tables):
        self.lib = L = lib
        self.tables = tables
        self.keep = []                    # NeuralNetClass copies stay alive all session: no cache key is reused
        L.drv_new.restype = C.c_void_p
        L.drv_new.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.drv_free.argtypes = [C.c_void_p]
        L.drv_set_thresholds.argtypes = [C.c_void_p, C.c_int16, C.c_int16]
        L.drv_run.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 8
        L.drv_net_eval.argtypes = [C.c_void_p] * 7
        L.drv_net_exe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.drv_table_state.argtypes = [C.c_void_p] * 3
        L.drv_strides.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 3
        L.drv_feature.argtypes = [C.c_void_p] * 6
        L.drv_net_bytes.restype = C.c_longlong

    def dims(self, net):
        a, h, n = C.c_int(), C.c_int(), C.c_int()
        self.lib.drv_strides(net, C.byref(a), C.byref(h), C.byref(n))
        return a.value, h.value, n.value

    def new(self, t, net=None):
        return self.lib.drv_new(net or t.net, t.mean, t.stdR, t.nn_id)

    def run(self, inst, net, pcm, reset=0, taps=True):
        pcm = np.ascontiguousarray(pcm, np.int16)
        T = len(pcm) // 160
        res = np.zeros(T, RESULT_DT)
        tp = Taps(T, *self.dims(net)) if taps else None
        a = [_p(getattr(tp, n)) for n in tp.names()] if taps else [None] * 7
        assert self.lib.drv_run(inst, reset, _p(pcm), T, _p(res), *a) == 0
        return res, tp

    def net_eval(self, net, x, h, c):
        a_s, h_s, n_o = self.dims(net)
        x = np.ascontiguousarray(x, np.int16)
        h = np.ascontiguousarray(h, np.int16).copy()
        c = np.ascontiguousarray(c, np.int32).copy()
        act, logits, final = np.zeros(a_s, np.int16), np.zeros(n_o, np.int32), np.zeros(n_o, np.int32)
        assert self.lib.drv_net_eval(net, _p(x), _p(h), _p(c), _p(act), _p(logits), _p(final)) == 0
        return act, logits, h, c, final

    def table_state(self, net):
        h_s = self.dims(net)[1]
        h, c = np.zeros(h_s, np.int16), np.zeros(h_s, np.int32)
        self.lib.drv_table_state(net, _p(h), _p(c))
        return h, c

    def copy_struct(self, src):
        """a NeuralNetClass at a new address holding the bytes of the one at src"""
        n = int(self.lib.drv_net_bytes())
        buf = C.create_string_buffer(n)
        C.memmove(buf, src, n)
        self.keep.append(buf)
        return C.addressof(buf)


def _compile(d, nb):
    """every (model, accumulator mode) table and the driver, linked into one library next to the binding's"""
    from nnsp_b200 import capi
    inc = ["-I", os.path.join(ROOT, "include", "nnsp_compat"), "-I", os.path.join(ROOT, "include")]
    entries = []
    for acc32 in (False, True):
        for nn_id, f in MODEL_FILE.items():
            entries.append(("%s_%s" % (MODEL_NAME[nn_id], ACC[acc32]), nn_id, open(os.path.join(nb.MODEL_DIR, f), "rb").read(), acc32))
        for case in SYNTH:
            entries.append(("%s_%s" % (case[0], ACC[acc32]), case[1], net_case_blob(case, acc32), acc32))
    procs, objs = [], []
    for name, nn_id, blob, acc32 in entries:
        src, obj = os.path.join(d, "def_%s.c" % name), os.path.join(d, "def_%s.o" % name)
        open(src, "wb").write(nb.Model.from_blob(blob).to_table_text(name))
        procs.append(subprocess.Popen(["gcc", "-c", "-fPIC", "-w"] + inc + (["-DDEF_ACC32BIT_OPT"] if acc32 else []) + [src, "-o", obj],
                                      stderr=subprocess.PIPE))
        objs.append(obj)
    drv = os.path.join(d, "dropin_driver.o")
    procs.append(subprocess.Popen(["gcc", "-c", "-O1", "-fPIC", "-Wall", "-Werror"] + inc + [os.path.join(ROOT, "tests", "dropin_driver.c"), "-o", drv],
                                  stderr=subprocess.PIPE))
    for p in procs:
        err = p.communicate()[1]
        assert p.returncode == 0, err.decode()
    so = os.path.join(d, "libdropin_app.so")
    lib_dir = os.path.dirname(os.path.abspath(capi.LIB_PATH))
    r = subprocess.run(["gcc", "-shared", "-o", so, drv] + objs + [os.path.abspath(capi.LIB_PATH), "-Wl,-rpath," + lib_dir],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(so)
    return lib, {(name, acc32): Table(lib, name, nn_id, blob, acc32) for name, nn_id, blob, acc32 in entries}


@pytest.fixture(scope="module")
def D(nb, tmp_path_factory):
    nb.kernel_launches()                  # loads libnnsp_b200.so first: the driver binds to this same instance
    lib, tables = _compile(str(tmp_path_factory.mktemp("dropin")), nb)
    return Dropin(lib, tables)


def shipped(D, nn_id, acc32):
    return D.tables[("%s_%s" % (MODEL_NAME[nn_id], ACC[acc32]), acc32)]


def synth_table(D, case, acc32):
    return D.tables[("%s_%s" % (case[0], ACC[acc32]), acc32)]


def oracle_model(oracle, t):
    return oracle.load_model(t.blob, t.acc32)


def assert_same(got, want, what):
    (r_g, t_g), (r_w, t_w) = got, want
    for f in r_w.dtype.names:
        bad = np.nonzero((r_g[f] != r_w[f]).reshape(len(r_w), -1).any(axis=1))[0]
        assert len(bad) == 0, "%s: result %s differs first at frame %d" % (what, f, bad[0])
    if t_w is None:
        return
    for n in t_w.names():
        a, b = getattr(t_g, n), getattr(t_w, n)
        assert a.shape == b.shape, (what, n, a.shape, b.shape)
        bad = np.nonzero((a != b).reshape(len(b), -1).any(axis=1))[0]
        assert len(bad) == 0, "%s: tap %s differs first at frame %d" % (what, n, bad[0])


def test_tables_read_back_as_the_models_they_were_written_from(nb, D):
    """The compiled tables are the intended models: from_net gives the blob, with the acc32 layer functions exactly
    where the table was compiled with -DDEF_ACC32BIT_OPT."""
    for (name, acc32), t in D.tables.items():
        want = nb.Model.from_blob(t.blob, acc32=acc32).to_blob()
        assert nb.Model.from_net(t.net, t.mean, t.stdR, t.nn_id).to_blob() == want, name


# ---- against the reference's recorded outputs -------------------------------------------------------------------
@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
@pytest.mark.parametrize("nn_id", [0, 1, 2], ids=["s2i", "vad", "kws"])
def test_shipped_streams_match_the_recorded_reference(nb, D, nn_id, acc32):
    """NNSPClass_exec with every tap: the wav excerpts and the 12 synthetic streams, records and tap hashes."""
    t = shipped(D, nn_id, acc32)
    inst = D.new(t)
    n0 = nb.kernel_launches()
    try:
        for w in WAVS:
            key = "%s_%s_%s" % (MODEL_NAME[nn_id], ACC[acc32], w)
            res, tp = D.run(inst, t.net, G["wav_" + w], reset=1)
            assert (res4(res) == G[key + "_res"]).all(), key
            assert [sha(getattr(tp, n)) for n in tp.names()] == list(G[key + "_sha"]), key
        x = nb.synth_pcm(12, 200)
        key = "synth_%s_%s" % (MODEL_NAME[nn_id], ACC[acc32])
        for s in range(12):
            res, tp = D.run(inst, t.net, x[s], reset=1)
            assert (res4(res) == G[key + "_res"][s]).all(), (key, s)
            assert [sha(getattr(tp, n)) for n in tp.names()] == list(G[key + "_sha"][s]), (key, s)
    finally:
        D.lib.drv_free(inst)
    assert nb.kernel_launches() - n0 >= 3 * 250 + 12 * 200


def _check_net_vectors(D, net, x, h0, c0, want, key):
    """NeuralNetClass_exe on each vector: every layer through debug_layer (the int16 copy-out of layers 0..L-2), the
    int32 output of the full evaluation (every stack here ends in a linear layer), and the new state both as
    returned and as left in the table's own arrays"""
    act_w, logits_w, h1_w, c1_w = want
    for i in range(len(x)):
        act, logits, h1, c1, final = D.net_eval(net, x[i], h0[i], c0[i])
        assert (act == act_w[i]).all() and (logits == logits_w[i]).all(), (key, i)
        assert (final == logits_w[i]).all(), (key, i)
        assert (h1 == h1_w[i]).all() and (c1 == c1_w[i]).all(), (key, i)
        th, tc = D.table_state(net)
        assert (th == h1_w[i]).all() and (tc == c1_w[i]).all(), (key, i)


@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
@pytest.mark.parametrize("nn_id", [0, 1, 2], ids=["s2i", "vad", "kws"])
def test_shipped_network_vectors_match_the_recorded_reference(nb, D, nn_id, acc32):
    t = shipped(D, nn_id, acc32)
    key = "net_%s_%s" % (MODEL_NAME[nn_id], ACC[acc32])
    n0 = nb.kernel_launches()
    _check_net_vectors(D, t.net, G["net_x"], G[key + "_h0"], G[key + "_c0"],
                       [G[key + k] for k in ("_act", "_logits", "_h1", "_c1")], key)
    # one launch per debug_layer tap (k = 1..L) and one for the full evaluation
    assert nb.kernel_launches() - n0 == len(G["net_x"]) * (nb.Model.from_blob(t.blob).numlayers + 1)


@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
@pytest.mark.parametrize("case", NET_CASES + NET_CRAFTED, ids=[c[0] for c in NET_CASES + NET_CRAFTED])
def test_synthetic_network_vectors_match_the_recorded_reference(D, case, acc32):
    N = np.load(GOLDEN_NETS)
    t = synth_table(D, case, acc32)
    key = "%s_%s" % (case[0], ACC[acc32])
    h_s = net_case_dims(case)[1]
    _check_net_vectors(D, t.net, N["x"], N[key + "_h0"][:, :h_s], N[key + "_c0"][:, :h_s],
                       [N[key + k] for k in ("_act", "_logits", "_h1", "_c1")], key)


def test_front_end_windows_match_the_recorded_reference(nb, D, oracle):
    """FeatureClass_execute on the adversarial windows: the log-mel row equals the reference's, and context row 5 the
    oracle's standardisation of the same window with each shipped model's statistics."""
    wins = G["fe_windows"]
    for nn_id in (0, 1, 2):
        t = shipped(D, nn_id, False)
        m = oracle.model(nn_id, False)
        for i, w in enumerate(wins):
            logmel, ctx = np.zeros(40, np.int32), np.zeros(240, np.int16)
            D.lib.drv_feature(t.net, t.mean, t.stdR, _p(np.ascontiguousarray(w)), _p(logmel), _p(ctx))
            assert (logmel == G["fe_logmel"][i]).all(), (nn_id, i)
            # three frames from a zeroed buffer leave exactly this window in the analysis buffer
            _, tp = oracle.nnsp_run(m, w, h_stride=D.dims(t.net)[1])
            assert (tp.logmel[2] == logmel).all() and (ctx[200:] == tp.feat[2]).all(), (nn_id, i)
            assert (ctx[160:200] == 0).all()          # row 5 of a fresh FeatureClass, slid up by one


# ---- against the oracle -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
@pytest.mark.parametrize("case", SYNTH, ids=[c[0] for c in SYNTH])
def test_synthetic_stacks_whole_streams_match_oracle(nb, D, oracle, case, acc32):
    """NNSPClass_exec on layer stacks the shipped tables never have: two LSTMs (state gathered from and scattered to
    several pt_hstate arrays), no LSTM, an 81-wide state, saturating feature rows; every tap and the final state in
    the table's arrays."""
    t = synth_table(D, case, acc32)
    m = oracle_model(oracle, t)
    h_s = net_case_dims(case)[1]
    pcm = nb.synth_pcm(6, 50)
    inst = D.new(t)
    try:
        for s in (0, 2, 5):
            got = D.run(inst, t.net, pcm[s], reset=1)
            want = oracle.nnsp_run(m, pcm[s], h_stride=h_s)
            assert_same(got, want, "%s_%s stream %d" % (case[0], ACC[acc32], s))
            th, tc = D.table_state(t.net)
            assert (th == want[1].h[-1]).all() and (tc == want[1].c[-1]).all()
    finally:
        D.lib.drv_free(inst)


def test_reset_of_a_live_instance_keeps_context_row_5(nb, D, oracle):
    """NNSPClass_reset on a live instance (what the controllers do) keeps context row 5 (feature_module.c:39-42)."""
    pcm = nb.synth_pcm(1, 80, first_stream=9)[0]
    for nn_id in (1, 0):
        t = shipped(D, nn_id, False)
        m = oracle.model(nn_id, False)
        st = oracle.lib.nnsp_oracle_stream_new()
        oracle.nnsp_run(m, pcm[:40 * 160], state=st, reset=1, taps=False)
        want = oracle.nnsp_run(m, pcm[40 * 160:], state=st, reset=2)
        oracle.lib.nnsp_oracle_stream_free(st)
        inst = D.new(t)
        D.run(inst, t.net, pcm[:40 * 160], reset=1, taps=False)
        got = D.run(inst, t.net, pcm[40 * 160:], reset=2)
        D.lib.drv_free(inst)
        assert_same(got, want, "reset nn_id %d" % nn_id)


# table, new (thresh_prob, th_count): values that change the decisions of these streams (the test asserts that they
# do). The shipped S2I model never leaves intent 0 on them, so a synthetic stack with 41 outputs stands in for it.
NEW_THRESHOLDS = {"vad": ((1, False), (2000, 1)), "kws": ((2, False), (1000, 0)),
                  "s2i_post": (("lstm_wide", False), (16383, 1))}


@pytest.mark.parametrize("which", list(NEW_THRESHOLDS))
def test_thresholds_changed_through_the_init_pointers_mid_stream(nb, D, oracle, which):
    """NNSPClass_exec reads *pt_thresh_prob and *pt_th_count_trigger on every frame."""
    (key, acc32), (tp_new, tc_new) = NEW_THRESHOLDS[which]
    t = shipped(D, key, acc32) if isinstance(key, int) else D.tables[(key + "_" + ACC[acc32], acc32)]
    m = oracle_model(oracle, t)
    h_s = D.dims(t.net)[1]
    pcm = nb.synth_pcm(8, 160, first_stream=20)
    changed = 0
    inst = D.new(t)
    try:
        for s in range(8):
            st = oracle.lib.nnsp_oracle_stream_new()
            w1 = oracle.nnsp_run(m, pcm[s, :70 * 160], state=st, reset=1, h_stride=h_s)
            w2 = oracle.nnsp_run(m, pcm[s, 70 * 160:], thresh_prob=tp_new, th_count=tc_new, state=st, reset=0, h_stride=h_s)
            oracle.lib.nnsp_oracle_stream_free(st)
            unchanged, _ = oracle.nnsp_run(m, pcm[s], taps=False, h_stride=h_s)
            changed += int((unchanged[70:] != w2[0]).any())
            D.lib.drv_set_thresholds(inst, 16383, 4)
            g1 = D.run(inst, t.net, pcm[s, :70 * 160], reset=1)
            D.lib.drv_set_thresholds(inst, tp_new, tc_new)
            g2 = D.run(inst, t.net, pcm[s, 70 * 160:], reset=0)
            assert_same(g1, w1, "stream %d, first thresholds" % s)
            assert_same(g2, w2, "stream %d, new thresholds" % s)
    finally:
        D.lib.drv_free(inst)
    assert changed > 0


def test_three_instances_fed_in_turn(nb, D, oracle):
    """VAD, KWS and S2I instances live at once and take one frame each in turn; the KWS instance is reset part way.
    Each equals its own oracle run."""
    T, cut = 90, 47
    pcm = nb.synth_pcm(3, T, first_stream=30)
    ids = (1, 2, 0)
    insts = [D.new(shipped(D, i, False)) for i in ids]
    got = [(np.zeros(T, RESULT_DT), Taps(T, *D.dims(shipped(D, i, False).net))) for i in ids]
    try:
        for f in range(T):
            for k, i in enumerate(ids):
                reset = 1 if f == 0 else (2 if (i == 2 and f == cut) else 0)
                r, tp = D.run(insts[k], shipped(D, i, False).net, pcm[k, f * 160:(f + 1) * 160], reset=reset)
                got[k][0][f] = r[0]
                for n in tp.names():
                    getattr(got[k][1], n)[f] = getattr(tp, n)[0]
    finally:
        for inst in insts:
            D.lib.drv_free(inst)
    for k, i in enumerate(ids):
        m = oracle.model(i, False)
        if i == 2:
            st = oracle.lib.nnsp_oracle_stream_new()
            a = oracle.nnsp_run(m, pcm[k, :cut * 160], state=st, reset=1)
            b = oracle.nnsp_run(m, pcm[k, cut * 160:], state=st, reset=2)
            oracle.lib.nnsp_oracle_stream_free(st)
            want = (np.concatenate([a[0], b[0]]), Taps(T, *D.dims(shipped(D, i, False).net)))
            for n in want[1].names():
                setattr(want[1], n, np.concatenate([getattr(a[1], n), getattr(b[1], n)]))
        else:
            want = oracle.nnsp_run(m, pcm[k])
        assert_same(got[k], want, "instance %d (nn_id %d)" % (k, i))


def test_four_host_threads(nb, D, oracle):
    """Four threads, each with its own instance and table, call NNSPClass_exec concurrently (ctypes releases the
    GIL); each stream equals its own oracle run."""
    jobs = [(shipped(D, 0, False), 0), (shipped(D, 1, True), 1), (shipped(D, 2, False), 2),
            (synth_table(D, NET_CASES[1], False), 3)]
    pcm = nb.synth_pcm(4, 120, first_stream=40)
    start = threading.Barrier(len(jobs))

    def work(job):
        t, s = job
        inst = D.new(t)
        try:
            start.wait()
            a = D.run(inst, t.net, pcm[s, :60 * 160], reset=1)
            b = D.run(inst, t.net, pcm[s, 60 * 160:], reset=0)
        finally:
            D.lib.drv_free(inst)
        return a, b

    with ThreadPoolExecutor(len(jobs)) as ex:
        out = list(ex.map(work, jobs))
    for (t, s), (a, b) in zip(jobs, out):
        want_r, want_t = oracle.nnsp_run(oracle_model(oracle, t), pcm[s], h_stride=D.dims(t.net)[1])
        got_t = Taps(0, 1, 1, 1)
        for n in want_t.names():
            setattr(got_t, n, np.concatenate([getattr(a[1], n), getattr(b[1], n)]))
        assert_same((np.concatenate([a[0], b[0]]), got_t), (want_r, want_t), "thread on %s" % t.name)


# ---- the model cache ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
def test_model_cache_either_call_order(nb, D, acc32):
    """A NeuralNetClass first seen by NeuralNetClass_exe (entry built with nn_id -1 and zero statistics) then run by
    NNSPClass_exec, and one first seen by NNSPClass_exec then evaluated by NeuralNetClass_exe: both stay exact."""
    nn_id = 1
    t = shipped(D, nn_id, acc32)
    key = "net_%s_%s" % (MODEL_NAME[nn_id], ACC[acc32])
    want_net = [G[key + k] for k in ("_act", "_logits", "_h1", "_c1")]
    x = nb.synth_pcm(4, 200)
    skey = "synth_%s_%s" % (MODEL_NAME[nn_id], ACC[acc32])

    def stream(net):
        inst = D.new(t, net)
        try:
            for s in range(4):
                res, tp = D.run(inst, net, x[s], reset=1)
                assert (res4(res) == G[skey + "_res"][s]).all(), (skey, s)
                assert [sha(getattr(tp, n)) for n in tp.names()] == list(G[skey + "_sha"][s]), (skey, s)
        finally:
            D.lib.drv_free(inst)

    net_first = D.copy_struct(t.net)
    _check_net_vectors(D, net_first, G["net_x"], G[key + "_h0"], G[key + "_c0"], want_net, key)
    stream(net_first)
    exec_first = D.copy_struct(t.net)
    stream(exec_first)
    _check_net_vectors(D, exec_first, G["net_x"], G[key + "_h0"], G[key + "_c0"], want_net, key)


def test_one_struct_refilled_with_another_table(nb, D):
    """An application that fills one NeuralNetClass with the table it needs gets that table's network on every call:
    the cached upload is rebuilt when the struct's bytes change. Tables A and B have the same shape and different
    weights and accumulators."""
    N = np.load(GOLDEN_NETS)
    case = NET_CASES[1]                                           # two LSTMs
    h_s = net_case_dims(case)[1]
    A, B = synth_table(D, case, False), synth_table(D, case, True)
    storage = D.copy_struct(A.net)
    n = int(D.lib.drv_net_bytes())
    want = {}
    for tb in (A, B):
        key = "%s_%s" % (case[0], ACC[tb.acc32])
        want[tb.acc32] = (key, N[key + "_h0"][:, :h_s], N[key + "_c0"][:, :h_s], [N[key + k] for k in ("_act", "_logits", "_h1", "_c1")])
    # the same inputs give different outputs on A and B, so running the wrong table cannot pass
    _, h0, c0, w_a = want[False]
    assert not (D.net_eval(B.net, N["x"][0], h0[0], c0[0])[1] == w_a[1][0]).all()
    for tb in (A, B, A):
        C.memmove(storage, tb.net, n)
        key, h0, c0, w = want[tb.acc32]
        _check_net_vectors(D, storage, N["x"], h0, c0, w, key)


# ---- launches ---------------------------------------------------------------------------------------------------------
def test_launch_counts(nb, D):
    """An untapped NNSPClass_exec run of T frames launches exactly T kernels; NeuralNetClass_exe with debug_layer 0
    copies its input and launches nothing."""
    t = shipped(D, 0, False)
    pcm = nb.synth_pcm(1, 37, first_stream=3)[0]
    inst = D.new(t)
    n0 = nb.kernel_launches()
    D.run(inst, t.net, pcm, reset=1, taps=False)
    D.lib.drv_free(inst)
    assert nb.kernel_launches() - n0 == 37
    x = np.arange(240, dtype=np.int16) * 131
    out = np.zeros(240, np.int32)
    n0 = nb.kernel_launches()
    D.lib.drv_net_exe(t.net, _p(x), _p(out), 0)
    assert nb.kernel_launches() == n0
    assert (out.view(np.int16)[:240] == x).all()
