"""Models at the limits of include/nnsp_b200.h -- 10 layers, 128 units, 128 outputs -- and LSTM shapes the shipped models
never select (tests/common.py NET_LIMITS), through every network path that accepts them, against the oracle on every tap:

  batch     : both accumulator modes, 37 streams (two full 16-stream tiles and a partial one), one tapped 130-frame call and
              a second handle in untapped calls of uneven lengths; the path "automatic" resolves to, the tcgen05 layer-0
              launches (NNSP_B200_TC5 0 and 2) and which scan_kernel specialisation ran are asserted;
  net_eval  : adversarial inputs and LSTM states on every accepting path, against the oracle's NeuralNetClass_exe;
  refusals  : shapes past the limits return the named error with the limit in nnsp_b200_last_error(), launch nothing,
              and leave the device able to run a shipped model bit-exact;
  coverage  : together, the tests of this file launch all six scan_kernel specialisations.

A second LSTM whose state starts at an offset that is not a multiple of 4 (lstm_off41, lstm_off6, lstm_7_5_3, lstm_41_87)
has no IMMA or scan-split form; the dp2a kernels read its old h through an aligned copy (nnsp_net.cuh stage_h_row)."""
import ctypes as C
import os
from collections import Counter

import numpy as np
import pytest

from common import (NET_CASCADE_EDGES, NET_CASES, NET_CRAFTED, NET_LIMITS, NET_TC5_SATURATING, SCAN_KINDS, adversarial_net_inputs,
                    adversarial_states, chunks, lstm_offsets, lstm_scan_kinds, make_blob, net_case_blob, net_case_dims, scan_kind,
                    widen_text)

TAPS = ["feat", "act", "logits", "hstate", "cstate", "post"]
ORACLE_TAP = dict(feat="feat", act="act", logits="logits", hstate="h", cstate="c", post="post")
MODEL_FILE = {0: "s2i.nnspm", 1: "vad.nnspm", 2: "kws_galaxy.nnspm"}
S, T = 37, 130
CHUNKS = chunks(T, (50, 3, 1, 77))
ERR_ARG, ERR_UNSUPPORTED = -1, -4

# name -> (the path "automatic" resolves to, the paths that accept the stack, layer 0 qualifies for the tcgen05 kernel)
EXPECT = {
    "lstm_off41": ("dp2a", {"dp2a"}, False),
    "lstm_off6": ("dp2a", {"dp2a"}, False),
    "lstm_7_5_3": ("dp2a", {"dp2a"}, False),
    "lstm_41_87": ("dp2a", {"dp2a"}, False),
    "max_width": ("split", {"split", "imma", "dp2a"}, False),
    "max_width_m128": ("split", {"split", "imma", "dp2a"}, False),
    "ten_layers": ("split", {"split", "imma", "dp2a"}, True),
    "ten_layers_last_lstm": ("imma", {"imma", "dp2a"}, False),       # no scan-split form: the last layer is an LSTM
    "scan_h32_kt4": ("split", {"split", "imma", "dp2a"}, False),
    "scan_h48_kt4": ("split", {"split", "imma", "dp2a"}, False),
    "scan_h72_kt2": ("split", {"split", "imma", "dp2a"}, True),
    "tc5_rows80_m128": ("split", {"split", "imma", "dp2a"}, True),
}
LIMITS = {c[0]: c for c in NET_LIMITS}


def scan_launches(nb):
    return Counter(nb.scan_kernel_launches())


def _first_diff(a, o):
    t = int(np.nonzero((a != o).reshape(len(a), -1).any(axis=1))[0][0])
    return t, int(np.nonzero(a[t].reshape(-1) != o[t].reshape(-1))[0][0])


@pytest.fixture(scope="module")
def launched():
    """scan_kernel launches of this module, by kind"""
    return Counter()


def test_expectations_cover_net_limits():
    assert set(EXPECT) == set(LIMITS)
    for name, (auto, ok, _) in EXPECT.items():
        case = LIMITS[name]
        offs = lstm_offsets(case[2], case[3])
        assert auto in ok and "dp2a" in ok
        assert (ok == {"dp2a"}) == any(o % 4 for o in offs), name          # an unaligned state offset rules out the MMA forms


def test_scan_dispatch_reaches_every_kind():
    """the dispatch rule of launch_split_layers, restated (common.scan_kind): the LSTMs of the scan-split stacks and of the
    shipped models (VAD 28 after 28 inputs, KWS 64 after 64, S2I 72 after 72) select all six specialisations; the
    existing stacks alone select four"""
    shipped = Counter({"4,4,1": 1, "8,2,2": 1, "9,2,3": 1})
    assert (scan_kind(28, 28), scan_kind(64, 64), scan_kind(72, 72)) == ("4,4,1", "8,2,2", "9,2,3")
    old = Counter()
    for c in NET_CASES + NET_CRAFTED + NET_TC5_SATURATING + NET_CASCADE_EDGES:
        old += lstm_scan_kinds(c[2], c[3])
    assert set(old + shipped) == {"4,4,1", "8,2,2", "9,2,3", "16,1,0"}
    new = Counter()
    for name, (auto, _, _) in EXPECT.items():
        if auto == "split":
            new += lstm_scan_kinds(LIMITS[name][2], LIMITS[name][3])
    assert set(new + shipped) == set(SCAN_KINDS)


def _oracle_runs(oracle, m_or, pcm, h_stride):
    return [oracle.nnsp_run(m_or, pcm[s], h_stride=h_stride) for s in range(len(pcm))]


def _check(name, path, want, res, taps=None):
    for s, (r, tp) in enumerate(want):
        assert (r == res[s]).all(), "%s/%s: results differ on stream %d" % (name, path, s)
        if taps is None:
            continue
        for t in TAPS:
            a, o = taps[t][s], getattr(tp, ORACLE_TAP[t])
            assert a.shape == o.shape, (name, path, t, a.shape, o.shape)
            if not (a == o).all():
                f, u = _first_diff(a, o)
                raise AssertionError("%s/%s: tap %s differs on stream %d frame %d unit %d: gpu %d oracle %d" % (name, path, t, s, f, u, a[f].reshape(-1)[u], o[f].reshape(-1)[u]))


@pytest.mark.gpu
@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
@pytest.mark.parametrize("case", NET_LIMITS, ids=[c[0] for c in NET_LIMITS])
def test_batch_every_path(nb, oracle, monkeypatch, launched, case, acc32):
    name, nn_id, sizes, types = case[:4]
    auto, accept, tc5 = EXPECT[name]
    raw = net_case_blob(case, acc32)
    m = nb.Model.from_blob(raw, acc32=acc32)
    m_or = oracle.load_model(raw, acc32)
    _, h_stride, _ = net_case_dims(case)
    pcm = nb.synth_pcm(S, T, first_stream=70 + len(name))
    want = _oracle_runs(oracle, m_or, pcm, h_stride or 1)
    kinds = lstm_scan_kinds(sizes, types)
    runs = [("auto", None)] + ([("split", "0"), ("split", "2")] if tc5 else [("split", None)]) + [("imma", None), ("dp2a", None)]
    ran = set()
    for path, tc5_env in runs:
        if tc5_env is None:
            monkeypatch.delenv("NNSP_B200_TC5", raising=False)
        else:
            monkeypatch.setenv("NNSP_B200_TC5", tc5_env)
        n0 = nb.kernel_launches()
        try:
            b = nb.NNSPBatch(m, S, nn_path=path)
        except nb.NnspError as e:
            assert path not in accept and "formulation" in str(e), (name, path, str(e))
            continue
        assert path in accept or path == "auto", (name, path)
        resolved = b.nn_path
        if path == "auto":
            assert resolved == auto, (name, resolved)
            if auto == "split":
                monkeypatch.setenv("NNSP_B200_TC5", "0")             # the tcgen05 launches are counted on the forced runs
        ran.add(resolved)
        k0, t0 = scan_launches(nb), nb.tc5_launches()
        res, taps = b.exec(pcm, taps=True)
        dk = scan_launches(nb) - k0
        launched.update(dk)
        assert dk == (kinds if resolved == "split" else Counter()), (name, path, dict(dk))
        assert nb.tc5_launches() - t0 == (1 if (resolved == "split" and tc5 and tc5_env == "2") else 0), (name, path, tc5_env)
        b.close()
        _check(name, path, want, res, taps)
        # a second handle: the same frames in untapped calls of uneven lengths
        b = nb.NNSPBatch(m, S, nn_path=path)
        got, t = [], 0
        for n in CHUNKS:
            got.append(b.exec(pcm[:, t * 160:(t + n) * 160]))
            t += n
        b.close()
        _check(name, path + " untapped in %s" % CHUNKS, want, np.concatenate(got, axis=1))
        assert nb.kernel_launches() > n0
    assert ran == accept, (name, ran)


@pytest.mark.gpu
@pytest.mark.parametrize("acc32", [False, True], ids=["acc64", "acc32"])
@pytest.mark.parametrize("case", NET_LIMITS, ids=[c[0] for c in NET_LIMITS])
def test_net_eval_every_path(nb, oracle, launched, case, acc32):
    name = case[0]
    auto, accept, _ = EXPECT[name]
    raw = net_case_blob(case, acc32)
    m = nb.Model.from_blob(raw, acc32=acc32)
    m_or = oracle.load_model(raw, acc32)
    a_s, h_s, n_o = net_case_dims(case)
    rng = np.random.default_rng(len(name) + 5 * acc32)
    x = adversarial_net_inputs(rng)
    h0, c0 = adversarial_states(rng, len(x), h_s)
    want = [oracle.net_eval(m_or, x[i], h0[i], c0[i]) for i in range(len(x))]
    for path in ["auto", "split", "imma", "dp2a"]:
        if path != "auto" and path not in accept:
            with pytest.raises(nb.NnspError, match="formulation"):
                nb.net_eval(m, x, h0, c0, nn_path=path)
            continue
        k0 = scan_launches(nb)
        act, logits, h1, c1 = nb.net_eval(m, x, h0, c0, nn_path=path)
        launched.update(scan_launches(nb) - k0)
        for i, (wa, wl, wh, wc) in enumerate(want):
            assert (act[i] == wa).all() and (logits[i] == wl).all(), (name, path, i)
            assert (h1[i] == wh).all() and (c1[i] == wc).all(), (name, path, i)


def _shipped_bit_exact(nb, oracle, nn_id=1, frames=24):
    m = nb.Model.from_blob(os.path.join(nb.MODEL_DIR, MODEL_FILE[nn_id]))
    pcm = nb.synth_pcm(4, frames, first_stream=3)
    b = nb.NNSPBatch(m, 4)
    res = b.exec(pcm)
    b.close()
    m_or = oracle.model(nn_id, False)
    for s in range(4):
        r, _ = oracle.nnsp_run(m_or, pcm[s], taps=False)
        assert (r == res[s]).all(), (nn_id, s)


def _refused(nb, rc, code, *words):
    from nnsp_b200 import capi
    msg = capi.lib().nnsp_b200_last_error()
    assert rc == code, (rc, msg)
    for w in words:
        assert w in msg, (w, msg)


def _blob(nn_id, sizes, types):
    nl = len(types)
    acts = [1] * (nl - 1) + [3 if types[-1] == 0 else 1]
    return make_blob(nn_id, sizes, types, acts, [7] + [5] * (nl - 1), [8] + [15] * (nl - 1), [14] + [13] * (nl - 1))


@pytest.mark.gpu
def test_refusals_name_the_limit_and_launch_nothing(nb, oracle):
    from nnsp_b200 import capi
    L = capi.lib()
    n0 = nb.kernel_launches()
    h = C.c_void_p()
    # a layer of 129 units, and 129 outputs: the loaders refuse them
    for sizes, types in (((240, 129, 64, 48), (0, 1, 0)), ((240, 64, 64, 129), (0, 1, 0))):
        raw = _blob(0, sizes, types)
        _refused(nb, L.nnsp_b200_model_from_blob(raw, len(raw), C.byref(h)), ERR_UNSUPPORTED, b"129", b"128")
        small = tuple(v if i == 0 else min(v, 128) for i, v in enumerate(sizes))
        text = widen_text(nb.Model.from_blob(_blob(0, small, types)).to_table_text("s2i"), small, sizes)
        _refused(nb, L.nnsp_b200_model_from_table_text(text, len(text), 0, 0, C.byref(h)), ERR_UNSUPPORTED, b"129", b"128")
    # 11 layers in table text
    text = nb.Model.from_blob(_blob(1, (240,) + (8,) * 9 + (2,), (0,) * 10)).to_table_text("vad")
    text11 = text.replace(b"\n\t10, // layers", b"\n\t11, // layers")
    assert text11 != text
    _refused(nb, L.nnsp_b200_model_from_table_text(text11, len(text11), 1, 0, C.byref(h)), ERR_ARG, b"numlayers 11", b"10")
    # LSTM state of 65 + 64 = 129: the model loads, no handle takes it
    m129 = nb.Model.from_blob(_blob(2, (240, 16, 65, 64, 2), (0, 1, 1, 0)))
    shipped = {i: nb.Model.from_blob(os.path.join(nb.MODEL_DIR, MODEL_FILE[i])) for i in (0, 1)}
    b = C.c_void_p()
    _refused(nb, L.nnsp_b200_batch_create(m129.h, 4, 0, 16383, 4, C.byref(b)), ERR_UNSUPPORTED, b"129", b"128")
    arr = (C.c_void_p * 3)(shipped[0].h, shipped[1].h, m129.h)
    seq = (C.c_int * 3)(1, 2, 0)
    p = capi.CascadeParams()
    L.nnsp_b200_cascade_default_params(C.byref(p))
    _refused(nb, L.nnsp_b200_cascade_create(arr, seq, 3, C.byref(p), 4, 0, C.byref(b)), ERR_UNSUPPORTED, b"129", b"128")
    x = np.zeros((1, 240), np.int16)
    hs, cs = np.zeros((1, 129), np.int16), np.zeros((1, 129), np.int32)
    act, lg = np.zeros((1, 96), np.int16), np.zeros((1, 2), np.int32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    _refused(nb, L.nnsp_b200_net_eval(m129.h, 0, 1, 1, ptr(x), ptr(hs), ptr(cs), ptr(act), ptr(lg), ptr(hs), ptr(cs)), ERR_UNSUPPORTED, b"129", b"128")
    # within the header's limits, but the dp2a kernel cannot hold the weights: 240 -> 128, LSTM 128, eight fc 128 -> 128
    big = nb.Model.from_blob(_blob(0, (240,) + (128,) * 10, (0, 1) + (0,) * 8))
    _refused(nb, L.nnsp_b200_batch_create(big.h, 4, 0, 16383, 4, C.byref(b)), ERR_UNSUPPORTED, b"shared memory", b"227 KB")
    # a cascade trio whose three weight images do not fit one CTA
    wide = nb.Model.from_blob(_blob(2, (240, 128, 128, 128, 2), (0, 1, 0, 0)))
    s2i = nb.Model.from_blob(_blob(0, (240, 128, 96, 128), (0, 1, 0)))
    arr = (C.c_void_p * 3)(s2i.h, shipped[1].h, wide.h)
    _refused(nb, L.nnsp_b200_cascade_create(arr, seq, 3, C.byref(p), 4, 0, C.byref(b)), ERR_UNSUPPORTED, b"shared memory", b"227 KB")
    assert nb.kernel_launches() == n0
    _shipped_bit_exact(nb, oracle)


@pytest.mark.gpu
@pytest.mark.parametrize("nn_id", [0, 1, 2])
def test_shipped_scan_kinds(nb, oracle, launched, nn_id):
    """the shipped models on the scan-split path: S2I <9,2,3>, VAD <4,4,1>, KWS <8,2,2>, bit-exact"""
    m = nb.Model.from_blob(os.path.join(nb.MODEL_DIR, MODEL_FILE[nn_id]))
    pcm = nb.synth_pcm(S, 40, first_stream=11)
    b = nb.NNSPBatch(m, S, nn_path="split")
    k0 = scan_launches(nb)
    res = b.exec(pcm)
    dk = scan_launches(nb) - k0
    b.close()
    launched.update(dk)
    assert set(dk) == {{0: "9,2,3", 1: "4,4,1", 2: "8,2,2"}[nn_id]}, dict(dk)
    m_or = oracle.model(nn_id, False)
    for s in range(S):
        r, _ = oracle.nnsp_run(m_or, pcm[s], taps=False)
        assert (r == res[s]).all(), (nn_id, s)


@pytest.mark.gpu
def test_every_scan_kind_was_launched(nb, launched):
    """runs last in this module: the tests above launched all six scan_kernel specialisations"""
    from nnsp_b200.api import SCAN_KERNELS
    assert SCAN_KERNELS == SCAN_KINDS
    missing = [k for k in SCAN_KINDS if launched[k] == 0]
    assert not missing, (missing, dict(launched))
