"""The reference's on-disk model format -- generated C source `evb/src/def_nn{id}_{name}.c`
(python/c_code_table_converter.py:143-347, layout python/nnsp_pack/c_weight_man.py:5-124) -- read and
written as text by libnnsp_b200 (nnsp_model_text.c), no C compiler on the load path. Host logic only."""
import ctypes as C
import hashlib
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

from common import NET_LIMITS, ROOT, have_reference_tree, make_blob, net_case_blob, widen_text

REF_SRC = "/root/reference/evb/src"
FILES = {"s2i": ("def_nn0_s2i.c", 0, "s2i.nnspm"), "vad": ("def_nn1_vad.c", 1, "vad.nnspm"),
         "kws_galaxy": ("def_nn2_kws_galaxy.c", 2, "kws_galaxy.nnspm")}


def test_text_round_trip_of_the_shipped_models(nb):
    """blob -> table text -> model must give the same model (weights, Q-formats, activations, stats)."""
    nb = nb
    for name, (_, nn_id, blob) in FILES.items():
        raw = open(os.path.join(nb.MODEL_DIR, blob), "rb").read()
        m = nb.Model.from_blob(raw)
        text = m.to_table_text(name)
        assert text.startswith(b"#include <stdint.h>\n") and (b"NeuralNetClass net_%s = {" % name.encode()) in text
        m2 = nb.Model.from_table_text(text)                    # nn_id inferred from the table name
        assert m2.nn_id == nn_id and m2.to_blob() == raw
        m3 = nb.Model.from_table_text(text, acc32=True)        # the #ifdef DEF_ACC32BIT_OPT branch
        assert m3.acc32 and not m2.acc32
        m3.set_acc32(False)
        assert m3.to_blob() == raw


@pytest.mark.parametrize("sizes,types", [((240, 7, 5, 3), (0, 1, 0)), ((240, 13, 9, 2), (0, 0, 0)),
                                         ((240, 6, 10, 10, 41), (0, 1, 1, 0)), ((240, 1, 1, 2), (0, 1, 0))])
def test_text_round_trip_odd_shapes(nb, sizes, types):
    """1/2/3-row remainder blocks and odd column counts of the ARM interleave (c_weight_man.py:5-47), lstm
    layers whose width is not a multiple of 4 -- shapes the shipped models never exercise."""
    nb = nb
    nl = len(types)
    raw = make_blob(2, sizes, types, [1, 1, 0, 3][:nl - 1] + [3], [7, 5, 5, 6][:nl], [8, 15, 15, 12][:nl], [14, 13, 15, 15][:nl], seed=sum(sizes))
    m = nb.Model.from_blob(raw)
    text = m.to_table_text("kws_odd")
    m2 = nb.Model.from_table_text(text)
    assert m2.to_blob() == raw


@pytest.mark.parametrize("acc32", [False, True])
@pytest.mark.parametrize("case", NET_LIMITS, ids=[c[0] for c in NET_LIMITS])
def test_text_round_trip_at_the_model_limits(nb, case, acc32):
    """10 layers, 128 units and outputs, unaligned LSTM offsets; a last LSTM keeps its qbit_input_rec (qbit_input[nl],
    which a 10-layer table reads from qbit_bias[0])"""
    raw = net_case_blob(case, acc32)
    m = nb.Model.from_blob(raw)
    text = m.to_table_text("kws_lim")
    assert nb.Model.from_table_text(text, nn_id=case[1]).to_blob() == raw


def test_text_writer_refuses_a_last_lstm_qbit_input_rec_a_table_cannot_hold(nb):
    """with 10 layers the table has no qbit_input[10]: a last LSTM reads qbit_bias[0] there, so any other value is refused
    rather than written as a different model; with fewer layers the value is written and read back"""
    from nnsp_b200 import capi
    case = [c for c in NET_LIMITS if c[0] == "ten_layers_last_lstm"][0]
    name, nn_id, sizes, types, acts, qk, qi, qb = case[:8]
    assert qi[10] == qb[0]
    bad = make_blob(nn_id, sizes, types, list(acts), list(qk), list(qi[:10]) + [qb[0] - 1], list(qb))
    m = nb.Model.from_blob(bad)
    n = C.c_size_t()
    L = capi.lib()
    assert L.nnsp_b200_model_to_table_text(m.h, b"vad", None, 0, C.byref(n)) == -4          # NNSP_B200_ERR_UNSUPPORTED
    assert b"qbit_bias[0]" in L.nnsp_b200_last_error()
    with pytest.raises(nb.NnspError, match="qbit_bias"):
        m.to_table_text("vad")
    # 3 layers, last LSTM with qbit_input_rec 12: the 4th qi entry of the table
    raw = make_blob(1, (240, 16, 8, 2), (0, 0, 1), [1, 1, 1], [7, 5, 6], [8, 15, 15, 12], [14, 13, 14])
    text = nb.Model.from_blob(raw).to_table_text("vad")
    assert b"{8,15,15,12,}, // qbit_i" in text
    assert nb.Model.from_table_text(text).to_blob() == raw


@pytest.mark.parametrize("last_fc", [True, False])
def test_width_and_output_limits(nb, last_fc):
    """128 units in a hidden layer and 128 outputs are accepted, 129 refused with the limit named, from the container and
    from table text alike"""
    from nnsp_b200 import capi
    L = capi.lib()
    for hidden, n_out, ok in ((128, 128, True), (129, 64, False), (64, 129, False)):
        types = (0, 1, 0) if last_fc else (0, 0, 1)
        sizes = (240, hidden, 64, n_out) if last_fc else (240, 64, hidden, n_out)
        raw = make_blob(0, sizes, types, [1, 1, 3 if last_fc else 1], [7, 5, 6], [8, 15, 15], [14, 13, 15])
        h = C.c_void_p()
        rc = L.nnsp_b200_model_from_blob(raw, len(raw), C.byref(h))
        assert (rc == 0) == ok, (sizes, rc)
        if ok:
            text = nb.Model.from_blob(raw).to_table_text("s2i")
            assert nb.Model.from_table_text(text).to_blob() == raw
            L.nnsp_b200_model_free(h)
            continue
        assert rc == -4 and b"exceeds" in L.nnsp_b200_last_error() and b"128" in L.nnsp_b200_last_error(), (sizes, rc)
        # the same shape as table text: write the 128-wide model, widen one layer in the text
        small = tuple(v if i == 0 else min(v, 128) for i, v in enumerate(sizes))
        text = nb.Model.from_blob(make_blob(0, small, types, [1, 1, 3 if last_fc else 1], [7, 5, 6], [8, 15, 15], [14, 13, 15])).to_table_text("s2i")
        wide = widen_text(text, small, sizes)
        hh = C.c_void_p()
        assert L.nnsp_b200_model_from_table_text(wide, len(wide), 0, 0, C.byref(hh)) == -4, sizes
        assert b"exceeds" in L.nnsp_b200_last_error() and b"128" in L.nnsp_b200_last_error()
        # the rewrite itself is sound: applied to the 128-wide sizes it gives a table the reader takes
        ok_text = widen_text(text, small, small)
        assert L.nnsp_b200_model_from_table_text(ok_text, len(ok_text), 0, 0, C.byref(hh)) == 0
        L.nnsp_b200_model_free(hh)


def test_text_reader_rejects_malformed_tables(nb):
    nb = nb
    raw = open(os.path.join(nb.MODEL_DIR, "vad.nnspm"), "rb").read()
    text = nb.Model.from_blob(raw).to_table_text("vad")
    bad = [
        text.replace(b"const uint16_t vad_bias3[]={", b"const uint16_t vad_bias3[]={0x0001,"),       # one element too many
        text.replace(b"(int8_t*) vad_kernel_rec1", b"(int8_t*) 0"),                                    # lstm without recurrent table
        text.replace(b"{fc,lstm,fc,fc,fc,}", b"{fc,gru,fc,fc,fc,}"),                                   # layer type the reference lacks
        text.replace(b"NeuralNetClass net_vad", b"int net_vad"),                                       # no struct literal
        text.replace(b"(int8_t*) vad_kernel2,", b"(int8_t*) vad_kernel9,"),                            # undefined array
        text[: len(text) // 2],                                                                        # truncated file
    ]
    for t in bad:
        assert t != text
        with pytest.raises(nb.NnspError):
            nb.Model.from_table_text(t)
    renamed = text.replace(b"vad", b"mystery")
    with pytest.raises(nb.NnspError):
        nb.Model.from_table_text(renamed)                                                              # id cannot be inferred
    assert nb.Model.from_table_text(renamed, nn_id=1).to_blob() == raw


@pytest.mark.skipif(not have_reference_tree(), reason="needs /root/reference")
def test_reference_table_files_parse_to_the_compiled_models(nb):
    """The three shipped def_nn*.c files, read as text, equal the models obtained by COMPILING them
    (nnsp_b200/models/*.nnspm were exported from the compiled reference objects); s2i and kws ship with
    CRLF line ends and stray blank lines. The VAD file is reproduced byte for byte (modulo CRLF) by the writer."""
    nb = nb
    for name, (src, nn_id, blob) in FILES.items():
        text = open(os.path.join(REF_SRC, src), "rb").read()
        m = nb.Model.from_table_text(text)
        assert m.nn_id == nn_id
        assert m.to_blob() == open(os.path.join(nb.MODEL_DIR, blob), "rb").read()
        ours = m.to_table_text(name)
        norm = lambda b: b"\n".join(l for l in b.replace(b"\r\n", b"\n").split(b"\n") if l.strip())
        assert norm(ours) == norm(text), "writer output differs from %s beyond blank lines / line ends" % src
    vad = open(os.path.join(REF_SRC, "def_nn1_vad.c"), "rb").read()
    assert nb.Model.from_table_text(vad).to_table_text("vad") == vad.replace(b"\r\n", b"\n")


def test_emitted_text_is_valid_c_for_the_reference_headers(nb):
    """The writer's output compiles against the drop-in headers (same declarations as the reference's) and the
    linked table, read back through nnsp_b200_model_from_net, is the same model. With -DDEF_ACC32BIT_OPT only the
    layer_func addresses (tags in libnnsp_b200.so, referenced from another shared object) make it the acc32 model.
    Besides the shipped models, a synthetic stack with sigmoid layers: the ACTIVATION_TYPE enumerator is `sigmoid`."""
    nb = nb
    import ctypes as C
    tables = [(name, nn_id, open(os.path.join(nb.MODEL_DIR, blob), "rb").read()) for name, (_, nn_id, blob) in FILES.items()]
    tables.append(("two_lstm_sigmoid", 2, make_blob(2, (240, 24, 20, 12, 9, 2), (0, 1, 0, 1, 0), [2, 1, 2, 1, 3], [6, 5, 5, 5, 6],
                                                    [8, 15, 15, 15, 15], [13, 13, 15, 14, 15], seed=3)))
    with tempfile.TemporaryDirectory() as d:
        for (name, nn_id, raw), acc32 in [(t, a) for t in tables for a in (False, True)]:
            src = os.path.join(d, "def_nn%d_%s.c" % (nn_id, name))
            text = nb.Model.from_blob(raw).to_table_text(name)
            open(src, "wb").write(text)
            so = os.path.join(d, "tbl_%s_%d.so" % (name, acc32))
            r = subprocess.run(["gcc", "-shared", "-fPIC", "-w", "-I", os.path.join(ROOT, "include", "nnsp_compat"), "-I", os.path.join(ROOT, "include")]
                               + (["-DDEF_ACC32BIT_OPT"] if acc32 else [])
                               + [src, "-o", so, "-L", os.path.join(ROOT, "nnsp_b200"), "-lnnsp_b200", "-Wl,-rpath," + os.path.join(ROOT, "nnsp_b200")],
                               capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            T = C.CDLL(so)
            net = C.addressof(C.c_char.in_dll(T, "net_" + name))
            mean = C.addressof(C.c_char.in_dll(T, "feature_mean_" + name))
            stdr = C.addressof(C.c_char.in_dll(T, "feature_stdR_" + name))
            m2 = nb.Model.from_net(net, mean, stdr, nn_id)
            assert m2.acc32 == acc32, (name, acc32)
            assert m2.to_blob() == nb.Model.from_blob(raw, acc32=acc32).to_blob(), (name, acc32)
            assert (m2.to_blob() == raw) != acc32, (name, acc32)       # the acc32 flag is part of the container
