"""The reference's on-disk model format -- generated C source `evb/src/def_nn{id}_{name}.c`
(python/c_code_table_converter.py:143-347, layout python/nnsp_pack/c_weight_man.py:5-124) -- read and
written as text by libnnsp_b200 (nnsp_model_text.c), no C compiler on the load path. Host logic only."""
import hashlib
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

from common import ROOT, have_reference_tree, make_blob

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
