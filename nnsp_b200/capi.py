"""ctypes binding of the C ABI in include/nnsp_b200.h (libnnsp_b200.so, built in-tree).

Pure plumbing: no arithmetic happens in Python. The library has no CPU path, so every compute
call raises :class:`NnspError` on a machine without a usable B200 (sm_100) device.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NNSP_B200_LIB") or os.path.join(HERE, "libnnsp_b200.so")   # env override: kernel-variant experiments only

RESULT_DT = np.dtype([("trigger", "<i2"), ("outputs", "<i2", (3,))])
CASCADE_RESULT_DT = np.dtype([("stage_id", "i1"), ("pos_after", "i1"), ("detected", "<i2"),
                              ("outputs", "<i2", (3,)), ("cnt_timeout", "<u2")])


class Taps(C.Structure):
    _fields_ = [("logmel", C.c_void_p), ("feat", C.c_void_p), ("act", C.c_void_p), ("logits", C.c_void_p),
                ("hstate", C.c_void_p), ("cstate", C.c_void_p), ("post", C.c_void_p)]


class CascadeParams(C.Structure):
    _fields_ = [(n, C.c_int16) for n in (
        "thresh_prob_vad", "thresh_cnts_vad", "frs_vbufBk_s2i", "thresh_timeout_s2i", "thresh_prob_s2i",
        "thresh_cnts_s2i", "frs_vbufBk_kws", "thresh_timeout_kws", "thresh_prob_kws", "thresh_cnts_kws")]


class StreamHeader(C.Structure):
    """nnsp_b200_stream_header: the head of every stream record (Cascade.export_streams)"""
    _fields_ = [("magic", C.c_uint32), ("version", C.c_uint32), ("record_bytes", C.c_uint32), ("len_seq", C.c_int32),
                ("seq", C.c_int32 * 3), ("frs_vbufBk_kws", C.c_int16), ("frs_vbufBk_s2i", C.c_int16),
                ("model_fnv1a", C.c_uint64 * 3), ("reserved", C.c_uint64)]


STREAM_MAGIC, STREAM_VERSION = 0x5353504E, 1


class NnspError(RuntimeError):
    pass


_lib = None

# every symbol include/nnsp_b200.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = """nnsp_b200_version nnsp_b200_strerror nnsp_b200_last_error nnsp_b200_kernel_launches nnsp_b200_tc5_launches
nnsp_b200_cascade_kernel_launches nnsp_b200_model_from_net nnsp_b200_model_from_table_text nnsp_b200_model_to_table_text nnsp_b200_model_from_blob nnsp_b200_model_to_blob nnsp_b200_model_set_acc32
nnsp_b200_model_info nnsp_b200_model_free nnsp_b200_batch_create nnsp_b200_batch_reset nnsp_b200_batch_exec
nnsp_b200_batch_exec_host nnsp_b200_batch_exec_host_async nnsp_b200_batch_wait_host nnsp_b200_batch_sync nnsp_b200_batch_last_kernel_ms nnsp_b200_batch_dims
nnsp_b200_batch_stream nnsp_b200_batch_set_nn_path nnsp_b200_batch_get_nn_path nnsp_b200_batch_destroy nnsp_b200_cascade_default_params nnsp_b200_cascade_create
nnsp_b200_cascade_reset nnsp_b200_cascade_set_stream_params nnsp_b200_cascade_exec nnsp_b200_cascade_exec_host nnsp_b200_cascade_exec_host_async nnsp_b200_cascade_wait_host nnsp_b200_cascade_sync
nnsp_b200_cascade_last_kernel_ms nnsp_b200_cascade_stream nnsp_b200_cascade_set_path nnsp_b200_cascade_destroy nnsp_b200_feature_stages
nnsp_b200_table nnsp_b200_ingest_audadc nnsp_b200_device_count nnsp_b200_device_pci_bus_id nnsp_b200_dev_alloc nnsp_b200_dev_free nnsp_b200_host_alloc_pinned
nnsp_b200_host_free_pinned nnsp_b200_memcpy_h2d nnsp_b200_memcpy_d2h nnsp_b200_memset nnsp_b200_event_create
nnsp_b200_event_record nnsp_b200_event_elapsed_ms nnsp_b200_event_destroy nnsp_b200_int_peak nnsp_b200_net_eval
nnsp_b200_group_create_batch nnsp_b200_group_create_cascade nnsp_b200_group_size nnsp_b200_group_range nnsp_b200_group_reset nnsp_b200_group_set_stream_params
nnsp_b200_group_exec_host nnsp_b200_group_exec_host_async nnsp_b200_group_wait nnsp_b200_group_destroy
nnsp_b200_batch_set_host_format nnsp_b200_cascade_set_host_format nnsp_b200_wav_info nnsp_b200_wav_read_frames nnsp_b200_wav_load_streams nnsp_b200_cascade_timeline
nnsp_b200_cascade_exec_ragged nnsp_b200_cascade_exec_host_ragged_async nnsp_b200_scan_kernel_launches
nnsp_b200_cascade_reset_streams nnsp_b200_group_reset_streams
nnsp_b200_cascade_stream_state_bytes nnsp_b200_cascade_export_streams nnsp_b200_cascade_import_streams
nnsp_b200_group_stream_state_bytes nnsp_b200_group_export_streams nnsp_b200_group_import_streams""".split()


def lib():
    """Load libnnsp_b200.so (fails loudly if the CUDA extension has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NnspError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no Python or CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i16, ci, ll = C.c_void_p, C.c_int16, C.c_int, C.c_longlong
    L.nnsp_b200_version.restype = C.c_char_p
    L.nnsp_b200_strerror.restype = C.c_char_p
    L.nnsp_b200_strerror.argtypes = [ci]
    L.nnsp_b200_last_error.restype = C.c_char_p
    L.nnsp_b200_kernel_launches.restype = ll
    L.nnsp_b200_tc5_launches.restype = ll
    L.nnsp_b200_cascade_kernel_launches.restype = ll
    L.nnsp_b200_cascade_kernel_launches.argtypes = [ci]
    L.nnsp_b200_scan_kernel_launches.restype = ll
    L.nnsp_b200_scan_kernel_launches.argtypes = [ci]
    L.nnsp_b200_model_from_net.argtypes = [vp, vp, vp, ci, C.POINTER(vp)]
    L.nnsp_b200_model_from_table_text.argtypes = [C.c_char_p, C.c_size_t, ci, ci, C.POINTER(vp)]
    L.nnsp_b200_model_to_table_text.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.nnsp_b200_model_from_blob.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    L.nnsp_b200_model_to_blob.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.nnsp_b200_model_set_acc32.argtypes = [vp, ci]
    L.nnsp_b200_model_info.argtypes = [vp, C.POINTER(ci), C.POINTER(ci), vp, C.POINTER(ci)]
    L.nnsp_b200_model_free.argtypes = [vp]
    L.nnsp_b200_model_free.restype = None
    L.nnsp_b200_batch_create.argtypes = [vp, ci, ci, i16, i16, C.POINTER(vp)]
    L.nnsp_b200_batch_reset.argtypes = [vp]
    L.nnsp_b200_batch_exec.argtypes = [vp, vp, ll, ci, vp, C.POINTER(Taps)]
    L.nnsp_b200_batch_exec_host.argtypes = [vp, vp, ll, ci, vp]
    L.nnsp_b200_batch_exec_host_async.argtypes = [vp, vp, ll, ci, vp, C.POINTER(ll)]
    L.nnsp_b200_batch_wait_host.argtypes = [vp, ll]
    L.nnsp_b200_batch_sync.argtypes = [vp]
    L.nnsp_b200_batch_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float * 3)]
    L.nnsp_b200_batch_dims.argtypes = [vp] + [C.POINTER(ci)] * 4
    L.nnsp_b200_batch_stream.argtypes = [vp]
    L.nnsp_b200_batch_stream.restype = vp
    L.nnsp_b200_batch_set_nn_path.argtypes = [vp, ci]
    L.nnsp_b200_batch_get_nn_path.argtypes = [vp]
    L.nnsp_b200_batch_destroy.argtypes = [vp]
    L.nnsp_b200_batch_destroy.restype = None
    if hasattr(L, "nnsp_b200_cascade_create"):
        L.nnsp_b200_cascade_default_params.argtypes = [C.POINTER(CascadeParams)]
        L.nnsp_b200_cascade_default_params.restype = None
        L.nnsp_b200_cascade_create.argtypes = [C.POINTER(vp), C.POINTER(ci), ci, C.POINTER(CascadeParams), ci, ci, C.POINTER(vp)]
        L.nnsp_b200_cascade_reset.argtypes = [vp]
        L.nnsp_b200_cascade_set_stream_params.argtypes = [vp, ci, ci, vp]
        L.nnsp_b200_cascade_reset_streams.argtypes = [vp, vp, ci, ci]
        L.nnsp_b200_cascade_stream_state_bytes.argtypes = [vp]
        L.nnsp_b200_cascade_stream_state_bytes.restype = C.c_size_t
        L.nnsp_b200_cascade_export_streams.argtypes = [vp, vp, ci, vp]
        L.nnsp_b200_cascade_import_streams.argtypes = [vp, vp, ci, vp]
        L.nnsp_b200_cascade_exec.argtypes = [vp, vp, ll, ci, vp, C.POINTER(Taps)]
        L.nnsp_b200_cascade_exec_host.argtypes = [vp, vp, ll, ci, vp]
        L.nnsp_b200_cascade_exec_host_async.argtypes = [vp, vp, ll, ci, vp, C.POINTER(ll)]
        L.nnsp_b200_cascade_exec_ragged.argtypes = [vp, vp, ll, ci, vp, vp, C.POINTER(Taps)]
        L.nnsp_b200_cascade_exec_host_ragged_async.argtypes = [vp, vp, ll, ci, vp, vp, C.POINTER(ll)]
        L.nnsp_b200_cascade_wait_host.argtypes = [vp, ll]
        L.nnsp_b200_cascade_sync.argtypes = [vp]
        L.nnsp_b200_cascade_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float * 3)]
        L.nnsp_b200_cascade_stream.argtypes = [vp]
        L.nnsp_b200_cascade_stream.restype = vp
        L.nnsp_b200_cascade_set_path.argtypes = [vp, ci]
        L.nnsp_b200_cascade_destroy.argtypes = [vp]
        L.nnsp_b200_cascade_destroy.restype = None
    L.nnsp_b200_feature_stages.argtypes = [ci, vp, ci, vp, vp, vp, vp, vp]
    L.nnsp_b200_ingest_audadc.argtypes = [ci, vp, vp, ll, vp]
    L.nnsp_b200_table.argtypes = [C.c_char_p, C.POINTER(vp), C.POINTER(ci)]
    L.nnsp_b200_dev_alloc.argtypes = [ci, C.c_size_t, C.POINTER(vp)]
    L.nnsp_b200_dev_free.argtypes = [ci, vp]
    L.nnsp_b200_host_alloc_pinned.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.nnsp_b200_host_free_pinned.argtypes = [vp]
    L.nnsp_b200_memcpy_h2d.argtypes = [ci, vp, vp, C.c_size_t]
    L.nnsp_b200_memcpy_d2h.argtypes = [ci, vp, vp, C.c_size_t]
    L.nnsp_b200_memset.argtypes = [ci, vp, ci, C.c_size_t]
    L.nnsp_b200_event_create.argtypes = [ci, C.POINTER(vp)]
    L.nnsp_b200_event_record.argtypes = [vp, vp]
    L.nnsp_b200_event_elapsed_ms.argtypes = [vp, vp, C.POINTER(C.c_float)]
    L.nnsp_b200_event_destroy.argtypes = [vp]
    L.nnsp_b200_int_peak.argtypes = [ci, C.POINTER(C.c_double * 4)]
    L.nnsp_b200_net_eval.argtypes = [vp, ci, ci, ci] + [vp] * 7
    L.nnsp_b200_group_create_batch.argtypes = [vp, ci, C.POINTER(ci), ci, i16, i16, C.POINTER(vp)]
    L.nnsp_b200_group_create_cascade.argtypes = [C.POINTER(vp), C.POINTER(ci), ci, C.POINTER(CascadeParams), ci, C.POINTER(ci), ci, C.POINTER(vp)]
    L.nnsp_b200_group_size.argtypes = [vp]
    L.nnsp_b200_group_range.argtypes = [vp, ci, C.POINTER(ci), C.POINTER(ci), C.POINTER(ci)]
    L.nnsp_b200_group_reset.argtypes = [vp]
    L.nnsp_b200_group_set_stream_params.argtypes = [vp, ci, ci, vp]
    L.nnsp_b200_group_reset_streams.argtypes = [vp, vp, ci, ci]
    L.nnsp_b200_group_stream_state_bytes.argtypes = [vp]
    L.nnsp_b200_group_stream_state_bytes.restype = C.c_size_t
    L.nnsp_b200_group_export_streams.argtypes = [vp, vp, ci, vp]
    L.nnsp_b200_group_import_streams.argtypes = [vp, vp, ci, vp]
    L.nnsp_b200_group_exec_host.argtypes = [vp, vp, ll, ci, vp]
    L.nnsp_b200_group_exec_host_async.argtypes = [vp, vp, ll, ci, vp, C.POINTER(ll)]
    L.nnsp_b200_group_wait.argtypes = [vp, ll]
    L.nnsp_b200_group_destroy.argtypes = [vp]
    L.nnsp_b200_group_destroy.restype = None
    L.nnsp_b200_batch_set_host_format.argtypes = [vp, ci]
    L.nnsp_b200_cascade_timeline.argtypes = [vp, vp, C.POINTER(ci)]
    L.nnsp_b200_cascade_set_host_format.argtypes = [vp, ci]
    L.nnsp_b200_wav_info.argtypes = [C.c_char_p, C.POINTER(ci), C.POINTER(ci), C.POINTER(ci), C.POINTER(ll)]
    L.nnsp_b200_wav_read_frames.argtypes = [C.c_char_p, ci, ll, ci, vp, C.POINTER(ci)]
    L.nnsp_b200_wav_load_streams.argtypes = [C.POINTER(C.c_char_p), ci, ci, ll, ci, vp, ll, vp]
    _lib = L
    return L


def check(rc, what=""):
    if rc != 0:
        L = lib()
        raise NnspError("%s: %s [%s]" % (what or "nnsp_b200", L.nnsp_b200_strerror(rc).decode(),
                                         L.nnsp_b200_last_error().decode()))
