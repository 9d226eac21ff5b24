"""Host-side mirror of the reference interface, batched.

Reference (single instance, C)                      here (n_streams instances, CUDA behind the C ABI)
  NNSPClass_init / _reset / _exec                    NNSPBatch(model, n_streams, ...) / .reset() / .exec()
  nnCntrlClass_init / _reset / _exec                 Cascade(models, seq, ...)        / .reset() / .exec()
  a linked def_nn*.c table                           Model.from_blob() / Model.from_net()
Same argument meaning (thresholds, frame = 160 int16 samples, trigger / outputs[3] results) and
the same error behaviour for the legacy calls (they cannot fail); the batched calls raise
NnspError on CUDA failure -- there is no CPU fallback.
"""
import ctypes as C
import os

import numpy as np

from . import capi
from .capi import CASCADE_RESULT_DT, RESULT_DT, NnspError, check, lib

FRAME = 160
S2I, VAD, KWS = 0, 1, 2


class Model:
    def __init__(self, handle):
        self.h = handle
        L = lib()
        nid, nl, acc = C.c_int(), C.c_int(), C.c_int()
        sizes = (C.c_int16 * 11)()
        check(L.nnsp_b200_model_info(self.h, C.byref(nid), C.byref(nl), sizes, C.byref(acc)), "model_info")
        self.nn_id, self.numlayers, self.acc32 = nid.value, nl.value, bool(acc.value)
        self.size_layer = list(sizes)[: nl.value + 1]

    @classmethod
    def from_blob(cls, blob, acc32=None):
        if isinstance(blob, (str, os.PathLike)):
            with open(blob, "rb") as f:
                blob = f.read()
        h = C.c_void_p()
        buf = C.create_string_buffer(bytes(blob), len(blob))
        check(lib().nnsp_b200_model_from_blob(buf, len(blob), C.byref(h)), "model_from_blob")
        m = cls(h)
        if acc32 is not None:
            m.set_acc32(acc32)
        return m

    @classmethod
    def from_table_text(cls, text, nn_id=-1, acc32=False):
        """A model from the reference's generated table source (evb/src/def_nn{id}_{name}.c), parsed as text."""
        if isinstance(text, (str, os.PathLike)) and os.path.exists(text):
            with open(text, "rb") as f:
                text = f.read()
        if isinstance(text, str):
            text = text.encode()
        h = C.c_void_p()
        check(lib().nnsp_b200_model_from_table_text(text, len(text), nn_id, int(bool(acc32)), C.byref(h)), "model_from_table_text")
        return cls(h)

    def to_table_text(self, nn_name):
        n = C.c_size_t()
        check(lib().nnsp_b200_model_to_table_text(self.h, nn_name.encode(), None, 0, C.byref(n)), "model_to_table_text")
        buf = C.create_string_buffer(n.value + 1)
        check(lib().nnsp_b200_model_to_table_text(self.h, nn_name.encode(), buf, n.value, C.byref(n)), "model_to_table_text")
        return buf.raw[: n.value]

    @classmethod
    def from_net(cls, net_ptr, mean_ptr, stdr_ptr, nn_id):
        h = C.c_void_p()
        check(lib().nnsp_b200_model_from_net(net_ptr, mean_ptr, stdr_ptr, nn_id, C.byref(h)), "model_from_net")
        return cls(h)

    def set_acc32(self, acc32):
        check(lib().nnsp_b200_model_set_acc32(self.h, int(bool(acc32))), "model_set_acc32")
        self.acc32 = bool(acc32)

    def to_blob(self):
        n = C.c_size_t()
        check(lib().nnsp_b200_model_to_blob(self.h, None, 0, C.byref(n)), "model_to_blob")
        buf = C.create_string_buffer(n.value)
        check(lib().nnsp_b200_model_to_blob(self.h, buf, n.value, C.byref(n)), "model_to_blob")
        return buf.raw[: n.value]

    def __del__(self):
        try:
            if self.h:
                lib().nnsp_b200_model_free(self.h)
                self.h = None
        except Exception:
            pass


class DeviceArray:
    """A dense array in HBM owned by the library's allocator (cudaMalloc)."""

    def __init__(self, shape, dtype, device=0, zero=True):
        self.shape, self.dtype, self.device = tuple(shape), np.dtype(dtype), device
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = C.c_void_p()
        check(lib().nnsp_b200_dev_alloc(device, max(self.nbytes, 16), C.byref(self.ptr)), "dev_alloc")
        if zero:
            check(lib().nnsp_b200_memset(device, self.ptr, 0, max(self.nbytes, 16)), "memset")

    @classmethod
    def from_host(cls, a, device=0):
        a = np.ascontiguousarray(a)
        d = cls(a.shape, a.dtype, device, zero=False)
        check(lib().nnsp_b200_memcpy_h2d(device, d.ptr, a.ctypes.data_as(C.c_void_p), a.nbytes), "h2d")
        return d

    def to_host(self):
        out = np.empty(self.shape, self.dtype)
        check(lib().nnsp_b200_memcpy_d2h(self.device, out.ctypes.data_as(C.c_void_p), self.ptr, self.nbytes), "d2h")
        return out

    def free(self):
        if self.ptr:
            lib().nnsp_b200_dev_free(self.device, self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedArray:
    """Page-locked host array (cudaMallocHost) exposed as numpy."""

    def __init__(self, shape, dtype):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = C.c_void_p()
        check(lib().nnsp_b200_host_alloc_pinned(max(self.nbytes, 16), C.byref(self.ptr)), "host_alloc_pinned")
        buf = (C.c_char * self.nbytes).from_address(self.ptr.value)
        self.array = np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            lib().nnsp_b200_host_free_pinned(self.ptr)
            self.ptr = C.c_void_p()


def _make_taps(S, T, act_stride, h_stride, n_out, device):
    arrs = dict(
        logmel=DeviceArray((S, T, 40), np.int32, device), feat=DeviceArray((S, T, 40), np.int16, device),
        act=DeviceArray((S, T, max(act_stride, 1)), np.int16, device), logits=DeviceArray((S, T, max(n_out, 1)), np.int32, device),
        hstate=DeviceArray((S, T, max(h_stride, 1)), np.int16, device), cstate=DeviceArray((S, T, max(h_stride, 1)), np.int32, device),
        post=DeviceArray((S, T, 16), np.int16, device))
    t = capi.Taps(**{k: v.ptr for k, v in arrs.items()})
    return t, arrs


class NNSPBatch:
    """n_streams independent NNSPClass instances of one model on one GPU."""

    NN_PATH = {"auto": 0, "dp2a": 1, "imma": 2, "split": 3}

    def __init__(self, model, n_streams, device=0, thresh_prob=16383, th_count=4, nn_path="auto"):
        self.model, self.S, self.device = model, int(n_streams), device
        self.h = C.c_void_p()
        check(lib().nnsp_b200_batch_create(model.h, self.S, device, thresh_prob, th_count, C.byref(self.h)), "batch_create")
        if nn_path != "auto":
            check(lib().nnsp_b200_batch_set_nn_path(self.h, self.NN_PATH[nn_path]), "batch_set_nn_path")
        a, hs, no = C.c_int(), C.c_int(), C.c_int()
        check(lib().nnsp_b200_batch_dims(self.h, None, C.byref(a), C.byref(hs), C.byref(no)), "batch_dims")
        self.act_stride, self.h_stride, self.n_out = a.value, hs.value, no.value

    @property
    def nn_path(self):
        """'dp2a' / 'imma' / 'split': the network path the next call takes."""
        return {v: k for k, v in self.NN_PATH.items()}[lib().nnsp_b200_batch_get_nn_path(self.h)]

    def set_nn_path(self, nn_path):
        check(lib().nnsp_b200_batch_set_nn_path(self.h, self.NN_PATH[nn_path]), "batch_set_nn_path")

    def reset(self):
        check(lib().nnsp_b200_batch_reset(self.h), "batch_reset")

    def sync(self):
        check(lib().nnsp_b200_batch_sync(self.h), "batch_sync")

    def exec_device(self, pcm_dev, stride, n_frames, results_dev=None, taps=None):
        """Asynchronous; pcm_dev / results_dev are DeviceArray (or raw pointers)."""
        p = pcm_dev.ptr if isinstance(pcm_dev, DeviceArray) else pcm_dev
        r = results_dev.ptr if isinstance(results_dev, DeviceArray) else results_dev
        check(lib().nnsp_b200_batch_exec(self.h, p, stride, n_frames, r, C.byref(taps) if taps is not None else None), "batch_exec")

    def exec(self, pcm, taps=False):
        """pcm: int16 [S, T*160] numpy. Returns results [S, T] (and a dict of tap arrays)."""
        pcm = np.ascontiguousarray(pcm, np.int16)
        assert pcm.ndim == 2 and pcm.shape[0] == self.S and pcm.shape[1] % FRAME == 0
        T = pcm.shape[1] // FRAME
        d_pcm = DeviceArray.from_host(pcm, self.device)
        d_res = DeviceArray((self.S, T), RESULT_DT, self.device)
        tp, arrs = (None, None)
        if taps:
            tp, arrs = _make_taps(self.S, T, self.act_stride, self.h_stride, self.n_out, self.device)
        self.exec_device(d_pcm, pcm.shape[1], T, d_res, tp)
        self.sync()
        res = d_res.to_host()
        out = {k: v.to_host() for k, v in arrs.items()} if taps else None
        d_pcm.free(); d_res.free()
        if arrs:
            for v in arrs.values():
                v.free()
        return (res, out) if taps else res

    HOST_FORMAT = {"pcm16": 0, "audadc": 1}

    def set_host_format(self, fmt):
        """'pcm16' (default) or 'audadc': the host-buffer calls then take uint32 raw AUDADC words, conditioned on the device"""
        check(lib().nnsp_b200_batch_set_host_format(self.h, self.HOST_FORMAT[fmt]), "batch_set_host_format")

    def exec_host(self, pcm, results=None):
        """End-to-end call with host buffers (H2D + kernels + D2H inside)."""
        assert pcm.dtype in (np.int16, np.uint32) and pcm.flags.c_contiguous and pcm.shape[0] == self.S
        T = pcm.shape[1] // FRAME
        if results is None:
            results = np.empty((self.S, T), RESULT_DT)
        check(lib().nnsp_b200_batch_exec_host(self.h, pcm.ctypes.data_as(C.c_void_p), pcm.shape[1], T,
                                              results.ctypes.data_as(C.c_void_p)), "batch_exec_host")
        return results

    def exec_host_async(self, pcm, results):
        """exec_host without the final wait: returns a ticket for wait_host. `pcm` and `results` (pinned) must stay
        untouched until then."""
        assert pcm.dtype == np.int16 and pcm.flags.c_contiguous and pcm.shape[0] == self.S
        T = pcm.shape[1] // FRAME
        assert results is None or (results.dtype == RESULT_DT and results.flags.c_contiguous and results.shape == (self.S, T))
        ticket = C.c_longlong(0)
        check(lib().nnsp_b200_batch_exec_host_async(self.h, pcm.ctypes.data_as(C.c_void_p), pcm.shape[1], T,
                                                    results.ctypes.data_as(C.c_void_p) if results is not None else None,
                                                    C.byref(ticket)), "batch_exec_host_async")
        return ticket.value

    def wait_host(self, ticket):
        check(lib().nnsp_b200_batch_wait_host(self.h, ticket), "batch_wait_host")

    def last_kernel_ms(self):
        ms = (C.c_float * 3)()
        check(lib().nnsp_b200_batch_last_kernel_ms(self.h, C.byref(ms)), "last_kernel_ms")
        return list(ms)

    @property
    def stream(self):
        return lib().nnsp_b200_batch_stream(self.h)

    def close(self):
        if self.h:
            lib().nnsp_b200_batch_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Cascade:
    """n_streams independent nnCntrlClass controllers (VAD -> KWS -> S2I by default)."""

    def __init__(self, models, n_streams, seq=(VAD, KWS, S2I), params=None, device=0):
        L = lib()
        self.models, self.S, self.device = models, int(n_streams), device
        arr = (C.c_void_p * 3)(*[m.h if m is not None else None for m in models])
        seq_a = (C.c_int * len(seq))(*seq)
        p = capi.CascadeParams()
        L.nnsp_b200_cascade_default_params(C.byref(p))
        if params:
            for k, v in params.items():
                setattr(p, k, v)
        self.params = p
        self._counts_in_flight = {}          # ticket -> host counts of a ragged host call, kept alive until it completes
        self.h = C.c_void_p()
        check(L.nnsp_b200_cascade_create(arr, seq_a, len(seq), C.byref(p), self.S, device, C.byref(self.h)), "cascade_create")

    PATH = {"auto": 0, "sequential": 1, "sorted": 2}

    def set_path(self, path):
        check(lib().nnsp_b200_cascade_set_path(self.h, self.PATH[path]), "cascade_set_path")

    def params_array(self):
        return np.array([getattr(self.params, n) for n, _ in capi.CascadeParams._fields_], np.int16)

    def reset(self):
        check(lib().nnsp_b200_cascade_reset(self.h), "cascade_reset")

    def reset_streams(self, streams, fresh=False):
        """Reset the listed streams before the next call of any kind, without waiting for the device: nnCntrlClass_reset of
        their controllers (stage position and context row 5 of every instance kept), or with fresh=True the state a new
        handle starts from. Per-stream parameters are kept either way."""
        s = np.ascontiguousarray(streams, np.int32).ravel()
        check(lib().nnsp_b200_cascade_reset_streams(self.h, s.ctypes.data_as(C.c_void_p), len(s), 1 if fresh else 0),
              "cascade_reset_streams")

    def set_stream_params(self, first_stream, params):
        """params: [n][10] int16, rows in the field order of ParamCntrlClass (what params_array() returns for the handle)"""
        p = np.ascontiguousarray(params, np.int16).reshape(-1, len(capi.CascadeParams._fields_))
        check(lib().nnsp_b200_cascade_set_stream_params(self.h, int(first_stream), len(p), p.ctypes.data_as(C.c_void_p)), "cascade_set_stream_params")

    def sync(self):
        check(lib().nnsp_b200_cascade_sync(self.h), "cascade_sync")

    def exec_device(self, pcm_dev, stride, n_frames, results_dev=None, taps=None):
        p = pcm_dev.ptr if isinstance(pcm_dev, DeviceArray) else pcm_dev
        r = results_dev.ptr if isinstance(results_dev, DeviceArray) else results_dev
        check(lib().nnsp_b200_cascade_exec(self.h, p, stride, n_frames, r, C.byref(taps) if taps is not None else None), "cascade_exec")

    def exec(self, pcm, taps=False):
        pcm = np.ascontiguousarray(pcm, np.int16)
        T = pcm.shape[1] // FRAME
        d_pcm = DeviceArray.from_host(pcm, self.device)
        d_res = DeviceArray((self.S, T), CASCADE_RESULT_DT, self.device)
        tp, arrs = (None, None)
        if taps:
            tp, arrs = _make_taps(self.S, T, 1, 128, 1, self.device)
        self.exec_device(d_pcm, pcm.shape[1], T, d_res, tp)
        self.sync()
        res = d_res.to_host()
        out = {k: v.to_host() for k, v in arrs.items()} if taps else None
        d_pcm.free(); d_res.free()
        if arrs:
            for v in arrs.values():
                v.free()
        return (res, out) if taps else res

    def exec_ragged_device(self, pcm_dev, stride, max_frames, n_frames_dev, results_dev=None, taps=None):
        """Asynchronous ragged call on device buffers: stream s advances by n_frames_dev[s] (int32, on the device) frames"""
        p = pcm_dev.ptr if isinstance(pcm_dev, DeviceArray) else pcm_dev
        n = n_frames_dev.ptr if isinstance(n_frames_dev, DeviceArray) else n_frames_dev
        r = results_dev.ptr if isinstance(results_dev, DeviceArray) else results_dev
        check(lib().nnsp_b200_cascade_exec_ragged(self.h, p, stride, max_frames, n, r, C.byref(taps) if taps is not None else None),
              "cascade_exec_ragged")

    def exec_ragged(self, pcm, n_frames, taps=False):
        """pcm: int16 [S, T*160]; stream s advances by n_frames[s] (0..T) of its frames, as if nnCntrlClass_exec ran n_frames[s]
        times on it. Records (and tap rows) of frames t >= n_frames[s] are "no frame": stage_id -1, every other field 0."""
        pcm = np.ascontiguousarray(pcm, np.int16)
        T = pcm.shape[1] // FRAME
        counts = np.ascontiguousarray(n_frames, np.int32)
        assert counts.shape == (self.S,)
        d_pcm = DeviceArray.from_host(pcm, self.device)
        d_cnt = DeviceArray.from_host(counts, self.device)
        d_res = DeviceArray((self.S, T), CASCADE_RESULT_DT, self.device)
        tp, arrs = (None, None)
        if taps:
            tp, arrs = _make_taps(self.S, T, 1, 128, 1, self.device)
        self.exec_ragged_device(d_pcm, pcm.shape[1], T, d_cnt, d_res, tp)
        self.sync()
        res = d_res.to_host()
        out = {k: v.to_host() for k, v in arrs.items()} if taps else None
        d_pcm.free(); d_cnt.free(); d_res.free()
        if arrs:
            for v in arrs.values():
                v.free()
        return (res, out) if taps else res

    def set_host_format(self, fmt):
        check(lib().nnsp_b200_cascade_set_host_format(self.h, NNSPBatch.HOST_FORMAT[fmt]), "cascade_set_host_format")

    def exec_host(self, pcm, results=None):
        T = pcm.shape[1] // FRAME
        if results is None:
            results = np.empty((self.S, T), CASCADE_RESULT_DT)
        check(lib().nnsp_b200_cascade_exec_host(self.h, pcm.ctypes.data_as(C.c_void_p), pcm.shape[1], T,
                                                results.ctypes.data_as(C.c_void_p)), "cascade_exec_host")
        return results

    def exec_host_async(self, pcm, results):
        """exec_host without the final wait (pinned `pcm` / `results` untouched until wait_host(ticket))."""
        assert pcm.dtype == np.int16 and pcm.flags.c_contiguous and pcm.shape[0] == self.S
        T = pcm.shape[1] // FRAME
        assert results.dtype == CASCADE_RESULT_DT and results.flags.c_contiguous and results.shape == (self.S, T)
        ticket = C.c_longlong(0)
        check(lib().nnsp_b200_cascade_exec_host_async(self.h, pcm.ctypes.data_as(C.c_void_p), pcm.shape[1], T,
                                                      results.ctypes.data_as(C.c_void_p), C.byref(ticket)), "cascade_exec_host_async")
        return ticket.value

    def exec_host_ragged_async(self, pcm, n_frames, results):
        """exec_host_async with a frame count per stream (0..T): `pcm` (int16, or uint32 AUDADC words after
        set_host_format('audadc')) and `results` (pinned) must stay untouched until wait_host(ticket). Counts outside
        0..T raise NnspError and queue nothing."""
        assert pcm.dtype in (np.int16, np.uint32) and pcm.flags.c_contiguous and pcm.shape[0] == self.S
        T = pcm.shape[1] // FRAME
        assert results.dtype == CASCADE_RESULT_DT and results.flags.c_contiguous and results.shape == (self.S, T)
        counts = np.ascontiguousarray(n_frames, np.int32)
        assert counts.shape == (self.S,)
        ticket = C.c_longlong(0)
        check(lib().nnsp_b200_cascade_exec_host_ragged_async(self.h, pcm.ctypes.data_as(C.c_void_p), pcm.shape[1], T,
                                                             counts.ctypes.data_as(C.c_void_p), results.ctypes.data_as(C.c_void_p),
                                                             C.byref(ticket)), "cascade_exec_host_ragged_async")
        self._counts_in_flight[ticket.value] = counts
        return ticket.value

    def wait_host(self, ticket):
        check(lib().nnsp_b200_cascade_wait_host(self.h, ticket), "cascade_wait_host")
        for t in [t for t in self._counts_in_flight if t <= ticket]:      # calls complete in ticket order
            del self._counts_in_flight[t]

    def last_kernel_ms(self):
        ms = (C.c_float * 3)()
        check(lib().nnsp_b200_cascade_last_kernel_ms(self.h, C.byref(ms)), "last_kernel_ms")
        return list(ms)

    def timeline(self):
        """[[front start, front done, chain start, chain done], ...] in ms for the last <= 8 device-buffer calls"""
        ms = np.zeros((8, 4), np.float32)
        n = C.c_int()
        check(lib().nnsp_b200_cascade_timeline(self.h, ms.ctypes.data_as(C.c_void_p), C.byref(n)), "cascade_timeline")
        return ms[: n.value].tolist()

    @property
    def stream(self):
        return lib().nnsp_b200_cascade_stream(self.h)

    def close(self):
        if self.h:
            lib().nnsp_b200_cascade_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Group:
    """Several GPUs of one box behind one handle (nnsp_b200_group_*): streams block-partitioned over `devices`, one host
    thread per device inside the library, host buffers in and out. models: one Model (batched NNSPClass) or a list of
    three indexed by NNSP id (cascade)."""

    def __init__(self, models, n_streams, devices, seq=(VAD, KWS, S2I), params=None, thresh_prob=16383, th_count=4):
        L = lib()
        self.S, self.devices = int(n_streams), list(devices)
        dev = (C.c_int * len(self.devices))(*self.devices)
        self.h = C.c_void_p()
        self.is_cascade = isinstance(models, (list, tuple))
        self.models = models
        if self.is_cascade:
            arr = (C.c_void_p * 3)(*[m.h if m is not None else None for m in models])
            seq_a = (C.c_int * len(seq))(*seq)
            p = capi.CascadeParams()
            L.nnsp_b200_cascade_default_params(C.byref(p))
            for k, v in (params or {}).items():
                setattr(p, k, v)
            check(L.nnsp_b200_group_create_cascade(arr, seq_a, len(seq), C.byref(p), self.S, dev, len(self.devices), C.byref(self.h)), "group_create_cascade")
        else:
            check(L.nnsp_b200_group_create_batch(models.h, self.S, dev, len(self.devices), thresh_prob, th_count, C.byref(self.h)), "group_create_batch")
        self.result_dt = CASCADE_RESULT_DT if self.is_cascade else RESULT_DT

    def ranges(self):
        out = []
        for k in range(lib().nnsp_b200_group_size(self.h)):
            d, f, n = C.c_int(), C.c_int(), C.c_int()
            check(lib().nnsp_b200_group_range(self.h, k, C.byref(d), C.byref(f), C.byref(n)), "group_range")
            out.append((d.value, f.value, n.value))
        return out

    def reset(self):
        check(lib().nnsp_b200_group_reset(self.h), "group_reset")

    def reset_streams(self, streams, fresh=False):
        """cascade groups: Cascade.reset_streams in the group's stream numbering, queued in order with the group's calls"""
        s = np.ascontiguousarray(streams, np.int32).ravel()
        check(lib().nnsp_b200_group_reset_streams(self.h, s.ctypes.data_as(C.c_void_p), len(s), 1 if fresh else 0),
              "group_reset_streams")

    def set_stream_params(self, first_stream, params):
        """cascade groups: params [n][10] int16 in the field order of ParamCntrlClass, global stream numbering"""
        p = np.ascontiguousarray(params, np.int16).reshape(-1, len(capi.CascadeParams._fields_))
        check(lib().nnsp_b200_group_set_stream_params(self.h, int(first_stream), len(p), p.ctypes.data_as(C.c_void_p)), "group_set_stream_params")

    def exec_host(self, pcm, results=None):
        assert pcm.dtype == np.int16 and pcm.flags.c_contiguous and pcm.shape[0] == self.S
        T = pcm.shape[1] // FRAME
        if results is None:
            results = np.empty((self.S, T), self.result_dt)
        check(lib().nnsp_b200_group_exec_host(self.h, pcm.ctypes.data_as(C.c_void_p), pcm.shape[1], T,
                                              results.ctypes.data_as(C.c_void_p)), "group_exec_host")
        return results

    def exec_host_async(self, pcm, results):
        assert pcm.dtype == np.int16 and pcm.flags.c_contiguous and pcm.shape[0] == self.S
        T = pcm.shape[1] // FRAME
        assert results.dtype == self.result_dt and results.flags.c_contiguous and results.shape == (self.S, T)
        t = C.c_longlong(0)
        check(lib().nnsp_b200_group_exec_host_async(self.h, pcm.ctypes.data_as(C.c_void_p), pcm.shape[1], T,
                                                    results.ctypes.data_as(C.c_void_p), C.byref(t)), "group_exec_host_async")
        return t.value

    def wait(self, ticket):
        check(lib().nnsp_b200_group_wait(self.h, ticket), "group_wait")

    def close(self):
        if self.h:
            lib().nnsp_b200_group_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def feature_stages(windows, device=0):
    """windows: int16 [n, 480]. Every intermediate of the front end, computed on the GPU."""
    w = np.ascontiguousarray(windows, np.int16)
    n = w.shape[0]
    out = dict(fft_in=np.zeros((n, 512), np.int32), spec=np.zeros((n, 514), np.int32), pspec=np.zeros((n, 257), np.int32),
               mel=np.zeros((n, 40), np.int32), logmel=np.zeros((n, 40), np.int32))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    check(lib().nnsp_b200_feature_stages(device, p(w), n, p(out["fft_in"]), p(out["spec"]), p(out["pspec"]),
                                         p(out["mel"]), p(out["logmel"])), "feature_stages")
    return out


def ingest_audadc(raw, device=0):
    """raw: uint32 [..., n*160] AUDADC words -> conditioned int16 PCM of the same shape (main_nnsp.cc:58-65), on the GPU."""
    raw = np.ascontiguousarray(raw, np.uint32)
    assert raw.size % FRAME == 0
    d_raw = DeviceArray.from_host(raw, device)
    d_pcm = DeviceArray(raw.shape, np.int16, device, zero=False)
    check(lib().nnsp_b200_ingest_audadc(device, d_raw.ptr, d_pcm.ptr, raw.size // FRAME, None), "ingest_audadc")
    out = d_pcm.to_host()
    d_raw.free(); d_pcm.free()
    return out


def net_eval(model, x, h0=None, c0=None, nn_path="auto", device=0):
    """NeuralNetClass_exe on explicit inputs: x int16 [n, 240], h0 int16 / c0 int32 [n, h_stride] (None = zeros).
    Returns (act [n, act_stride], logits [n, n_out], h1, c1) computed by the CUDA network kernels of `nn_path`."""
    x = np.ascontiguousarray(x, np.int16)
    n = x.shape[0]
    assert x.shape == (n, 240)
    sz = model.size_layer
    b = NNSPBatch(model, 1, device)                    # only for the strides the engine reports
    a_s, h_s, n_o = b.act_stride, b.h_stride, b.n_out
    b.close()
    hs = max(h_s, 1)
    h0 = np.zeros((n, hs), np.int16) if h0 is None else np.ascontiguousarray(h0, np.int16)
    c0 = np.zeros((n, hs), np.int32) if c0 is None else np.ascontiguousarray(c0, np.int32)
    assert h0.shape == (n, hs) and c0.shape == (n, hs), (h0.shape, c0.shape, hs, sz)
    act = np.zeros((n, max(a_s, 1)), np.int16)
    logits = np.zeros((n, n_o), np.int32)
    h1, c1 = np.zeros((n, hs), np.int16), np.zeros((n, hs), np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    check(lib().nnsp_b200_net_eval(model.h, device, NNSPBatch.NN_PATH[nn_path], n, p(x), p(h0), p(c0), p(act), p(logits),
                                   p(h1), p(c1)), "net_eval")
    return act[:, :a_s], logits, h1[:, :h_s], c1[:, :h_s]


def wav_info(path):
    """(sample_rate, channels, bits, samples per channel) of a RIFF/WAVE file"""
    r, c, b, n = C.c_int(), C.c_int(), C.c_int(), C.c_longlong()
    check(lib().nnsp_b200_wav_info(os.fsencode(path), C.byref(r), C.byref(c), C.byref(b), C.byref(n)), "wav_info")
    return r.value, c.value, b.value, n.value


def wav_load_streams(paths, n_frames, channel=0, first_frame=0):
    """int16 [len(paths), n_frames * 160]: stream s = frames first_frame.. of paths[s] (16 kHz, 16-bit PCM), zero padded;
    also returns the number of frames that held file samples, per stream"""
    n = len(paths)
    arr = (C.c_char_p * n)(*[os.fsencode(p) for p in paths])
    pcm = np.zeros((n, n_frames * FRAME), np.int16)
    got = np.zeros(n, np.int32)
    check(lib().nnsp_b200_wav_load_streams(arr, n, channel, first_frame, n_frames, pcm.ctypes.data_as(C.c_void_p),
                                           n_frames * FRAME, got.ctypes.data_as(C.c_void_p)), "wav_load_streams")
    return pcm, got


def table(name):
    p, eb = C.c_void_p(), C.c_int()
    n = lib().nnsp_b200_table(name.encode(), C.byref(p), C.byref(eb))
    if n < 0:
        raise NnspError("unknown table %r" % name)
    ct = C.c_int16 if eb.value == 2 else C.c_int32
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), (n,)).copy()


class Event:
    """CUDA event recorded on an engine handle's stream (nnsp_b200_event_*)."""

    def __init__(self, device=0):
        self.ptr = C.c_void_p()
        check(lib().nnsp_b200_event_create(device, C.byref(self.ptr)), "event_create")

    def record(self, stream):
        check(lib().nnsp_b200_event_record(self.ptr, stream), "event_record")

    def elapsed_ms_to(self, stop):
        ms = C.c_float()
        check(lib().nnsp_b200_event_elapsed_ms(self.ptr, stop.ptr, C.byref(ms)), "event_elapsed_ms")
        return ms.value


def device_pci_bus_id(device=0):
    """PCI bus id of CUDA device `device` (how NVML / nvidia-smi address the same GPU)."""
    buf = C.create_string_buffer(32)
    L = lib()
    L.nnsp_b200_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_int]
    check(L.nnsp_b200_device_pci_bus_id(device, buf, 32), "device_pci_bus_id")
    return buf.value.decode()


def int_peak(device=0):
    """dict of self-measured integer-pipe peaks (giga lane-instructions/s): imad, mixed, imad_wide, idp2a."""
    g = (C.c_double * 4)()
    check(lib().nnsp_b200_int_peak(device, C.byref(g)), "int_peak")
    return dict(imad=g[0], mixed=g[1], imad_wide=g[2], idp2a=g[3])


def device_count():
    return lib().nnsp_b200_device_count()


def kernel_launches():
    return lib().nnsp_b200_kernel_launches()


def tc5_launches():
    return lib().nnsp_b200_tc5_launches()


CASCADE_KERNELS = ("narrow", "wide", "replay")


def cascade_kernel_launches():
    """launches of the cascade's per-stream network kernels so far: {"narrow": cascade_kernel<CsNarrow>, "wide":
    cascade_kernel<CsWide>, "replay": cascade_replay_kernel}"""
    return {k: lib().nnsp_b200_cascade_kernel_launches(i) for i, k in enumerate(CASCADE_KERNELS)}


SCAN_KERNELS = ("4,4,1", "4,4,0", "8,2,2", "9,2,3", "9,2,0", "16,1,0")


def scan_kernel_launches():
    """launches of the split path's LSTM scan kernel so far, by specialisation scan_kernel<NT, MINB, KT>: {"4,4,1": n, ...}
    in dispatch order (KT 0: k-step counts read at run time)"""
    return {k: lib().nnsp_b200_scan_kernel_launches(i) for i, k in enumerate(SCAN_KERNELS)}
