"""nnsp_b200 -- B200-native batched implementation of the ns-nnsp streaming inference hot path.

The product is libnnsp_b200.so (C ABI in include/nnsp_b200.h, CUDA kernels in nnsp_b200/csrc).
This package is the thin host-side binding used by the tests and bench.py.
"""
from .api import (CASCADE_RESULT_DT, FRAME, KWS, RESULT_DT, S2I, VAD, Cascade, DeviceArray, Event, Group, Model, NNSPBatch,
                  NnspError, PinnedArray, cascade_kernel_launches, scan_kernel_launches, device_count, device_pci_bus_id, feature_stages, ingest_audadc, int_peak, kernel_launches, net_eval, tc5_launches, table, wav_info, wav_load_streams)
from .synth import adversarial_windows, synth_pcm

MODEL_DIR = __import__("os").path.join(__import__("os").path.dirname(__import__("os").path.abspath(__file__)), "models")   # the shipped def_nn*.c tables as NNSPM1 containers
