"""Shared helpers for the parity tests."""
import hashlib
import os
import re

import struct

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "golden_v1.npz")
GOLDEN_NETS = os.path.join(ROOT, "tests", "golden", "golden_nets_v1.npz")
MODEL_NAME = {0: "s2i", 1: "vad", 2: "kws"}
TAP_NAMES = ["logmel", "feat", "act", "logits", "h", "c", "post"]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def golden():
    return np.load(GOLDEN)


def res4(res):
    """structured result array -> int16 [T, 4] (trigger, outputs[3])"""
    return res.view(np.int16).reshape(len(res), 4)


def have_reference_tree():
    return os.path.isdir("/root/reference/ns-nnsp/src")


def make_blob(nn_id, sizes, types, acts, qk, qi, qb, seed=0, fill=None):
    """NNSPM1 container (DESIGN.md) with random table-layout weights: any byte string is a valid table.
    qi: qbit_input of each layer, and optionally one more entry: qbit_input[nl], the qbit_input_rec of a last LSTM layer
    (0 when absent, as in a table whose initialiser stops at nl). fill: every kernel byte gets this int8 value instead
    (crafted extremes: -128, 127)."""
    rng = np.random.default_rng(seed)
    nl = len(types)
    hdr = b"NNSPM1\0\0" + struct.pack("<ii", nn_id, nl)
    sl = list(sizes) + [0] * (11 - len(sizes))
    hdr += struct.pack("<11h", *sl) + b"\0\0"
    hdr += rng.integers(-200000, 200000, 40, dtype=np.int32).tobytes() + rng.integers(1, 40000, 40, dtype=np.int32).tobytes()
    recs, body = b"", b""
    for i in range(10):
        if i < nl:
            rows, cols = sizes[i + 1], sizes[i]
            nr = 4 * rows if types[i] == 1 else rows
            kb, rb, bc = nr * cols, (nr * rows if types[i] == 1 else 0), nr
            qin = qi[i + 1] if i + 1 < len(qi) else 0
            recs += struct.pack("<10i", types[i], acts[i], qk[i], qi[i], qb[i], 0, kb, rb, bc, qin)
            for n in (kb, rb):
                a = rng.integers(-128, 128, n, dtype=np.int8)
                if fill is not None:
                    a[:] = fill
                a = a.tobytes()
                body += a + b"\0" * (-len(a) % 4)
            a = rng.integers(-32768, 32768, bc, dtype=np.int16).tobytes()
            body += a + b"\0" * (-len(a) % 4)
        else:
            recs += b"\0" * 40
    return hdr + recs + body


# Synthetic layer stacks the shipped tables never exercise; shared by tests/test_gpu_models.py (whole streams) and the
# network-evaluation fixtures (tests/golden/make_golden_nets.py, tests/test_golden.py, tests/test_gpu_neteval.py).
#   name, nn_id, sizes, types (0 fc, 1 lstm), acts (0 relu6 1 tanh 2 sigmoid 3 linear), qk, qi, qb
NET_CASES = [
    ("fc_only", 1, (240, 33, 17, 2), (0, 0, 0), (1, 0, 3), (7, 5, 6), (8, 15, 12), (14, 15, 15)),
    ("two_lstm", 2, (240, 24, 20, 12, 9, 2), (0, 1, 0, 1, 0), (1, 1, 2, 1, 3), (6, 5, 5, 5, 6), (8, 15, 15, 15, 15), (13, 13, 15, 14, 15)),
    ("lstm_wide", 0, (240, 40, 100, 41), (0, 1, 0), (0, 1, 3), (7, 4, 5), (8, 15, 15), (14, 14, 14)),        # 13 unit groups
    ("lstm_requant", 0, (240, 40, 100, 41), (0, 1, 0), (0, 1, 3), (7, 4, 5), (8, 12, 15), (14, 14, 14)),     # qbit_input_rec != qbit_input
    ("lstm_last_fc_sigmoid", 1, (240, 10, 6, 2), (0, 1, 0), (2, 1, 3), (7, 6, 7), (8, 15, 15), (15, 12, 15)),
    ("odd_widths", 2, (240, 7, 5, 3, 2), (0, 1, 0, 0), (1, 1, 0, 3), (7, 5, 5, 7), (8, 15, 15, 12), (14, 13, 15, 15)),
    ("big_shifts", 1, (240, 16, 16, 2), (0, 1, 0), (1, 1, 3), (3, 7, 2), (8, 15, 15), (6, 15, 4)),
    ("bias_shift_18", 1, (240, 16, 16, 2), (0, 1, 0), (1, 1, 3), (12, 7, 2), (8, 15, 15), (2, 15, 4)),  # layer 0 needs the 64-bit finish
]
# crafted for the clamps and wraps of affine.c:186-249, affine_acc32b.c:187-249, lstm.c:106-115, activation.c:31-69
#   ..., fill (None = random weights)
NET_CRAFTED = [
    # lstm input Q8 -> recurrent Q15: shift_64b / shift_32b of the input half by +7 (saturates under ACC32BIT_OPT)
    ("shx_left7", 1, (240, 24, 16, 2), (0, 1, 0), (1, 1, 3), (7, 6, 7), (8, 8, 15), (14, 13, 15), None),
    # lstm input Q15 -> recurrent Q9: right shift of the input half
    ("shx_right6", 1, (240, 24, 16, 2), (0, 1, 0), (1, 1, 3), (7, 6, 7), (8, 15, 9), (14, 13, 15), None),
    # qk + qi = 30 with a Q0 bias: bias << 30 (wraps modulo 2^32 under ACC32BIT_OPT), output shift -15
    ("bias_shift_30", 1, (240, 16, 16, 2), (0, 1, 0), (1, 1, 3), (15, 15, 15), (15, 15, 15), (0, 0, 0), None),
    # every weight -128 / +127: largest dot products, tanh_fix far past 5.0, cell state driven into sat32
    ("all_m128", 2, (240, 32, 32, 2), (0, 1, 0), (1, 1, 3), (7, 5, 7), (8, 15, 15), (14, 13, 15), -128),
    ("all_p127", 2, (240, 32, 32, 2), (0, 1, 0), (2, 1, 3), (7, 5, 7), (8, 15, 15), (14, 13, 15), 127),
    ("all_m128_q0", 0, (240, 40, 40, 41), (0, 1, 0), (1, 1, 3), (0, 0, 0), (8, 15, 15), (15, 15, 15), -128),   # qs = 15: no output shift
]
# stacks the tcgen05 layer 0 takes (tanh fc 240 -> <= 80, exact 32-bit finish, an LSTM behind it) whose standardisation
# saturates: Q15 feature rows (feat_rshift 15) with the header's random means and stdR put most feature values at -32768
# or 32767, so the hi / lo byte split reaches hi = -128 and hi = 127, lo = 255; every weight -128 / +127 or random.
#   ..., fill (None = random weights)
NET_TC5_SATURATING = [
    ("sat_feat_m128", 2, (240, 32, 32, 2), (0, 1, 0), (1, 1, 3), (7, 5, 7), (15, 15, 15), (14, 13, 15), -128),
    ("sat_feat_p127", 2, (240, 32, 32, 2), (0, 1, 0), (1, 1, 3), (7, 5, 7), (15, 15, 15), (14, 13, 15), 127),
    ("sat_feat_random", 1, (240, 24, 16, 2), (0, 1, 0), (1, 1, 3), (7, 6, 7), (15, 15, 15), (14, 13, 15), None),
]
# stacks on either side of the rule that gives the cascade's sequential kernel its narrow shape (every layer at most 80
# wide, LSTM state at most 80, at most 48 outputs): exactly 80 / 48, then each limit crossed alone. The two LSTMs of
# kws_wide_h81 hold 40 + 41 units: a state offset that is a multiple of 4 keeps the scan-split form (NET_LIMITS has the
# 41 + 40 order, which only the dp2a kernels take).
NET_CASCADE_EDGES = [
    ("s2i_narrow_edge", 0, (240, 80, 80, 48), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 14, 14)),
    ("s2i_wide_rows81", 0, (240, 81, 80, 48), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 14, 14)),
    ("s2i_wide_out49", 0, (240, 80, 80, 49), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 14, 14)),
    ("kws_wide_h81", 2, (240, 40, 40, 41, 2), (0, 1, 1, 0), (1, 1, 1, 3), (7, 5, 5, 6), (8, 15, 15, 15), (14, 13, 13, 15)),
]

# stacks at the limits of include/nnsp_b200.h (10 layers, 128 units, 128 outputs) and on the LSTM shapes the shipped models
# never select. Kept out of NET_CASES: tests/golden/golden_nets_v1.npz is generated from the reference tree.
#   lstm_*: a second LSTM whose state offset is 1, 2 or 3 (mod 4) -- no IMMA or scan-split form, the dp2a kernels read the
#     old h through an aligned copy; lstm_41_87 ends at h_stride 128, lstm_off6 fits the cascade's narrow shape.
#   max_width*: LSTM state, widest layer and outputs at 128, scan_kernel<16,1,0>; layer 0 has 100 units because with 128
#     the dp2a weight image and scratch exceed 227 KB of shared memory. Every layer keeps MmaLayer.fast in both modes
#     (scan-split); _m128: every weight -128, the largest accumulators that bound admits.
#   ten_layers: two aligned LSTMs and a run of six fc layers in one seg_kernel; ten_layers_last_lstm: a last LSTM, whose
#     qbit_input_rec a 10-layer table reads from qbit_bias[0] (the 11th qi entry), so only that value round-trips. A
#     10-layer table gives its last layer that entry whatever the layer type: ten_layers carries it too.
#   scan_*: input and state need different numbers of 32-wide k-steps (scan_kernel<4,4,0>, <9,2,0>).
#   tc5_rows80_m128: the tcgen05 layer 0 at its 80-row limit, weights -128, Q15 (saturating) feature rows.
#   ..., fill (None = random weights)
NET_LIMITS = [
    ("lstm_off41", 2, (240, 16, 41, 40, 2), (0, 1, 1, 0), (1, 1, 1, 3), (7, 5, 5, 6), (8, 15, 15, 15), (14, 13, 13, 15), None),
    ("lstm_off6", 2, (240, 12, 6, 6, 2), (0, 1, 1, 0), (1, 1, 1, 3), (7, 5, 5, 6), (8, 15, 15, 15), (14, 13, 13, 15), None),
    ("lstm_7_5_3", 1, (240, 12, 7, 5, 3, 2), (0, 1, 1, 1, 0), (1, 1, 1, 1, 3), (7, 5, 5, 5, 6), (8, 15, 15, 15, 15),
     (14, 13, 13, 13, 15), None),
    ("lstm_41_87", 2, (240, 16, 41, 87, 2), (0, 1, 1, 0), (1, 1, 1, 3), (7, 5, 5, 6), (8, 15, 15, 15), (14, 13, 13, 15), None),
    ("max_width", 0, (240, 100, 128, 128), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 13, 15), None),
    ("max_width_m128", 0, (240, 100, 128, 128), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 13, 15), -128),
    ("ten_layers", 1, (240, 16, 24, 16, 20, 12, 12, 12, 12, 8, 2), (0, 1, 0, 1, 0, 0, 0, 0, 0, 0), (1, 1, 0, 1, 2, 0, 1, 2, 0, 3),
     (7, 5, 6, 5, 6, 6, 5, 6, 6, 6), (8, 15, 15, 15, 15, 12, 15, 15, 12, 15, 14), (14, 13, 15, 13, 15, 15, 14, 15, 15, 15), None),
    ("ten_layers_last_lstm", 1, (240, 16, 12, 12, 12, 12, 12, 12, 12, 12, 4), (0, 0, 0, 0, 0, 0, 0, 0, 0, 1), (1, 2, 0, 1, 2, 0, 1, 2, 0, 1),
     (7, 6, 6, 5, 6, 6, 5, 6, 6, 5), (8, 15, 12, 15, 15, 12, 15, 15, 12, 15, 14), (14, 15, 15, 14, 15, 15, 14, 15, 15, 13), None),
    ("scan_h32_kt4", 1, (240, 100, 32, 2), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 13, 15), None),
    ("scan_h48_kt4", 2, (240, 100, 48, 2), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 13, 15), None),
    ("scan_h72_kt2", 0, (240, 40, 72, 41), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 13, 15), None),
    ("tc5_rows80_m128", 2, (240, 80, 64, 2), (0, 1, 0), (1, 1, 3), (7, 5, 7), (15, 15, 15), (14, 13, 15), -128),
]


# scan_kernel<NT, MINB, KT> specialisations in the order launch_split_layers tries them (nnsp_b200_scan_kernel_launches)
SCAN_KINDS = ("4,4,1", "4,4,0", "8,2,2", "9,2,3", "9,2,0", "16,1,0")


def scan_kind(cols, rows):
    """the scan_kernel specialisation launch_split_layers picks for an LSTM of `rows` units behind `cols` inputs: NT unit
    groups of 8, k-steps of 32 for the input (kt) and the state (ktr), compiled in only when they agree"""
    nt, kt, ktr = (rows + 7) // 8, (cols + 31) // 32, (rows + 31) // 32
    kq = kt if kt == ktr else 0
    if nt <= 4:
        return "4,4,1" if kq == 1 else "4,4,0"
    if nt <= 8 and kq == 2:
        return "8,2,2"
    if nt <= 9:
        return "9,2,3" if kq == 3 else "9,2,0"
    return "16,1,0"


def lstm_scan_kinds(sizes, types):
    """Counter of the scan kinds a stack's LSTM layers select"""
    from collections import Counter
    return Counter(scan_kind(sizes[i], sizes[i + 1]) for i, t in enumerate(types) if t == 1)


def lstm_offsets(sizes, types):
    """state offset of each LSTM layer in the [h_stride] row (LSTM states back to back)"""
    out, ho = [], 0
    for i, t in enumerate(types):
        if t == 1:
            out.append(ho)
            ho += sizes[i + 1]
    return out


def net_case_blob(case, acc32):
    name, nn_id, sizes, types, acts, qk, qi, qb = case[:8]
    fill = case[8] if len(case) > 8 else None
    return make_blob(nn_id, sizes, types, list(acts), list(qk), list(qi), list(qb), seed=len(name) + 7 * acc32, fill=fill)


def net_case_dims(case):
    """(act_stride, h_stride, n_out) of a case"""
    sizes, types = case[2], case[3]
    return sum(sizes[1:-1]), sum(sizes[i + 1] for i, t in enumerate(types) if t == 1), sizes[-1]


def adversarial_net_inputs(rng, n_in=240):
    xs = [np.full(n_in, 32767), np.full(n_in, -32768), np.zeros(n_in), np.where(np.arange(n_in) % 2 == 0, 32767, -32768),
          np.where(np.arange(n_in) % 3 == 0, -32768, 32767)]
    for _ in range(11):
        xs.append(rng.integers(-32768, 32768, n_in))
    return np.stack(xs).astype(np.int16)


def adversarial_states(rng, n, h_stride):
    hs = max(h_stride, 1)
    h = rng.integers(-32768, 32768, (n, hs)).astype(np.int16)
    c = rng.integers(-2 ** 31, 2 ** 31, (n, hs)).astype(np.int32)
    h[0] = 0; c[0] = 0
    c[1] = 2 ** 31 - 1; c[2] = -2 ** 31 + 1
    h[3] = 32767; h[4] = -32768
    return h, c


def chunks(k, pattern=(100,)):
    """lengths of the calls that cover k frames, cycling through `pattern`, the last one cut to length"""
    out, i = [], 0
    while sum(out) < k:
        out.append(min(pattern[i % len(pattern)], k - sum(out)))
        i += 1
    return out


def cascade_events(res, valid):
    """per stream and frame t of the oracle cascade records: a new instance starts at t (stage change, or the stage's
    instance was reset at t - 1), a detection at t, a time-out at t (the controller moved on without a detection, or the
    s2i-only counter wrapped). res: [S][T] records, valid: [S][T]."""
    sid, pos, det = res["stage_id"].astype(int), res["pos_after"].astype(int), res["detected"] != 0
    new = np.zeros(sid.shape, bool)
    new[:, 1:] = (sid[:, 1:] != sid[:, :-1]) | (valid[:, :-1] == 0)
    pos_before = np.concatenate([np.zeros((len(pos), 1), int), pos[:, :-1]], axis=1)
    cnt = res["cnt_timeout"].astype(int)
    wrapped = np.zeros(sid.shape, bool)
    wrapped[:, 1:] = (sid[:, 1:] == sid[:, :-1]) & (cnt[:, 1:] < cnt[:, :-1])
    timeout = ~det & (sid != 1) & ((pos != pos_before) | wrapped)       # 1: VAD, which has no time-out
    return new, det, timeout


def widen_text(text, small, sizes):
    """the table text of a model whose layer sizes are `small`, rewritten for `sizes`: the size list, and every kernel,
    recurrent kernel and bias array with as many zero entries as the new sizes need"""
    text = text.replace(("{%s,}, // nn size" % ",".join(map(str, small))).encode(), ("{%s,}, // nn size" % ",".join(map(str, sizes))).encode())
    types = re.search(rb"\{((?:fc|lstm),)+\}, // layer type", text).group(0).decode().strip("{}").split(",")[:len(sizes) - 1]
    for i, t in enumerate(types):
        rows, cols = sizes[i + 1], sizes[i]
        nr = 4 * rows if t == "lstm" else rows
        for arr, n, z in (("kernel%d" % i, nr * cols, b"0x00,"), ("kernel_rec%d" % i, nr * rows if t == "lstm" else 0, b"0x00,"),
                          ("bias%d" % i, nr, b"0x0000,")):
            if n:
                text = re.sub(rb"(_" + arr.encode() + rb"\[\]=\{)[^}]*(\};)", lambda mo: mo.group(1) + z * n + mo.group(2), text)
    return text
