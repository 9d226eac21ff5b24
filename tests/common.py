"""Shared helpers for the parity tests."""
import hashlib
import os

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
    fill: every kernel byte gets this int8 value instead (crafted extremes: -128, 127)."""
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
            qin = qi[i + 1] if i + 1 < nl else 0
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
# kws_wide_h81 hold 40 + 41 units: a state offset that is a multiple of 4 keeps the scan-split form (41 + 40 would not).
NET_CASCADE_EDGES = [
    ("s2i_narrow_edge", 0, (240, 80, 80, 48), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 14, 14)),
    ("s2i_wide_rows81", 0, (240, 81, 80, 48), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 14, 14)),
    ("s2i_wide_out49", 0, (240, 80, 80, 49), (0, 1, 0), (1, 1, 3), (7, 5, 6), (8, 15, 15), (14, 14, 14)),
    ("kws_wide_h81", 2, (240, 40, 40, 41, 2), (0, 1, 1, 0), (1, 1, 1, 3), (7, 5, 5, 6), (8, 15, 15, 15), (14, 13, 13, 15)),
]


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
