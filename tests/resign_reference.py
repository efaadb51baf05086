"""Host restatement of the resignation rule of advance_kernel (include/caro_b200.h, beside CARO_FLAG_*): the root
statistic, the playthrough draw and the false-positive definition.  Python floats are IEEE doubles rounded to nearest,
so a sequential loop of ``+`` and one ``/`` is exactly the kernel's __dadd_rn / __ddiv_rn chain; numpy float32 division
is __fdiv_rn."""
import ctypes as C
import os

import numpy as np

STREAM_RESIGN = 0x52455347  # kStreamResign, csrc/rng.cuh
HOSTCHECK = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native", "libhostcheck.so")


def root_stat(n_row, w_row):
    """max(v_root, v_best) of one root row (N masked counts, W float32), or None when the row has no visit."""
    n_row = [int(v) for v in n_row]
    w_row = np.asarray(w_row, dtype=np.float32)
    total = sum(n_row)
    if total == 0:
        return None
    acc = 0.0
    for w in w_row:  # action order, not np.sum (pairwise)
        acc = acc + float(w)
    v_root = acc / float(total)
    best = max(range(len(n_row)), key=lambda a: (n_row[a], -a))  # most visits, lowest action on ties
    v_best = float(np.float32(w_row[best]) / np.float32(n_row[best]))
    return max(v_root, v_best)


def u01d(hi, lo):
    return float(((hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0)


def philox(c0, c1, c2, c3, k0, k1):
    lib = C.CDLL(HOSTCHECK)
    out = (C.c_uint32 * 4)()
    lib.hc_philox(C.c_uint32(c0), C.c_uint32(c1), C.c_uint32(c2), C.c_uint32(c3), C.c_uint32(k0), C.c_uint32(k1), out)
    return [int(v) for v in out]


def is_playthrough(uid, seed, share):
    r = philox(uid & 0xFFFFFFFF, uid >> 32, 0, 0, (seed & 0xFFFFFFFF) ^ STREAM_RESIGN, seed >> 32)
    return u01d(r[0], r[1]) < share


def false_positive(min_stat, result, t):
    """Some player whose smallest statistic is < t did not lose (result is player 0's view)."""
    return any(min_stat[p] < t and result != (-1 if p == 0 else 1) for p in (0, 1))
