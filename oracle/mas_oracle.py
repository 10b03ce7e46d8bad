"""Oracle for Monotonic Alignment Search: a plain numpy restatement of the reference's algorithm
(training/vits2/monotonic_align/core.pyx:7-34, driver monotonic_align/__init__.py:6-22).  TEST INFRASTRUCTURE: only tests/,
__graft_entry__.smoke() and bench.py's CPU legs may import this; the product path is vosk_tts_b200/csrc (mas_kernel).

Pinned against the reference itself: oracle/build_ref_mas.py compiles the reference's own core.pyx into oracle/_ref/, and
tests/test_mas.py compares this restatement bit for bit with the committed fixtures tests/golden/mas_*.npz that
oracle/make_golden_mas.py and oracle/make_golden_reference.py generated from it.
"""
import numpy as np

MAX_NEG = np.float32(-1e9)


def maximum_path_each(value, t_y, t_x):
    """value: float32 [T_y, T_x], updated IN PLACE like the reference (core.pyx:16-29); returns int32 path [T_y, T_x].
    Forward pass: value[y, x] += max(value[y-1, x-1], value[y-1, x]) inside the band max(0, t_x + y - t_y) <= x < min(t_x, y + 1),
    with value[-1, -1] := 0 and everything else outside := -1e9.  Backtrack from (t_y - 1, t_x - 1) (core.pyx:31-34)."""
    path = np.zeros(value.shape, np.int32)
    for y in range(t_y):
        for x in range(max(0, t_x + y - t_y), min(t_x, y + 1)):
            v_cur = MAX_NEG if x == y else value[y - 1, x]
            if x == 0:
                v_prev = np.float32(0.0) if y == 0 else MAX_NEG
            else:
                v_prev = value[y - 1, x - 1]
            value[y, x] = np.float32(value[y, x] + max(v_prev, v_cur))
    index = t_x - 1
    for y in range(t_y - 1, -1, -1):
        path[y, index] = 1
        if index != 0 and (index == y or value[y - 1, index] < value[y - 1, index - 1]):
            index -= 1
    return path


def maximum_path(neg_cent, t_ys, t_xs):
    """neg_cent float32 [B, T_y, T_x] (a copy is modified), t_ys / t_xs int [B] -> int32 paths [B, T_y, T_x]
    (monotonic_align/__init__.py:15-22: lengths come from the mask sums)."""
    value = np.array(neg_cent, dtype=np.float32, copy=True)
    out = np.zeros(value.shape, np.int32)
    for b in range(value.shape[0]):
        out[b] = maximum_path_each(value[b], int(t_ys[b]), int(t_xs[b]))
    return out


def maximum_path_vectorised(neg_cent, t_ys, t_xs):
    """Same result, one numpy expression per row (for the large cases the pure loops would take minutes on)."""
    value = np.array(neg_cent, dtype=np.float32, copy=True)
    B, Ty, Tx = value.shape
    out = np.zeros(value.shape, np.int32)
    for b in range(B):
        t_y, t_x = int(t_ys[b]), int(t_xs[b])
        v = value[b]
        for y in range(t_y):
            lo, hi = max(0, t_x + y - t_y), min(t_x, y + 1)
            if hi <= lo:
                continue
            xs = np.arange(lo, hi)
            if y == 0:
                v_cur = np.full(xs.shape, MAX_NEG, np.float32)
                v_prev = np.where(xs == 0, np.float32(0.0), MAX_NEG).astype(np.float32)
            else:
                v_cur = np.where(xs == y, MAX_NEG, v[y - 1, np.minimum(xs, Tx - 1)]).astype(np.float32)
                v_prev = np.where(xs == 0, MAX_NEG, v[y - 1, np.maximum(xs - 1, 0)]).astype(np.float32)
            v[y, lo:hi] = (v[y, lo:hi] + np.maximum(v_prev, v_cur)).astype(np.float32)
        index = t_x - 1
        for y in range(t_y - 1, -1, -1):
            out[b, y, index] = 1
            if index != 0 and (index == y or v[y - 1, index] < v[y - 1, index - 1]):
                index -= 1
    return out
