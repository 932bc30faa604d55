#!/usr/bin/env python
"""Python model of the device cardinality search (csrc/kernels.cuh: spec_hist_add, k_radix_hist, radix_pick_block;
csrc/solver.cu: k_sel_begin): MSB-first radix select of the k-th largest magnitude key with digits of `dbits` bits, the
first levels optionally decided from speculative statistics built around a guess (the previous threshold).  The model
mirrors the kernels' digit arithmetic (shifts, masks, bins per thread, the `above < k <= above + |bucket|` test); it is
checked against a sort in tests/test_select_model.py for random keys, ties, zeros and right / wrong guesses.  Nothing in
the product imports it."""
import numpy as np

SPECBITS, SPECLEV, BINS = 11, 3, 2048


def pick(st, h):
    """radix_pick_block: thread t owns 2^w / 256 bins from the top down; the thread whose bins hold the k-th key decides."""
    bl = st["bits_left"]
    if bl <= 0:
        return
    w = min(st["dbits"], bl)
    nb = 1 << w
    per = nb >> 8
    k = st["k_rem"]
    top_down = np.asarray(h[:nb][::-1], dtype=np.int64)            # bins from the top down
    above = np.concatenate(([0], np.cumsum(top_down)))             # above[i]: keys in the i highest bins
    for t in range(256):
        lo, hi = t * per, (t + 1) * per                            # this thread's bins (top-down positions)
        excl, incl = int(above[lo]), int(above[hi])
        if incl >= k and excl < k:
            cum = excl
            for j in range(lo, hi):
                c = int(top_down[j])
                if cum + c >= k:
                    st.update(k_rem=k - cum, count_eq=c, prefix=(st["prefix"] << w) | (nb - 1 - j), bits_left=bl - w)
                    break
                cum += c
    h[:nb] = 0


def select(keys, k, KB, guess=0, dbits=11, spec=True):
    """Returns (state, number of real histogram passes).  state: prefix = threshold key, k_rem = tie quota,
    count_eq = keys equal to the threshold."""
    keys = np.asarray(keys).astype(np.uint64)

    def digit(sel, shift, w):                              # histogram of bits [shift, shift + w) of the selected keys
        return np.bincount(((keys[sel] >> np.uint64(shift)) & np.uint64((1 << w) - 1)).astype(np.int64), minlength=BINS)

    st = dict(prefix=0, k_rem=k, count_eq=0, bits_left=KB, key_bits=KB, dbits=dbits)
    passes = 0
    if spec:                                              # k_yl_spec + k_sel_begin
        sh = np.zeros((SPECLEV - 1, BINS), dtype=np.int64)
        g0 = guess >> (KB - SPECBITS)
        d0 = keys >> np.uint64(KB - SPECBITS)
        above = int(np.count_nonzero(d0 > np.uint64(g0)))
        same = d0 == np.uint64(g0)
        for lv in range(1, SPECLEV):
            bl = KB - SPECBITS * lv
            w = min(bl, SPECBITS)
            sel = same if lv == 1 else same & ((keys >> np.uint64(bl)) == np.uint64(guess >> bl))
            sh[lv - 1] = digit(sel, bl - w, w)
        bucket = int(sh[0].sum())
        if above < k <= above + bucket:
            st.update(prefix=g0, k_rem=k - above, count_eq=bucket, bits_left=KB - SPECBITS)
            for lv in range(1, SPECLEV):
                bl = st["bits_left"]
                if not (bl == KB - lv * SPECBITS and st["prefix"] == (guess >> bl)):
                    break
                pick(st, sh[lv - 1])
    for _ in range((KB + dbits - 1) // dbits):            # k_radix_hist launches: decided levels return at once
        bl = st["bits_left"]
        if bl <= 0:
            continue
        passes += 1
        w = min(dbits, bl)
        sel = slice(None) if bl >= KB else (keys >> np.uint64(bl)) == np.uint64(st["prefix"])
        pick(st, digit(sel, bl - w, w))
    assert st["bits_left"] == 0, st
    return st, passes
