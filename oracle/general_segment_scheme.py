"""TEST INFRASTRUCTURE ONLY (never imported by mica_b200/): a NumPy statement of the segment scheme of the GENERAL
resample path's z prefilter (mica_b200/csrc/resample.cu: iir_segment, prefilter_cols_seg<., 16>, seg16_plan), the
one integer maps take.  oracle/segment_scheme.py states the fast path's register scheme; this is its float64
counterpart: 16 segments per line, a 30-sample horizon, and the exact end initialisation at the line's last sample.

What it pins on the CPU: a block [g0, g0 + n) of a line of ng samples, cut on the WHOLE line's segment grid, gives
the whole line's float64 coefficients bit for bit -- provided the block holds the raw samples ``plan`` names -- and a
block cut into its OWN 16 segments (mirrored at its own ends) does not.

The arithmetic follows the kernel operation by operation, except that NumPy has no fused multiply-add: a * b + c is
rounded twice here, once on the GPU.  The bit-identity property does not depend on that (same operations on the same
inputs in the same order)."""
import numpy as np

POLE = np.float64(-0.26794919243112270647)          # sqrt(3) - 2
GAIN = (1.0 - POLE) * (1.0 - 1.0 / POLE)            # = 6
SEGS, HORIZON = 16, 30                              # prefilter_cols_seg<., 16>, kHorizon
MIN_LINE, MAX_LINE = 96, 800                        # kMinSegLine, kMaxSeg16Line


def seg_len(ng):
    return -(-ng // SEGS)


def plan(ng, need_lo, need_hi):
    """seg16_plan: (seg_lo, seg_causal_hi, seg_out_hi, causal_end, raw_lo, raw_hi) for global samples
    [need_lo, need_hi]."""
    ln = seg_len(ng)
    seg_lo, seg_out_hi = need_lo // ln, need_hi // ln
    k1 = min(ng, (seg_out_hi + 1) * ln)
    last = k1 - 1
    if k1 < ng:
        last = ng - 1 if k1 + HORIZON >= ng else k1 + HORIZON - 1
    if k1 >= ng and ng >= 2 and (ng - 2) // ln < seg_lo:
        seg_lo = (ng - 2) // ln
    seg_causal_hi = last // ln
    k0 = seg_lo * ln
    raw_lo = max(0, k0 - HORIZON)
    raw_hi = min(ng, max(last + 1, HORIZON - k0 + 1 if k0 < HORIZON else 0))
    return seg_lo, seg_causal_hi, seg_out_hi, last + 1, raw_lo, raw_hi


class _Block:
    """Lines [lines, n] holding global samples [g0, g0 + n): reads outside the block raise."""

    def __init__(self, data, g0):
        self.data, self.g0 = data, g0

    def __getitem__(self, k):
        loc = k - self.g0
        if not 0 <= loc < self.data.shape[1]:
            raise IndexError(f'sample {k} is outside the block [{self.g0}, {self.g0 + self.data.shape[1]})')
        return self.data[:, loc]

    def __setitem__(self, k, v):
        self.data[:, k - self.g0] = v


def prefilter(block, g0, ng, seg_lo=0, seg_causal_hi=SEGS - 1, seg_out_hi=SEGS - 1, causal_end=None):
    """prefilter_cols_seg<., 16> on ``block`` [lines, n] = samples [g0, g0 + n) of lines of ``ng`` samples (any
    numeric type).  Returns float64 [lines, n]: the coefficients of the samples of segments seg_lo..seg_out_hi;
    the other samples hold intermediate values."""
    z = POLE
    causal_end = ng if causal_end is None else causal_end
    ln = seg_len(ng)
    raw = _Block(block.astype(np.float64) * GAIN, g0)
    segs = [(s, s * ln, min(ng, s * ln + ln)) for s in range(SEGS) if s * ln < min(ng, s * ln + ln)]
    causal = [t for t in segs if seg_lo <= t[0] <= seg_causal_hi]
    anti = [t for t in segs if seg_lo <= t[0] <= seg_out_hi]
    state = {}
    for s, k0, _ in causal:                   # warm-ups read raw samples (before the first barrier)
        st = np.zeros(block.shape[0])
        for m in range(HORIZON - 1, -1, -1):
            st = z * st + raw[abs(k0 - 1 - m)]
        state[s] = st
    line = _Block(raw.data.copy(), g0)
    for s, k0, k1 in causal:                  # causal sweeps
        st = state[s]
        for k in range(k0, min(k1, causal_end)):
            st = z * st + raw[k]
            line[k] = st
    n = ng
    for s, k0, k1 in anti:                    # anticausal warm-ups read causal values (after the barrier)
        if k1 >= n:
            state[s] = None
            continue
        kk = k1 + HORIZON
        k = kk - 1
        st = np.zeros(block.shape[0])
        if kk >= n:
            st = (z / (z * z - 1.0)) * (line[n - 1] + z * line[n - 2])
            k = n - 2
        while k >= k1:
            st = z * st + (-z * line[k])
            k -= 1
        state[s] = st
    out = _Block(line.data.copy(), g0)
    for s, k0, k1 in anti:                    # anticausal sweeps (in place in the kernel; segments are disjoint)
        st, k = state[s], k1 - 1
        if st is None:
            st = (z / (z * z - 1.0)) * (line[n - 1] + z * line[n - 2])
            out[n - 1] = st
            k = n - 2
        while k >= k0:
            st = z * st + (-z * line[k])
            out[k] = st
            k -= 1
    return out.data
