"""numpy reference of upfirdn shared by the host tests: the direct polyphase formula in float64."""
import numpy as np

from iqwaveform_b200 import _plan


def direct(x_buf, table, n_taps, up, down, *, x_first, out_first, n_out):
    """float64 y[n] = sum_j hp[p][j] * x[i0 - j] over global outputs [out_first, out_first + n_out), reading
    only the buffer that holds global samples [x_first, x_first + len(x_buf)) (zero elsewhere).  Usable as
    `compute` of distributed.upfirdn_time_sharded."""
    x_buf = np.asarray(x_buf).astype(np.complex128)
    rows, lp = table.shape
    p, i0 = _plan.upfirdn_phase_index(np.arange(out_first, out_first + n_out), up, down)
    y = np.zeros(n_out, np.complex128)
    for j in range(lp):
        idx = i0 - j - x_first
        ok = (idx >= 0) & (idx < x_buf.size) & (p < rows)
        y[ok] += table[p[ok], j].astype(np.complex128) * x_buf[idx[ok]]
    return y
