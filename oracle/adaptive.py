"""The stopping schedule of wofdm_ber_run_adaptive (include/wofdm.h) in plain Python integers.

Input: the counters of every (window pair v, SNR point s, ensemble index e) -- summed over the channels, as one-index
segments {s, e, 1} of wofdm_ber_run_segments return them.  Output: what the adaptive call must return.  No numpy
arithmetic on the schedule: Python integers do not overflow, so the 128-bit arithmetic of the library is restated exactly.
"""
from __future__ import annotations

BIT, SYM = 0, 1     # WOFDM_TARGET_BIT_ERRORS, WOFDM_TARGET_SYMBOL_ERRORS


def _range_sum(row, lo, hi):
    """sum of row[lo:hi]; a row may also be any object with range_sum(lo, hi) (a synthetic ensemble too large to list)"""
    if hasattr(row, "range_sum"):
        return int(row.range_sum(lo, hi))
    return sum(int(x) for x in row[lo:hi])


def schedule(bit, sym, target, target_kind=SYM, first_block=1, ensemble_max=None):
    """bit, sym: nested sequences [n_var][n_snr][>= ensemble_max] of per-ensemble-index counts (rows: see _range_sum).
    Returns (ensemble_used [n_snr], bit_err [n_var][n_snr], sym_err [n_var][n_snr], rounds, blocks) with blocks the list of
    each round's {point: block}."""
    n_var, n_snr = len(bit), len(bit[0])
    E = int(ensemble_max if ensemble_max is not None else len(bit[0][0]))
    assert target >= 1 and first_block >= 1 and E >= 1 and target_kind in (BIT, SYM)
    used = [0] * n_snr
    block = [min(int(first_block), E)] * n_snr
    done = [False] * n_snr
    tb = [[0] * n_snr for _ in range(n_var)]
    ts = [[0] * n_snr for _ in range(n_var)]
    rounds, blocks = 0, []
    while not all(done):
        active = [s for s in range(n_snr) if not done[s]]           # ascending SNR order
        blocks.append({s: block[s] for s in active})
        rounds += 1
        for s in active:
            lo, hi = used[s], used[s] + block[s]
            for v in range(n_var):
                tb[v][s] += _range_sum(bit[v][s], lo, hi)
                ts[v][s] += _range_sum(sym[v][s], lo, hi)
        for s in active:
            used[s] += block[s]
            m = min((tb if target_kind == BIT else ts)[v][s] for v in range(n_var))
            if m >= target or used[s] == E:
                done[s] = True
                continue
            nb = min(E - used[s], 2 * block[s])
            if m > 0:
                nb = min(nb, max(1, -(-(target - m) * used[s] // m)))   # ceil((target - m) * e / m)
            block[s] = nb
    return used, tb, ts, rounds, blocks
