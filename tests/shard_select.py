"""Test infrastructure: the reference of the max-loc of sharded MPE / MAP (bnpp_mpe_shard_select).

Rank r's record is the words [r * stride, (r + 1) * stride) of a uint32 array, stride = 2 + nvars rounded up to an even
number: its value (a double, words 0-1) and its assignment (words 2 .. 2 + nvars).  The winner follows the rule of the
max kernels over the ranks (`mpe_oracle.max_last_axis`): rank 0 first, a later rank replaces it only if its value is
strictly greater -- ties keep the lowest rank and a NaN never replaces a number."""
import numpy as np


def stride(nvars):
    return (2 + nvars + 1) // 2 * 2


def pack(values, assignments):
    """records of len(values) ranks: value r and assignment r (a sequence of nvars uint32) -> flat uint32 array"""
    nvars = len(assignments[0])
    s = stride(nvars)
    rec = np.zeros((len(values), s), dtype=np.uint32)
    rec[:, 0:2] = np.asarray(values, dtype=np.float64).reshape(-1, 1).view(np.uint32)
    rec[:, 2:2 + nvars] = np.asarray(assignments, dtype=np.uint32)
    return rec.reshape(-1)


def select(records, nranks, nvars):
    """-> (winning rank, its value as a float64, its assignment as a uint32 array)"""
    rec = np.asarray(records, dtype=np.uint32).reshape(nranks, stride(nvars))
    values = np.ascontiguousarray(rec[:, 0:2]).view(np.float64).reshape(-1)
    best, win = values[0], 0
    for r in range(1, nranks):
        if values[r] > best:            # NaN > x and x > NaN are both false
            best, win = values[r], r
    return win, values[win], rec[win, 2:2 + nvars].copy()
