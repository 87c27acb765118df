"""Host restatement of the scenario-mixture draw (include/renv.h renv_env_mixture, DESIGN section 4.16).

Test infrastructure: uses the Philox restatement of oracle/f32_draws.py.  A reset of env id at tick t reads words x, y
of block (seed, id, t, purpose 6, slot 0); column j = x C >> 32; row j when y < q_j, else alias_j.
"""
import numpy as np

from oracle.f32_draws import draw_block

PURPOSE_MIXTURE = 6


def split(table):
    """(q, alias) int64 arrays of an int64 alias table (entry q | alias << 32)."""
    table = np.asarray(table, dtype=np.int64)
    return table & 0xFFFFFFFF, (table >> 32) & 0xFFFF


def draw_rows(seed, ids, ticks, table):
    """Rows drawn by the resets of env ids ``ids`` at clock ``ticks`` (broadcast together) from ``table``."""
    q, alias = split(table)
    C = len(q)
    x, y = draw_block(seed, ids, ticks, PURPOSE_MIXTURE, 0)[:2]
    j = ((x.astype(np.uint64) * np.uint64(C)) >> np.uint64(32)).astype(np.int64)
    return np.where(y.astype(np.int64) < q[j], j, np.minimum(alias[j], C - 1))


def exact_counts(table):
    """Exact probability of every row under ``table``: (C,) Python ints over 2^64.  Column j is hit by the
    ceil((j + 1) 2^32 / C) - ceil(j 2^32 / C) values of x with x C >> 32 == j, and keeps its row for q_j of the 2^32
    values of y."""
    q, alias = split(table)
    C = len(q)
    out = [0] * C
    for j in range(C):
        hits = ((((j + 1) << 32) + C - 1) // C) - (((j << 32) + C - 1) // C)
        keep = int(q[j])
        out[j] += hits * keep
        out[min(int(alias[j]), C - 1)] += hits * ((1 << 32) - keep)
    return out
