"""numpy restatement of the round rule by which the GPU Felzenszwalb (csrc/pcm_felzenszwalb.cuh) runs the two
passes of `felzenszwalb_oracle._merge` in parallel.

TEST INFRASTRUCTURE ONLY (see oracle/pcm_oracle.py header).

The rule decides, in each round, only edges whose outcome the sequential pass is certain to give:
  merge pass     an edge at position p with current roots ra != rb; m[X] = the earliest remaining edge at X whose X side
                 accepts it (cost < limit[X]).  p < m[ra] or p < m[rb]: certain rejection, dropped.  p == m[ra] == m[rb]:
                 certain merge, applied as the sequential pass applies it.  Everything else waits for the next round.
  min-size pass  an edge between two components of min_size pixels or more is dropped; an edge that is the earliest
                 remaining edge of both its components is merged; everything else waits.
The rule is deterministic, so the device reports the same round counts as this restatement.
"""
import numpy as np

_NONE = np.iinfo(np.int64).max


def merge_rounds(e0, e1, costs, n, scale, min_size):
    """Edges already in the stable cost order (as `_merge` takes them).  Returns (root, merge rounds, min-size rounds):
    root[i] = the root of vertex i, the smallest vertex of its component, as `_merge` returns it."""
    e0, e1 = np.asarray(e0, np.int64), np.asarray(e1, np.int64)
    costs = np.asarray(costs, np.float64)
    parent = np.arange(n)
    size = np.ones(n, np.int64)
    limit = np.full(n, 0.0 + scale / 1)

    def apply(ra, rb, c=None):
        lo, hi = np.minimum(ra, rb), np.maximum(ra, rb)
        total = size[ra] + size[rb]
        parent[hi] = lo
        size[lo] = total
        if c is not None:
            limit[lo] = c + scale / total

    pos, merge = np.arange(costs.size), 0
    while True:
        ra, rb = parent[e0[pos]], parent[e1[pos]]
        live = ra != rb
        pos, ra, rb = pos[live], ra[live], rb[live]
        if not pos.size:
            break
        merge += 1
        c = costs[pos]
        sa, sb = c < limit[ra], c < limit[rb]
        m = np.full(n, _NONE)
        np.minimum.at(m, ra[sa], pos[sa])
        np.minimum.at(m, rb[sb], pos[sb])
        reject = (pos < m[ra]) | (pos < m[rb])
        accept = (pos == m[ra]) & (pos == m[rb])
        apply(ra[accept], rb[accept], c[accept])
        parent = parent[parent]            # a round's merges form a matching: one jump restores depth 1
        pos = pos[~(reject | accept)]

    pos, small = np.arange(costs.size), 0
    while True:
        ra, rb = parent[e0[pos]], parent[e1[pos]]
        live = (ra != rb) & ((size[ra] < min_size) | (size[rb] < min_size))
        pos, ra, rb = pos[live], ra[live], rb[live]
        if not pos.size:
            break
        small += 1
        best = np.full(n, _NONE)
        np.minimum.at(best, ra, pos)
        np.minimum.at(best, rb, pos)
        accept = (best[ra] == pos) & (best[rb] == pos)
        apply(ra[accept], rb[accept])
        parent = parent[parent]
        pos = pos[~accept]
    return parent, merge, small
