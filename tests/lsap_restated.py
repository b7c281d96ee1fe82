"""Sequential restatement of scipy's rectangular linear_sum_assignment (Crouse's shortest augmenting path,
scipy/optimize/_lsap.py -> rectangular_lsap.cpp), tie rules included.  ct_track_step's --hungarian solver
(csrc/stream.cu, lsap_warp) runs these very steps, one warp per stream; tests/test_track_modes_cpu.py pins this
restatement to scipy pair for pair on tie-heavy and blocked matrices."""
import numpy as np


def lsap(cost):
  """(rows, cols) exactly as scipy.optimize.linear_sum_assignment(cost) returns them for a finite float64 cost."""
  cost = np.asarray(cost, np.float64)
  nr, nc = cost.shape
  if nr == 0 or nc == 0:
    return np.zeros(0, np.int64), np.zeros(0, np.int64)
  tr = nc < nr
  if tr:                                          # more rows than columns: solve the transpose
    cost = cost.T.copy()
    nr, nc = nc, nr
  u, v = np.zeros(nr), np.zeros(nc)
  path = -np.ones(nc, np.int64)
  col4row, row4col = -np.ones(nr, np.int64), -np.ones(nc, np.int64)
  for cur in range(nr):
    min_val = 0.0
    remaining = list(range(nc - 1, -1, -1))
    n_rem = nc
    row_seen, col_seen = np.zeros(nr, bool), np.zeros(nc, bool)
    spc = np.full(nc, np.inf)
    i, sink = cur, -1
    while sink == -1:                             # one Dijkstra round per column taken
      idx, low = -1, np.inf
      row_seen[i] = True
      for it in range(n_rem):
        j = remaining[it]
        r = ((min_val + cost[i, j]) - u[i]) - v[j]
        if r < spc[j]:
          path[j] = i
          spc[j] = r
        # among equal minima: the last unassigned column in scan order, else the first
        if spc[j] < low or (spc[j] == low and row4col[j] == -1):
          low, idx = spc[j], it
      min_val = low
      j = remaining[idx]
      if row4col[j] == -1:
        sink = j
      else:
        i = row4col[j]
      col_seen[j] = True
      n_rem -= 1
      remaining[idx] = remaining[n_rem]
    u[cur] += min_val
    for i in range(nr):
      if row_seen[i] and i != cur:
        u[i] += min_val - spc[col4row[i]]
    for j in range(nc):
      if col_seen[j]:
        v[j] -= min_val - spc[j]
    j = sink
    while True:                                   # augment along the path
      i = path[j]
      row4col[j] = i
      col4row[i], j = j, col4row[i]
      if i == cur:
        break
  if tr:
    order = np.argsort(col4row, kind='stable')
    return col4row[order], order
  return np.arange(nr), col4row
