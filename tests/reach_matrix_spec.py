"""The path-cost matrix (mlm_reach_matrix) restated from the spec in include/mlmap_b200.h on top of the reachability
field's restatement (tests/reach_spec.py): one scipy Dijkstra per row, that row's start cell its only source."""
import numpy as np

from reach_spec import field


def matrix(cls, starts_cells, goal_cells, K, unknown=False):
    """the matrix on a class grid [N_z, N_y, N_x]: row i is the field from box-relative start cell starts_cells[i] alone
    (no source when it lies outside the box), read at the box-relative goal cells; int64 costs, -1 unreachable, -2 for a
    goal outside the box.  The row's source is passable in its own row only."""
    goals = np.asarray(goal_cells, dtype=np.int64).reshape(-1, 3)
    dims = np.array(cls.shape[::-1])
    inside = ((goals >= 0) & (goals < dims)).all(1)
    g = np.where(inside[:, None], goals, 0)
    out = np.full((len(starts_cells), goals.shape[0]), -2, dtype=np.int64)
    for i, s in enumerate(starts_cells):
        f = field(cls, [s], K, unknown)
        out[i] = np.where(inside, f[g[:, 2], g[:, 1], g[:, 0]], -2)
    return out
