"""TEST INFRASTRUCTURE ONLY — CPU restatement of the reference's position→GSO builders.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs may import this module.  It is the checker, never the
product path.

Parity pin: ``tests/test_oracle_golden.py`` checks every function here against
golden vectors produced by *executing the reference itself*
(``oracle/make_golden.py``), and — when ``GFC_REFERENCE_ROOT`` names a checkout
of the original project — against the live reference.

Two builders exist upstream:

* ``binary_le``  — ``Scene.readADjMatrix`` (scene.py:140-154, called with
  MaxRange=2 at robot.py:654): ``A[i,j] = 1 if i != j and
  ((xi-xj)**2 + (yi-yj)**2)**0.5 <= R else 0``; python-float (fp64) arithmetic;
  returned flattened ``[1, N*N]``.
* ``sym_norm_lt`` — ``multiRobotSim.computeAdjacencyMatrix_fixedCommRadius``
  (utils/multirobotsim_dcenlocal.py:291-317): ``W = (pdist < R)``, zero
  diagonal, ``deg = W.sum(1)``, ``deg < 1e-9 -> isd = 0`` else
  ``isd = sqrt(1/deg)``, ``S = diag(isd) @ W @ diag(isd)``; fp64.
"""
import numpy as np

MODE_BINARY_LE = 0   # scene.py:147-149  (d <= R, values {0,1})
MODE_SYM_NORM_LT = 1  # multirobotsim_dcenlocal.py:307-315 (d < R, D^-1/2 W D^-1/2)
MODE_BINARY_LT = 2   # the W of mode 1 before normalisation (mask only)

ZERO_TOLERANCE = 1e-9  # multirobotsim_dcenlocal.py:51


def adjacency_scalar_le(pos_xy, max_range):
    """Scalar python-float loop, operation for operation as scene.py:143-152
    (``**2`` and ``**0.5`` on python floats).  Small inputs only.
    ``pos_xy``: [N,2] -> uint8 [N,N]."""
    n = len(pos_xy)
    out = np.zeros((n, n), dtype=np.uint8)
    for i in range(n):
        xi, yi = float(pos_xy[i][0]), float(pos_xy[i][1])
        for j in range(n):
            if i == j:
                continue
            xj, yj = float(pos_xy[j][0]), float(pos_xy[j][1])
            dij = ((xi - xj) ** 2 + (yi - yj) ** 2) ** 0.5
            out[i, j] = 1 if dij <= max_range else 0
    return out


def pairwise_dist(pos):
    """fp64 Euclidean distances, ``pos`` [B,N,2] -> [B,N,N]; squares, one add and a
    correctly rounded sqrt — the arithmetic of scene.py:147-148 and of scipy's
    ``pdist`` (multirobotsim_dcenlocal.py:306)."""
    p = np.asarray(pos, dtype=np.float64)
    dx = p[:, :, None, 0] - p[:, None, :, 0]
    dy = p[:, :, None, 1] - p[:, None, :, 1]
    return np.sqrt(dx * dx + dy * dy)


def adjacency(pos, radius, mode=MODE_BINARY_LE):
    """uint8 1-hop mask [B,N,N] for either comparison rule."""
    d = pairwise_dist(pos)
    if mode == MODE_BINARY_LE:
        a = d <= float(radius)
    else:
        a = d < float(radius)
    n = a.shape[1]
    a[:, np.arange(n), np.arange(n)] = False
    return a.astype(np.uint8)


def gso(pos, radius, mode=MODE_BINARY_LE):
    """GSO [B,N,N] float64 plus the uint8 mask.

    binary modes: S = mask (scene.py:140-154).
    sym_norm_lt : S = D^-1/2 W D^-1/2 with the zero-degree guard
                  (multirobotsim_dcenlocal.py:309-315)."""
    a = adjacency(pos, radius, mode)
    w = a.astype(np.float64)
    if mode != MODE_SYM_NORM_LT:
        return w, a
    deg = w.sum(axis=2)
    zero = np.abs(deg) < ZERO_TOLERANCE
    deg = np.where(zero, 1.0, deg)
    isd = np.sqrt(1.0 / deg)
    isd = np.where(zero, 0.0, isd)
    # (Deg @ W) @ Deg: left product first, as the reference's `Deg @ W[0] @ Deg`
    s = (isd[:, :, None] * w) * isd[:, None, :]
    return s, a


def random_geometric_positions(batch, n, box, seed, dtype=np.float32):
    """Synthetic swarm positions U(0, box)^2, SURVEY §8(d).  Stored in fp32 like
    the reference's recorded trajectories (V-REP C floats)."""
    rng = np.random.default_rng(seed)
    return (rng.random((batch, n, 2)) * box).astype(dtype)
