"""Float64 restatement of one device leapfrog step (mt_kernels.cuh: k_drift_max + k_drift, k_kick, k_energies; hmcmt_b200.cu:
k_accept), vectorised over the cells and written in the kernels' operation order, so that a kernel's result can be held to
round-off at any shape, chain count and block count.  Sums use math.fsum: the reference does not depend on summation order."""
import math

import numpy as np

MAX_STEP = 3.0          # largest |dm| of one drift (HMCSampler.jl:237-243)
MAX_BOUNCES = 500       # iterations of the reflection loop (each reflects at most twice) before the bounds flag (-21)


def drift(m, p, dt, lo, hi, invM=None):
    """dm = dt (invM p or p), rescaled to max |dm| = 3 when it is larger (a tie is not rescaled), m + dm reflected into
    [lo, hi] with a momentum flip per reflection (checkParameterBound! HMCSampler.jl:515-559).
    -> (m', p', reflections per element, whether some element hit the 500-reflection guard)."""
    m = np.asarray(m, dtype=np.float64)
    p = np.array(p, dtype=np.float64)
    gk = p if invM is None else invM @ p
    dm = dt * gk
    mx = np.abs(dm).max()
    if mx > MAX_STEP:
        dm = dm / mx * MAX_STEP
    v = m + dm
    bounces = np.zeros(len(v), dtype=np.int64)
    todo = ~((v <= hi) & (v >= lo))
    guard = False
    it = 0
    while todo.any():
        it += 1
        low = todo & (v < lo)                     # the < lo branch, then the > hi branch in the same iteration
        v[low] = 2.0 * lo - v[low]
        p[low] = -p[low]
        high = todo & (v > hi)
        v[high] = 2.0 * hi - v[high]
        p[high] = -p[high]
        bounces += low.astype(np.int64) + high.astype(np.int64)
        todo &= ~((v <= hi) & (v >= lo))
        if it >= MAX_BOUNCES and todo.any():
            guard = True
            break
    return v, p, bounces, guard


def kick(p, g, dt, scale=1.0):
    """p - scale dt g (k_kick with scale 1, k_kick_masked with 0.5 / 1)."""
    return np.asarray(p, dtype=np.float64) - scale * dt * np.asarray(g, dtype=np.float64)


def energies(m, mref, p, Wm, beta, invM=None):
    """(K, phi_m) = (1/2 p^T invM p, 1/2 beta (m - mref)^T Wm (m - mref)) (getKineticEnergy HMCSampler.jl:407-415, mnorm :393),
    each product summed exactly (math.fsum) and rounded once."""
    p = np.asarray(p, dtype=np.float64)
    gk = p if invM is None else invM @ p
    d = np.asarray(m, dtype=np.float64) - np.asarray(mref, dtype=np.float64)
    K = 0.5 * math.fsum(p * gk)
    phim = 0.5 * beta * math.fsum(d * (Wm @ d))
    return K, phim


def accept(H_start, H_fin, u):
    """The Metropolis decision of k_accept (HMCSampler.jl:149-186)."""
    hdif = H_start - H_fin
    return bool(hdif > 0.0 or u < math.exp(hdif))
