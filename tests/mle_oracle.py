"""float64 maximum-likelihood oracle for fit_likelihood: the exact maximiser by enumeration of all 2^N configurations.
TEST INFRASTRUCTURE ONLY; nothing under graphicalmodellearning.jl_b200/ imports it."""
import math

import numpy as np


def mle_exact(terms, num_spins: int, data_mean, lam: float, tol: float = 1e-14, max_outer: int = 100):
    """argmax_w  sum_t w_t m^_t - log Z(w) - lam * sum_{|t| >= 2} |w_t|  over the weights of the keys of `terms` (1-based
    index tuples; their values are the starting point), m^ = data_mean in key order.  float64 enumeration of all 2^N
    configurations; proximal Newton with the exact Hessian (the covariance of the features) and a coordinate-descent
    inner loop, stopped when the max-norm of the prox-gradient mapping at unit step is <= tol.  Returns the weights in
    key order."""
    keys = list(terms)
    w = np.array([float(terms[k]) for k in keys])
    dm = np.asarray(data_mean, dtype=np.float64)
    pen = np.array([len(k) >= 2 for k in keys])
    ids = np.arange(1 << num_spins)
    spins = (2 * ((ids[:, None] >> np.arange(num_spins)[None, :]) & 1) - 1).astype(np.float64)
    phi = np.stack([np.prod(spins[:, [i - 1 for i in k]], axis=1) for k in keys], axis=1)

    def smooth(x):
        e = phi @ x
        top = e.max()
        p = np.exp(e - top)
        z = p.sum()
        p /= z
        return top + math.log(z) - x @ dm, p

    def total(x):
        return smooth(x)[0] + lam * np.abs(x[pen]).sum()

    def soft(z, t):
        return np.sign(z) * max(abs(z) - t, 0.0)

    for _ in range(max_outer):
        f, p = smooth(w)
        m = p @ phi
        grad = m - dm
        step = w - grad
        step[pen] = np.sign(step[pen]) * np.maximum(np.abs(step[pen]) - lam, 0.0)
        if np.abs(step - w).max() <= tol:
            break
        H = phi.T @ (phi * p[:, None]) - np.outer(m, m)
        x = w.copy()
        for _sweep in range(10000):          # min_x grad.(x - w) + (x - w)' H (x - w) / 2 + lam |x_pen|_1
            change = 0.0
            for j in range(len(w)):
                a = H[j, j]
                b = grad[j] + H[j] @ (x - w)
                z = x[j] - b / a
                new = soft(z, lam / a) if pen[j] else z
                change = max(change, abs(new - x[j]))
                x[j] = new
            if change <= 1e-16:
                break
        d = x - w
        decrease = grad @ d + lam * (np.abs(x[pen]).sum() - np.abs(w[pen]).sum())
        t, f0 = 1.0, total(w)
        slack = 1e-14 * (1.0 + abs(f0))     # the rounding of log Z, which dominates near the optimum
        while total(w + t * d) > f0 + 0.25 * t * decrease + slack and t > 1e-10:
            t *= 0.5
        w = w + t * d
    return w
