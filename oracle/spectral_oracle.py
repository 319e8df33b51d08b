"""fp64 reference of the spectral step of one recursion node: the Fiedler pair of the normalised Laplacian and the
exact 1-D 2-means of its embedding, with the definitions the kernels use (csrc/spectral_dev.cuh:two_means_1d_body,
csrc/small.cu), computed plainly in float64 with no attempt to follow the GPU's order of summation.

Test infrastructure only (see oracle/__init__.py)."""

from __future__ import annotations

import numpy as np

DENSE_MAX = 1500  # dense eigh up to this size, Lanczos (ARPACK) above


def normalized_operator(W: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """N = D^-1/2 W D^-1/2 and s = sqrt(d), with an isolated vertex scaled by 1 (scipy's csgraph.laplacian rule)."""
    A = np.array(W, dtype=np.float64)
    np.fill_diagonal(A, 0.0)
    d = A.sum(axis=0)
    s = np.where(d == 0, 1.0, np.sqrt(d))
    return A / s[:, None] / s[None, :], s


def fiedler_reference(W: np.ndarray, dense: bool | None = None) -> tuple[float, float, np.ndarray]:
    """(lambda_2, lambda_3, u = x_2 / sqrt(d)) of L = I - D^-1/2 W D^-1/2: dense ``eigh`` up to DENSE_MAX vertices,
    ``eigsh`` on N (largest three, tol 1e-14, fixed start vector) above; ``dense`` forces one of the two.  lambda_3
    is NaN for m = 2."""
    m = W.shape[0]
    N, s = normalized_operator(W)
    if dense if dense is not None else m <= DENSE_MAX:
        from scipy.linalg import eigh

        k = min(3, m)
        vals, vecs = eigh(np.eye(m) - N, subset_by_index=(0, k - 1))
        lam3 = float(vals[2]) if k > 2 else float("nan")
        return float(vals[1]), lam3, vecs[:, 1] / s
    from scipy.sparse.linalg import eigsh

    vals, vecs = eigsh(N, k=3, which="LA", tol=1e-14, v0=np.ones(m))
    order = np.argsort(-vals)
    vals, vecs = vals[order], vecs[:, order]
    return float(1.0 - vals[1]), float(1.0 - vals[2]), vecs[:, 1] / s


def two_means_1d(u: np.ndarray) -> dict:
    """Exact 2-means of the Fiedler coordinate ``u`` (m >= 3), as the kernels define it.

    * sign: the entry of largest magnitude (smallest index on ties) is made positive;
    * best split after ``best`` sorted keys: maximises P^2/i + (S-P)^2/(m-i) over the centred prefix sums, smallest
      i on ties;
    * margin: the cut's two neighbouring keys to the midpoint of the two centroids, over the range of the keys;
    * stable splits: splits that Lloyd's iteration leaves unchanged (key[i-1] < midpoint < key[i]); runner-up: the
      best score of the other stable splits over the optimum's (0 if there is none);
    * side: ``u >= sorted[best]``.

    Also returns ``closest``: the smallest distance of a key to any split's centroid midpoint, over the range --
    where it is tiny, the stable count depends on rounding."""
    u = np.asarray(u, dtype=np.float64)
    m = len(u)
    arg = int(np.argmax(np.abs(u)))  # first index of the maximum
    if u[arg] < 0:
        u = -u
    keys = np.sort(u)
    mean = u.mean()
    c = keys - mean
    prefix = np.cumsum(c)[:-1]
    total = c.sum()
    cnt = np.arange(1, m)
    score = prefix**2 / cnt + (total - prefix) ** 2 / (m - cnt)
    best = int(np.argmax(score)) + 1
    mids = mean + 0.5 * (prefix / cnt + (total - prefix) / (m - cnt))
    stable = (keys[:-1] < mids) & (mids < keys[1:])
    others = stable.copy()
    others[best - 1] = False
    runner = float(score[others].max() / score[best - 1]) if others.any() and score[best - 1] > 0 else 0.0
    rng = max(keys[-1] - keys[0], 1e-300)
    mid = mids[best - 1]
    margin = min(abs(keys[best - 1] - mid), abs(keys[best] - mid)) / rng
    closest = float(np.min(np.minimum(np.abs(keys[:-1] - mids), np.abs(keys[1:] - mids))) / rng)
    return {
        "u": u,
        "sorted": keys,
        "best": best,
        "score": score,
        "margin": float(margin),
        "stable_splits": int(stable.sum()),
        "runner_up": runner,
        "side": (u >= keys[best]).astype(np.int32),
        "closest": closest,
    }
