"""float64 numpy restatement of the exact marginal likelihood (grf_b200/mll.py) and of the per-length training Gram
it is built on (PhiBlocks.training_gram, csrc/grf_gram.cu).

E[l n + i, l' n + j] = <M_l[x_i], M_l'[x_j]> over the float32 values of the per-length blocks.  A product of two
float32 values is exact in float64, so E differs from the exact value only in how its sums round: with k[R, C] the
number of columns rows R and C share and P[R, C] = sum_s |A[R, s] A[C, s]|, any float64 summation order is within
k u P of it (u = 2^-53), so two orders are within 2 k u P = 2^-52 k P of each other (gram_bound)."""

import numpy as np
import scipy.sparse as sp


def stacked_rows(mats, x):
    """A (scipy CSR, float64 [L n, N]) from the per-length scipy blocks M_l (float32 values) at the training ids x."""
    x = np.asarray(x, np.int64)
    return sp.vstack([m.astype(np.float32).astype(np.float64).tocsr()[x] for m in mats]).tocsr()


def gram(mats, x):
    a = stacked_rows(mats, x)
    return (a @ a.T).toarray()


def gram_bound(mats, x):
    a = abs(stacked_rows(mats, x))
    nz = a.copy()
    nz.data[:] = 1.0
    return 2.0 ** -52 * np.maximum((nz @ nz.T).toarray(), 1.0) * (a @ a.T).toarray()


def gram_split(mats, x, T):
    """E the way the device builds it: the upper triangle's light slots (t_s <= T) summed per cell in ascending
    column order, plus the dense H H^T of the heavy slots, then the upper triangle mirrored.  Returns (E, h, p_light)."""
    a = stacked_rows(mats, x).toarray()
    t = (a != 0).sum(axis=0)
    touched = t > 0
    heavy = touched & (t > T)
    light = touched & ~heavy
    al = a[:, light]
    e = np.zeros((a.shape[0], a.shape[0]))
    for s in range(al.shape[1]):                  # ascending column: the light kernel's order per cell
        nz = np.nonzero(al[:, s])[0]
        v = al[nz, s]
        e[np.ix_(nz, nz)] += np.outer(v, v)
    ah = a[:, heavy]
    e += ah @ ah.T
    iu = np.triu_indices(e.shape[0], 1)
    e[iu[1], iu[0]] = e[iu]
    return e, int(heavy.sum()), int((t[light].astype(np.int64) ** 2).sum())


def kernel(E, f, noise):
    """K = sum_{l, b} f_l f_b E[l, :, b, :] + sigma^2 I from E [L, n, L, n]."""
    f = np.asarray(f, np.float64)
    return np.einsum("l,libj,b->ij", f, E, f) + noise * np.eye(E.shape[1])


def neg_mll(E, f, noise, y):
    """-mll / n, as neg_mll_backward normalises it."""
    n = E.shape[1]
    k = kernel(E, f, noise)
    c = np.linalg.cholesky(k)
    a = np.linalg.solve(k, y)
    return (0.5 * y @ a + np.log(np.diag(c)).sum() + 0.5 * n * np.log(2 * np.pi)) / n


def neg_mll_grad(E, f, noise, y):
    """Closed form: d(-mll/n)/df_l = -sum_b f_b <W, E_lb> / n, d(-mll/n)/dsigma^2 = -(a.a - tr K^-1) / (2 n),
    W = a a^T - K^-1, a = K^-1 y."""
    n = E.shape[1]
    k = kernel(E, f, noise)
    kinv = np.linalg.inv(k)
    a = kinv @ y
    w = np.outer(a, a) - kinv
    eb = np.einsum("libj,b->lij", E, np.asarray(f, np.float64))
    gf = np.einsum("lij,ij->l", eb, w)
    return -gf / n, -0.5 * (a @ a - np.trace(kinv)) / n
