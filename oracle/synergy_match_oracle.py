"""CPU oracle for matched cosine similarity of synergy sets.  TEST INFRASTRUCTURE ONLY.

What a user of the synergy literature writes in numpy + scipy to compare two sets of synergies of the same rank:
every synergy vector (row) scaled to unit length - a row whose norm is 0 stays 0, so it has similarity 0 with
everything -, S = the k x k matrix of scalar products, the pairing `scipy.optimize.linear_sum_assignment(S,
maximize=True)`, and the mean of the matched similarities.  `brute_force` searches every permutation (small k) for
the tests that pin the optimum.
"""
import itertools

import numpy as np
from scipy.optimize import linear_sum_assignment


def unit_rows(H):
    H = np.asarray(H, dtype=np.float64)
    with np.errstate(over="ignore"):
        norms = np.linalg.norm(H, axis=1)  # a squared norm that overflows gives inf: the row becomes 0
    out = np.zeros_like(H)
    nz = norms > 0
    out[nz] = H[nz] / norms[nz, None]
    return out


def similarity(A, B):
    """S[i][j] = <a_i, b_j> / (||a_i|| ||b_j||), 0 where either row is zero."""
    return unit_rows(A) @ unit_rows(B).T


def match(A, B):
    """Returns (mean, sim, perm): perm[i] is the row of B paired with row i of A, sim[i] their similarity."""
    S = similarity(A, B)
    rows, cols = linear_sum_assignment(S, maximize=True)
    perm = np.empty(len(rows), dtype=np.int64)
    perm[rows] = cols
    sim = S[np.arange(len(perm)), perm]
    return float(sim.mean()), sim, perm


def brute_force(S):
    """The largest summed similarity over all permutations of the columns of S."""
    k = S.shape[0]
    perms = np.array(list(itertools.permutations(range(k))))
    return float(S[np.arange(k), perms].sum(axis=1).max())
