"""Float32 model of K11 (csrc/ewk_align.cuh): dynamic time warping of a segment's MFCC frames against a template's.

The device's arithmetic, operation for operation, so that the model matches it bit for bit:
    u_i[c] = f_i[c] - mean[c]                  (c < C, the context's n_mfcc; frames and mean as K3 / ewk_extract_mfcc give them)
    uu_i   = fma chain over c from +0 of u_i[c] * u_i[c];  r_i = 1 / sqrt(uu_i) if uu_i > 0 else 0   (template: v_j, s_j)
    dot_ij = fma chain over c from +0 of u_i[c] * v_j[c];  cost_ij = 1 - (dot_ij * r_i) * s_j
    D_00 = cost_00;  D_i0 = D_{i-1,0} + cost_i0;  D_0j = D_{0,j-1} + cost_0j
    D_ij = cost_ij + fmin(fmin(D_{i-1,j-1}, D_{i-1,j}), D_{i,j-1})
    distance = D_{n-1,m-1} / (n + m)
Every operation is rounded to float32 once (numpy's float32 +, -, *, /, sqrt are correctly rounded; fmaf32 is C's fmaf).
The DP is vectorised along anti-diagonals: every cell of a diagonal depends only on the two diagonals before it.
"""
from __future__ import annotations

import numpy as np

from .resample_restated import fmaf32

F32 = np.float32


def normalise(frames, mean, C):
    """(u [n, C], r [n]) of frames [n, >= C] and mean [>= C]."""
    u = (np.asarray(frames, F32)[:, :C] - np.asarray(mean, F32)[:C]).astype(F32)
    uu = np.zeros(len(u), F32)
    for c in range(C):
        uu = fmaf32(u[:, c], u[:, c], uu)
    with np.errstate(divide="ignore"):
        r = np.where(uu > 0, F32(1) / np.sqrt(uu), F32(0)).astype(F32)
    return u, r


def cost_matrix(u, r, v, s):
    """cost [n, m] = 1 - (dot * r_i) * s_j with dot the serial fma chain over c."""
    dot = np.zeros((len(u), len(v)), F32)
    for c in range(u.shape[1]):
        dot = fmaf32(u[:, c][:, None], v[:, c][None, :], dot)
    return (F32(1) - (dot * r[:, None]).astype(F32) * s[None, :]).astype(F32)


def accumulate(cost):
    """D_{n-1,m-1} of the DP over cost [n, m], anti-diagonal by anti-diagonal (float32)."""
    n, m = cost.shape
    prev2 = prev1 = None          # diagonals d-2 and d-1, indexed by i
    for d in range(n + m - 1):
        i = np.arange(max(0, d - m + 1), min(n, d + 1))
        j = d - i
        c = cost[i, j]
        cur = np.empty(n, F32)
        if d == 0:
            cur[0] = c[0]                                              # D_00
        else:
            out = np.empty(len(i), F32)
            top, left = i == 0, j == 0                                 # row 0 / column 0
            inner = ~top & ~left
            out[top] = prev1[0] + c[top]                               # D_{0,j-1} + cost
            out[left] = prev1[i[left] - 1] + c[left]                   # D_{i-1,0} + cost
            ii = i[inner]
            if ii.size:
                out[inner] = c[inner] + np.fmin(np.fmin(prev2[ii - 1], prev1[ii - 1]), prev1[ii])
            cur[i] = out
        prev2, prev1 = prev1, cur
    return prev1[n - 1]


def distance(seg_frames, seg_mean, tmpl_frames, tmpl_mean, C=20):
    """K11's distance of one segment against one template (float32)."""
    u, r = normalise(seg_frames, seg_mean, C)
    v, s = normalise(tmpl_frames, tmpl_mean, C)
    D = accumulate(cost_matrix(u, r, v, s))
    return F32(D / F32(len(u) + len(v)))


def distance_loop(seg_frames, seg_mean, tmpl_frames, tmpl_mean, C=20):
    """The same, cell by cell in scalar float32: the statement the vectorised model is checked against."""
    f, g = np.asarray(seg_frames, F32), np.asarray(tmpl_frames, F32)
    mu, mv = np.asarray(seg_mean, F32), np.asarray(tmpl_mean, F32)

    def norm(x, mean):
        rows = []
        for row in x:
            uc = [F32(row[c] - mean[c]) for c in range(C)]
            acc = F32(0)
            for a in uc:
                acc = F32(fmaf32(a, a, acc))
            rows.append((uc, F32(F32(1) / np.sqrt(acc)) if acc > 0 else F32(0)))
        return rows

    U, V = norm(f, mu), norm(g, mv)
    n, m = len(U), len(V)
    D = [[F32(0)] * m for _ in range(n)]
    for i in range(n):
        for j in range(m):
            dot = F32(0)
            for c in range(C):
                dot = F32(fmaf32(U[i][0][c], V[j][0][c], dot))
            cost = F32(F32(1) - F32(F32(dot * U[i][1]) * V[j][1]))
            if i == 0 and j == 0:
                D[i][j] = cost
            elif i == 0:
                D[i][j] = F32(D[0][j - 1] + cost)
            elif j == 0:
                D[i][j] = F32(D[i - 1][0] + cost)
            else:
                D[i][j] = F32(cost + np.fmin(np.fmin(D[i - 1][j - 1], D[i - 1][j]), D[i][j - 1]))
    return F32(D[n - 1][m - 1] / F32(n + m))


def distance_f64(seg_frames, seg_mean, tmpl_frames, tmpl_mean, C=20):
    """The same definition in float64 (no pinned rounding): the reference the float32 statement approximates."""
    u = np.asarray(seg_frames, np.float64)[:, :C] - np.asarray(seg_mean, np.float64)[:C]
    v = np.asarray(tmpl_frames, np.float64)[:, :C] - np.asarray(tmpl_mean, np.float64)[:C]
    nu, nv = np.linalg.norm(u, axis=1), np.linalg.norm(v, axis=1)
    r = np.where(nu > 0, 1 / np.where(nu > 0, nu, 1), 0)
    s = np.where(nv > 0, 1 / np.where(nv > 0, nv, 1), 0)
    cost = 1 - (u @ v.T) * r[:, None] * s[None, :]
    n, m = cost.shape
    D = np.full((n, m), np.inf)
    for i in range(n):
        for j in range(m):
            if i == 0 and j == 0:
                D[i, j] = cost[i, j]
            else:
                D[i, j] = cost[i, j] + min(D[i - 1, j - 1] if i and j else np.inf, D[i - 1, j] if i else np.inf,
                                           D[i, j - 1] if j else np.inf)
    return D[n - 1, m - 1] / (n + m)
