"""CPU references of the absolute pose fix (ekf_observe_pose) -- TEST INFRASTRUCTURE ONLY.

Neither the structured oracle (oracle/ekf_oracle.cpp) nor the extended-precision reference (tests/hp_reference.py) has
a pose fix of its own; this module applies one to each of them, from outside, on their state.

``oracle_observe_pose`` -- the fix written as the reference would write it in Robot.cpp with its GSL pattern (the pattern
    of Robot.cpp:516-602), applied in float64 to the structured oracle's full n x n matrix through its y / P views:
    PHt = P H' (NT), S = H P H' + R_sel, S^-1 by gsl_linalg_LU_decomp + LU_invert on the d x d block, d2 = v' S^-1 v (TN
    then NN as at :479-483), K = PHt S^-1 and KS = K S (NN, zero skip), P -= KS K' (NT), y += K v (NN, zero skip),
    normalize_radian(y[2]); the pose follows y[0:3].  numpy evaluates every elementwise operation with one IEEE rounding
    and no contraction, in the loop order written here.

``hp_observe_pose`` -- the same fix on an hp_reference.HPFilter in longdouble, with magnitudes formed as in
    HPFilter._update (from the absolute values of the current quantities).  The gain enters the filter's term list as the
    library's two rank-2 terms, (K_0, K_1) and (K_2, 0), in that order.  Its depth, counted from the operation counts of
    the kernels in the style of hp_reference's docstring:

    one absolute pose fix           DEPTH_POSE     = 44  S = P_sel + R (1), 3x3 LU (6: pivot quotient, two eliminations)
                                                         and its inverse (12: forward 4, back 8), K = P H' S^-1 (3
                                                         terms: 4), K S (4), the two rank-2 terms (2 x 4), v = z - y
                                                         (1) and its wrap (2), y += K v (4), the wrap of y[2] (2)

Both return status 1 (accepted: S nonsingular and d2 <= d2_max), 0 (rejected) or 2 (S singular); only an accepted fix
changes the state.
"""
import math

import numpy as np

import hp_reference as hp

LD = np.longdouble
DEPTH_POSE = 44
TWO_PI = 2.0 * math.pi


def selection(mask):
    return [c for c in range(3) if int(mask) & (1 << c)]


def normalize_radian(rad):
    """Robot.cpp:62-71 in double (C++ parses floor(..)*2.0*M_PI as (floor(..)*2.0)*M_PI)."""
    if rad > math.pi:
        return rad - (TWO_PI + math.floor(rad / TWO_PI) * 2.0 * math.pi)
    if rad < -math.pi:
        return rad + (TWO_PI + math.floor(abs(rad) / TWO_PI) * 2.0 * math.pi)
    return rad


def lu_inverse(S):
    """gsl_linalg_LU_decomp (first-largest partial pivot, elimination skipped on a zero pivot) + LU_invert on a d x d
    list of floats.  Returns (S^-1 as a d x d list, singular)."""
    d = len(S)
    a = [list(map(float, row)) for row in S]
    p = list(range(d))
    for j in range(d - 1):
        mx, piv = abs(a[j][j]), j
        for i in range(j + 1, d):
            if abs(a[i][j]) > mx:
                mx, piv = abs(a[i][j]), i
        if piv != j:
            a[j], a[piv] = a[piv], a[j]
            p[j], p[piv] = p[piv], p[j]
        ajj = a[j][j]
        if ajj != 0.0:
            for i in range(j + 1, d):
                l = a[i][j] / ajj
                a[i][j] = l
                for k in range(j + 1, d):
                    a[i][k] = a[i][k] - l * a[j][k]
    if any(a[i][i] == 0.0 for i in range(d)):
        return [[0.0] * d for _ in range(d)], True
    Si = [[0.0] * d for _ in range(d)]
    for col in range(d):
        x = [1.0 if p[i] == col else 0.0 for i in range(d)]
        for i in range(1, d):                                    # unit lower triangle
            s = x[i]
            for k in range(i):
                s -= a[i][k] * x[k]
            x[i] = s
        x[d - 1] = x[d - 1] / a[d - 1][d - 1]                   # upper triangle
        for i in range(d - 2, -1, -1):
            s = x[i]
            for k in range(i + 1, d):
                s -= a[i][k] * x[k]
            x[i] = s / a[i][i]
        for i in range(d):
            Si[i][col] = x[i]
    return Si, False


def _skip_axpy(acc, t, b):
    """acc += t * b where t != 0 (the reference-BLAS zero skip), elementwise."""
    return np.where(t != 0.0, acc + t * b, acc)


def oracle_observe_pose(o, z, R, mask=7, d2_max=math.inf, rows_per=512):
    """The fix on a StructuredOracle `o`.  Returns (status, d2, S (d x d), v (d))."""
    z = [float(v) for v in np.asarray(z, np.float64).reshape(3)]
    R = np.asarray(R, np.float64).reshape(3, 3)
    sel = selection(mask)
    d = len(sel)
    n, nl = o.n, 3 + 2 * o.lines
    y = np.ctypeslib.as_array(o._lib.ekfo_y_ptr(o._h), shape=(n,))
    P = o.P_view()
    S = [[(0.0 + (0.0 + float(P[r, c]) * 1.0)) + float(R[r, c]) for c in sel] for r in sel]   # H P (NN), (H P) H' (NT), + R
    Si, singular = lu_inverse(S)
    v = [z[c] - float(y[c]) for c in sel]
    v = [normalize_radian(vi) if c == 2 else vi for vi, c in zip(v, sel)]
    w = [0.0] * d                                                 # v' S^-1 (TN)
    for k in range(d):
        for c in range(d):
            if v[k] != 0.0:
                w[c] += v[k] * Si[k][c]
    d2 = 0.0                                                      # (NN)
    for c in range(d):
        if w[c] != 0.0:
            d2 += w[c] * v[c]
    if singular:
        return 2, d2, np.array(S), np.array(v)
    if not d2 <= d2_max:
        return 0, d2, np.array(S), np.array(v)
    ph = [0.0 + P[:nl, c] * 1.0 for c in sel]                     # P H' (NT), one structural 1 per column
    K = [np.zeros(nl) for _ in range(d)]
    for i in range(d):                                            # PHt S^-1 (NN)
        for c in range(d):
            K[c] = _skip_axpy(K[c], ph[i], Si[i][c])
    KS = [np.zeros(nl) for _ in range(d)]
    for i in range(d):                                            # K S (NN)
        for c in range(d):
            KS[c] = _skip_axpy(KS[c], K[i], S[i][c])
    for r0 in range(0, nl, rows_per):                             # P -= KS K' (NT, full matrix)
        r1 = min(nl, r0 + rows_per)
        t = np.zeros((r1 - r0, nl))
        for k in range(d):
            t = t + KS[k][r0:r1, None] * K[k][None, :]
        P[r0:r1, :nl] -= (0.0 + t)
    t = np.zeros(nl)                                              # y += K v (NN)
    for k in range(d):
        t = _skip_axpy(t, K[k], v[k])
    y[:nl] += t
    y[2] = normalize_radian(float(y[2]))
    o.set_pose(y[:3].copy())                                      # (x_pre: the next prediction overwrites it unread)
    return 1, d2, np.array(S), np.array(v)


def hp_observe_pose(ref, z, R, mask=7, d2_max=math.inf):
    """The fix on an hp_reference.HPFilter `ref`.  Returns (status, d2)."""
    sel = selection(mask)
    d, n, nl = len(sel), ref.n, ref.nl
    z = np.asarray(z, np.float64).reshape(3); Rm = np.asarray(R, np.float64).reshape(3, 3)
    PH, _ = ref.block(np.arange(nl), sel)                          # P H' = the selected columns of P
    S = PH[sel] + Rm[np.ix_(sel, sel)].astype(LD); aS = hp._f(S)
    if np.linalg.det(np.asarray(S, np.float64)) == 0:
        return 2, 0.0
    Si = np.linalg.inv(np.asarray(S, np.float64)).astype(LD)      # refined in extended precision
    for _ in range(3):
        Si = Si + Si @ (np.eye(d, dtype=LD) - S @ Si)
    v = z[sel].astype(LD) - ref.y[sel]; mv = np.abs(z[sel]) + hp._f(ref.y[sel])
    for i, c in enumerate(sel):
        if c == 2:
            v[i], wc = hp.normalize_radian(v[i]); mv[i] += float(wc)
    d2 = v @ Si @ v
    if not d2 <= LD(d2_max):
        return 0, float(d2)
    aSi, aPH = hp._f(Si), hp._f(PH)
    K = np.zeros((n, d), LD); mK = np.zeros((n, d))
    K[:nl] = PH @ Si
    mK[:nl] = aPH @ aSi + aPH @ (aSi @ aS @ aSi)
    KS = K @ S; mKS = mK @ aS
    ref.T = ref.T - KS[:3] @ K.T
    ref.mT = ref.mT + mKS[:3] @ mK.T
    pad = [np.zeros((n, 4), b.dtype) for b in (K, KS, mK, mKS)]
    for p, b in zip(pad, (K, KS, mK, mKS)):
        p[:, :d] = b
    ref._add_term(*(p[:, :2] for p in pad))
    if d == 3:
        ref._add_term(*(p[:, 2:] for p in pad))
    ref.y = ref.y + K @ v
    ref.my = ref.my + mK @ hp._f(v) + hp._f(K) @ mv
    ref.y[2], cw = hp.normalize_radian(ref.y[2]); ref.my[2] += float(cw)
    ref.pose = ref.y[:3].copy(); ref.mpose = ref.my[:3].copy()
    ref.xp = ref.y[:3].copy(); ref.mxp = ref.my[:3].copy()
    ref.depth += DEPTH_POSE
    return 1, float(d2)
