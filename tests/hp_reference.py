"""Extended-precision reference of Robot::localize (slam_ros/Robot.cpp:126-943) with a running error bound.

Plain numpy in ``np.longdouble`` (64-bit mantissa on x86-64, quad on aarch64).  It follows the mathematics of the
operation -- prediction, gate with first fit, gain, update, augmentation, map reset -- not the rounding order of
the reference or of the kernels, and calls neither the oracle nor the library.

Cost O(n m) per matched line.  Gating and gains only read rows 0-2, the 2x2 diagonal blocks and two columns of P.
The map part of P (rows and columns >= 3) is never touched by the prediction, so after k matched lines

    P[i, j] = B[i, j] - sum_k KS_k[i] K_k[j]          (i, j >= 3)

where B is the uploaded covariance, or for a row appended by the augmentation its value when it was appended
(earlier terms are zero in rows that did not exist yet).  Rows 0-2 are kept explicitly.  Blocks of P are formed only
when a test asks for them.

Error bound.  Every quantity x carries a magnitude mag(x): the value of the same computation with every input and
intermediate replaced by its absolute value, with products as |a| mag(b) + mag(a) |b| and smooth functions as
|f(a)| + |f'(a)| mag(a).  For P_ij that is mag(B_ij) + sum_k mag(KS_k[i]) mag(K_k[j]), with
mag(K) = mag(P H') |S^-1| + |P H'| mag(S^-1), mag(S^-1) = |S^-1| |S| |S^-1| (the componentwise sensitivity
of an inverse, which carries the condition of S), and mag(K S) = mag(K) |S|.  Magnitudes are formed from the absolute
values of the current quantities, not from earlier magnitudes, so they do not compound from scan to scan.  A sum or a product
whose inputs are off by at most d u mag(input), evaluated with one more rounding, is off by at most (d + 1) u mag;
a 2x2 inverse adds its own backward error (a few u |S|) to mag(S); CUDA's sin / cos are within 2 ulp.  So a device
result x that took at most D dependent roundings from exactly known inputs satisfies, to first order,

    |x - ref| <= C u mag(x),   u = 2**-53,   C = D.

D is counted in the code (``depth``), per stage, from the operation counts of the kernels:
    prediction                      DEPTH_PREDICT  = 6   trig of theta + u/2 (3), F P F' + Fu Q Fu' (3)
    one matched line (gain, update) DEPTH_LINE     = 36  cos/sin of the landmark angle (3), P H' (4 terms: 4),
                                                         S = H P H' + R (5 terms + R: 6), 2x2 LU inverse (8),
                                                         K = P H' S^-1 (3), K S (3), y += K v (3),
                                                         P - KS K' (two FMAs; four roundings in the exact
                                                         variant and the oracle: 4) -- 34, plus 2 for the angle wrap
    one appended landmark           DEPTH_AUGMENT  = 10  trig of the world angle (3), r (3), Gx P Gx' + Gl R Gl' (4)
The reference's own rounding (2**-64 relative per operation) is far below that and is not counted.  D grows with
the number of dependent steps since the state was exactly known (an upload, or creation); a bound with a constant C
would not hold over a long run, and a C fitted to observed errors would prove nothing.
"""
import math

import numpy as np

LD = np.longdouble
U = 2.0 ** -53
TWO_PI = LD(2.0 * math.pi)        # the reference's 2.0 * M_PI: a double constant, and part of the operation
PI = LD(math.pi)

DEPTH_GAIN = 32
DEPTH_TERM = 4
DEPTH_PREDICT = 6
DEPTH_AUGMENT = 10


def require_precision():
    nm = np.finfo(LD).nmant
    assert nm >= 63, ("np.longdouble has a %d-bit mantissa on this platform; the componentwise reference needs at "
                      "least 63 (x86-64 extended or IEEE quad)" % nm)


def normalize_radian(a):
    """Robot.cpp:62-71 on a scalar; returns (value, constant added or subtracted)."""
    if a > PI:
        c = TWO_PI + LD(math.floor(a / TWO_PI)) * TWO_PI
        return a - c, abs(c)
    if a < -PI:
        c = TWO_PI + LD(math.floor(abs(a) / TWO_PI)) * TWO_PI
        return a + c, abs(c)
    return a, LD(0)


def normalize_radians(a):
    """normalize_radian on an array; returns (values, |constant| per entry as float64)."""
    c = np.where(a > PI, TWO_PI + np.floor(a / TWO_PI) * TWO_PI,
                 np.where(a < -PI, -(TWO_PI + np.floor(np.abs(a) / TWO_PI) * TWO_PI), LD(0)))
    return a - c, np.abs(c).astype(np.float64)


def _f(x):
    return np.abs(np.asarray(x, dtype=np.float64))


class HPFilter:
    """One filter.  All state values are np.longdouble; magnitudes are float64 (they only scale a bound)."""

    def __init__(self, capacity_lines, gate=0.4, encoder_noise=0.024, reset_headroom=10):
        require_precision()
        self.cap = int(capacity_lines)
        self.n = 3 + 2 * self.cap
        self.gate = float(gate)
        self.enc = float(encoder_noise)
        self.headroom = int(reset_headroom)
        self.margins = []            # |sqrt|d2| - gate| / gate of every evaluated pair
        self.depth = 1
        n = self.n
        y = np.zeros(n); P = np.zeros((n, n)); P[0, 0] = P[1, 1] = 0.05     # Robot.cpp:20-35
        self.upload(y, P, 0)

    # ---- state ------------------------------------------------------------------------------------------
    def upload(self, y, P, n_lines):
        """The state ekf_upload receives: y[n], P[n, n] (symmetric), n_lines.  Known exactly: depth 0."""
        n, L = self.n, int(n_lines)
        nl = 3 + 2 * L
        self.L = L
        self.y = np.zeros(n, LD); self.y[:nl] = np.asarray(y, np.float64)[:nl]
        self.my = np.zeros(n); self.my[:nl] = _f(self.y[:nl])
        self.pose = self.y[:3].copy(); self.mpose = self.my[:3].copy()
        self.xp = self.pose.copy(); self.mxp = self.mpose.copy()
        # only the live nl x nl part is kept (entries outside it read as zero; appended rows come from `aug`), so a
        # filter of large capacity costs memory in proportion to its uploaded map, not to n^2
        self.base = np.array(np.asarray(P, np.float64)[:nl, :nl])
        self.T = np.zeros((3, n), LD); self.T[:, :nl] = self.base[:3, :nl]
        self.mT = _f(self.T)
        self.aug = {}                # appended row -> (values over columns <= its pair, magnitudes)
        self._clear_terms()
        self.depth = DEPTH_GAIN

    def _clear_terms(self):
        self.nt = 0                  # number of pending-term columns (2 per matched line) in the buffers below
        self._tb = [np.zeros((self.n, 0), LD), np.zeros((self.n, 0), LD), np.zeros((self.n, 0)), np.zeros((self.n, 0))]

    def _base(self, r, c):
        """base[r][:, c] (index arrays), zero outside the uploaded live block."""
        nb = self.base.shape[0]
        out = np.zeros((r.size, c.size))
        ri = np.nonzero(r < nb)[0]; ci = np.nonzero(c < nb)[0]
        if ri.size and ci.size:
            out[np.ix_(ri, ci)] = self.base[np.ix_(r[ri], c[ci])]
        return out

    @property
    def C(self):
        return self.depth

    @property
    def nl(self):
        return 3 + 2 * self.L

    def _terms(self):
        """(K, KS, mag K, mag KS), n x 2k: the k pending terms in the order they were formed."""
        return tuple(b[:, :self.nt] for b in self._tb)

    def _add_term(self, K, KS, mK, mKS):
        if self.nt + 2 > self._tb[0].shape[1]:           # grow geometrically: appending stays O(n) per term
            w = max(16, 2 * self._tb[0].shape[1])
            grown = []
            for b in self._tb:
                g = np.zeros((self.n, w), b.dtype); g[:, :self.nt] = b[:, :self.nt]
                grown.append(g)
            self._tb = grown
        for b, v in zip(self._tb, (K, KS, mK, mKS)):
            b[:, self.nt:self.nt + 2] = v
        self.nt += 2

    def block(self, rows, cols):
        """(value, magnitude) of P[rows][:, cols] (index arrays or ranges)."""
        r = np.asarray(rows, dtype=np.int64).reshape(-1); c = np.asarray(cols, dtype=np.int64).reshape(-1)
        val = self._base(r, c).astype(LD)
        for l, (v, mv) in sorted(self.aug.items()):
            ri = np.nonzero(r == l)[0]; ci = np.nonzero(c == l)[0]
            if ri.size:
                sel = c <= l
                val[np.ix_(ri, np.nonzero(sel)[0])] = v[c[sel]]
            if ci.size:
                sel = r <= l
                val[np.ix_(np.nonzero(sel)[0], ci)] = v[r[sel]][:, None]
        mag = _f(val)
        for l, (v, mv) in self.aug.items():
            ri = np.nonzero(r == l)[0]; ci = np.nonzero(c == l)[0]
            if ri.size:
                sel = c <= l
                mag[np.ix_(ri, np.nonzero(sel)[0])] = mv[c[sel]]
            if ci.size:
                sel = r <= l
                mag[np.ix_(np.nonzero(sel)[0], ci)] = mv[r[sel]][:, None]
        K, KS, mK, mKS = self._terms()
        if K.shape[1]:
            val -= KS[r] @ K[c].T
            mag += mKS[r] @ mK[c].T
        for t in range(3):                                   # rows / columns 0-2 are explicit
            ri = np.nonzero(r == t)[0]; ci = np.nonzero(c == t)[0]
            if ri.size:
                val[ri, :] = self.T[t, c]; mag[ri, :] = self.mT[t, c]
            if ci.size:
                val[:, ci] = self.T[t, r][:, None]; mag[:, ci] = self.mT[t, r][:, None]
        return val, mag

    def live(self):
        nl = self.nl
        Pv, Pm = self.block(np.arange(nl), np.arange(nl))
        return self.y[:nl].copy(), self.my[:nl].copy(), Pv, Pm

    def _diag_blocks(self, js):
        """P[a,a], P[a,b], P[b,b] (values and magnitudes) of landmarks js."""
        a = 3 + 2 * np.asarray(js, np.int64); b = a + 1
        out = []
        for p, q in ((a, a), (a, b), (b, b)):
            nb = self.base.shape[0]
            inb = (p < nb) & (q < nb)
            v = np.zeros(p.size, LD); v[inb] = self.base[p[inb], q[inb]]; m = _f(v)
            hi = np.maximum(p, q); lo = np.minimum(p, q)
            for key, (av, am) in self.aug.items():
                i = np.nonzero(hi == key)[0]
                v[i] = av[lo[i]]; m[i] = am[lo[i]]
            K, KS, mK, mKS = self._terms()
            if K.shape[1]:
                v = v - np.sum(KS[p] * K[q], axis=1)
                m = m + np.sum(mKS[p] * mK[q], axis=1)
            out.append((v, m))
        return out

    # ---- Robot.cpp:148-258 ------------------------------------------------------------------------------
    def predict(self, u):
        u = np.asarray(u, np.float64).astype(LD)
        x, mx = self.pose, self.mpose
        ang = x[2] + u[2] / 2; mang = mx[2] + float(abs(u[2] / 2))
        ca, sa = np.cos(ang), np.sin(ang)
        mca = float(abs(ca)) + float(abs(sa)) * mang; msa = float(abs(sa)) + float(abs(ca)) * mang
        au0 = float(abs(u[0]))
        self.xp = np.array([x[0] + u[0] * ca, x[1] + u[0] * sa, x[2] + u[2]], LD)
        self.mxp = np.array([mx[0] + au0 * mca, mx[1] + au0 * msa, mx[2] + float(abs(u[2]))])
        F02, F12 = -u[0] * sa, u[0] * ca
        mF02, mF12 = au0 * msa, au0 * mca
        T, mT = self.T, self.mT
        T0 = T[0] + F02 * T[2]; T1 = T[1] + F12 * T[2]
        mT0 = mT[0] + float(abs(F02)) * mT[2] + mF02 * _f(T[2])
        mT1 = mT[1] + float(abs(F12)) * mT[2] + mF12 * _f(T[2])
        T = np.stack([T0, T1, T[2].copy()]); mT = np.stack([mT0, mT1, mT[2].copy()])
        # the 3x3 corner gets F on the right as well (P_pre = T Fx')
        c0 = T[:, 0] + T[:, 2] * F02; c1 = T[:, 1] + T[:, 2] * F12
        mc0 = mT[:, 0] + mT[:, 2] * float(abs(F02)) + _f(T[:, 2]) * mF02
        mc1 = mT[:, 1] + mT[:, 2] * float(abs(F12)) + _f(T[:, 2]) * mF12
        T[:, 0] = c0; T[:, 1] = c1; mT[:, 0] = mc0; mT[:, 1] = mc1
        q = LD(self.enc) * (1 - 1 / (1 + abs(u[0])))
        Fu = np.array([[ca, 0, -u[0] * sa / 2], [sa, 1, u[0] * ca / 2], [0, 0, 1]], LD)
        mFu = np.array([[mca, 0, au0 * msa / 2], [msa, 0, au0 * mca / 2], [0, 0, 0]])
        Q = np.diag(np.array([q, 2 * q, q], LD))
        T[:, :3] += Fu @ Q @ Fu.T
        aF = _f(Fu)
        mq = self.enc * (1 + float(1 / (1 + abs(u[0]))))          # 1 - 1/(1+|u|) cancels: its magnitude is 1 + ...
        aQ = np.diag([mq, 2 * mq, mq])
        mT[:, :3] += aF @ aQ @ aF.T + mFu @ aQ @ aF.T + aF @ aQ @ mFu.T
        self.T, self.mT = T, mT
        self.matched = set()
        self.extra = []
        self.matches = 0
        self.depth += DEPTH_PREDICT

    # ---- Robot.cpp:367-489 for every unmatched landmark at once --------------------------------------------
    def gates(self, z, R):
        """(js, d2, rec) for every landmark not matched in this scan, in index order."""
        js = np.array([j for j in range(self.L) if j not in self.matched], np.int64)
        if js.size == 0:
            return js, np.zeros(0, LD), None
        a = 3 + 2 * js; b = a + 1
        y, my, xp, mxp = self.y, self.my, self.xp, self.mxp
        c, s = np.cos(y[a]), np.sin(y[a])
        g = xp[0] * s - xp[1] * c
        (daa, _), (dab, _), (dbb, _) = self._diag_blocks(js)
        T = self.T
        k = js.size
        C5 = np.zeros((k, 5, 5), LD)
        C5[:, :3, :3] = T[:, :3]
        for r in range(3):
            C5[:, r, 3] = C5[:, 3, r] = T[r, a]; C5[:, r, 4] = C5[:, 4, r] = T[r, b]
        C5[:, 3, 3] = daa; C5[:, 3, 4] = C5[:, 4, 3] = dab; C5[:, 4, 4] = dbb
        H = np.zeros((k, 2, 5), LD)
        H[:, 0, 2] = -1; H[:, 0, 3] = 1
        H[:, 1, 0] = -c; H[:, 1, 1] = -s; H[:, 1, 3] = g; H[:, 1, 4] = 1
        Rm = np.asarray(R, np.float64).reshape(2, 2)
        S = H @ C5 @ np.swapaxes(H, 1, 2) + Rm.astype(LD)
        det = S[:, 0, 0] * S[:, 1, 1] - S[:, 0, 1] * S[:, 1, 0]
        Si = np.empty_like(S)
        Si[:, 0, 0] = S[:, 1, 1] / det; Si[:, 1, 1] = S[:, 0, 0] / det
        Si[:, 0, 1] = -S[:, 0, 1] / det; Si[:, 1, 0] = -S[:, 1, 0] / det
        z = np.asarray(z, np.float64).astype(LD)
        h0, cw = normalize_radians(y[a] - xp[2])
        mh0 = _f(y[a]) + _f(xp[2]) + cw
        ca_, sa_ = c, s
        h1 = y[b] - (xp[0] * ca_ + xp[1] * sa_)
        mh1 = _f(y[b]) + _f(xp[0] * ca_) + _f(xp[1] * sa_) + (_f(xp[0] * sa_) + _f(xp[1] * ca_)) * _f(y[a])
        v0 = z[0] - h0; v1 = z[1] - h1
        mv0 = float(abs(z[0])) + mh0; mv1 = float(abs(z[1])) + mh1
        dn = np.abs(v0 - TWO_PI) < np.abs(v0)                       # Robot.cpp:471-475
        up = ~dn & (np.abs(v0 + TWO_PI) < np.abs(v0))
        v0 = np.where(dn, v0 - TWO_PI, np.where(up, v0 + TWO_PI, v0))
        mv0 = mv0 + np.where(dn | up, float(TWO_PI), 0.0)
        d2 = v0 * (Si[:, 0, 0] * v0 + Si[:, 1, 0] * v1) + v1 * (Si[:, 0, 1] * v0 + Si[:, 1, 1] * v1)
        rec = dict(js=js, c=c, s=s, g=g, S=S, Si=Si, v=np.stack([v0, v1], 1),
                   mv=np.stack([mv0, mv1], 1), det=det)
        return js, d2, rec

    def _first_fit(self, z, R):
        js, d2, rec = self.gates(z, R)
        gate = LD(self.gate)
        for i in range(js.size):
            if rec["det"][i] == 0:
                continue
            d = np.sqrt(abs(d2[i]))
            if math.isfinite(self.gate) and self.gate > 0:
                self.margins.append(float(abs(d - gate) / gate))
            if not (d > gate):
                return int(js[i]), i, rec
        return -1, -1, rec

    # ---- Robot.cpp:516-602 ------------------------------------------------------------------------------
    def _update(self, j, i, rec):
        n, nl = self.n, self.nl
        a, b = 3 + 2 * j, 4 + 2 * j
        cols, mcols = self.block(np.arange(nl), [0, 1, 2, a, b])
        c, s, g = rec["c"][i], rec["s"][i], rec["g"][i]
        P0, P1, P2, Pa, Pb = cols.T
        ph0 = Pa - P2; mph0 = _f(Pa) + _f(P2)
        ph1 = -c * P0 - s * P1 + g * Pa + Pb
        mph1 = float(abs(c)) * _f(P0) + float(abs(s)) * _f(P1) + float(abs(g)) * _f(Pa) + _f(Pb)
        PH = np.zeros((n, 2), LD); mPH = np.zeros((n, 2))
        PH[:nl, 0] = ph0; PH[:nl, 1] = ph1; mPH[:nl, 0] = mph0; mPH[:nl, 1] = mph1
        Si, S = rec["Si"][i], rec["S"][i]
        K = PH @ Si; mK = mPH @ _f(Si) + _f(PH) @ (_f(Si) @ _f(S) @ _f(Si))
        KS = K @ S; mKS = mK @ _f(S)
        v, mv = rec["v"][i], rec["mv"][i]
        # rows 0-2 explicitly, the rest through the term list
        self.T = self.T - KS[:3] @ K.T
        self.mT = self.mT + mKS[:3] @ mK.T
        self._add_term(K, KS, mK, mKS)
        self.y[:3] = self.xp; self.my[:3] = self.mxp
        self.y = self.y + K @ v
        self.my = self.my + mK @ _f(v) + _f(K) @ mv
        self.y[2], cw = normalize_radian(self.y[2]); self.my[2] += float(cw)
        self.pose = self.y[:3].copy(); self.mpose = self.my[:3].copy()
        self.xp = self.y[:3].copy(); self.mxp = self.my[:3].copy()
        self.depth += DEPTH_TERM

    # ---- Robot.cpp:792-866 ------------------------------------------------------------------------------
    def _augment(self, z, R):
        n, L = self.n, self.L
        l = 3 + 2 * L
        alfa, r = LD(float(z[0])), LD(float(z[1]))
        ca0, sa0 = np.cos(alfa), np.sin(alfa)
        p, mp = self.pose, self.mpose
        r = r + (p[0] * ca0 + p[1] * sa0)
        mr = float(abs(z[1])) + mp[0] * float(abs(ca0)) + float(abs(p[0] * ca0)) + mp[1] * float(abs(sa0)) + \
            float(abs(p[1] * sa0))
        alfa = alfa + p[2]; malfa = float(abs(z[0])) + mp[2]
        cw, sw = np.cos(alfa), np.sin(alfa)
        mcw = float(abs(cw)) + float(abs(sw)) * malfa; msw = float(abs(sw)) + float(abs(cw)) * malfa
        gl = self.y[1] * cw - self.y[0] * sw
        mgl = self.my[1] * float(abs(cw)) + float(abs(self.y[1])) * mcw + self.my[0] * float(abs(sw)) + \
            float(abs(self.y[0])) * msw
        alfa, wc = normalize_radian(alfa)
        self.y[l] = alfa; self.y[l + 1] = r
        self.my[l] = malfa + float(wc); self.my[l + 1] = mr
        T, mT = self.T, self.mT
        Gx = np.array([[0, 0, 1], [cw, sw, 0]], LD); mGx = np.array([[0, 0, 0], [mcw, msw, 0]])
        Gl = np.array([[1, 0], [gl, 1]], LD); mGl = np.array([[0, 0], [mgl, 0]])
        Rm = np.asarray(R, np.float64).reshape(2, 2)
        Prr, mPrr = T[:, :3], mT[:, :3]
        aGx, aGl = _f(Gx), _f(Gl)
        blk = Gx @ Prr @ Gx.T + Gl @ Rm.astype(LD) @ Gl.T
        mblk = (aGx @ mPrr @ aGx.T + mGx @ _f(Prr) @ aGx.T + aGx @ _f(Prr) @ mGx.T
                + aGl @ np.abs(Rm) @ aGl.T + mGl @ np.abs(Rm) @ aGl.T + aGl @ np.abs(Rm) @ mGl.T)
        # rows l and l+1 against every column j < l: Gx P[0:3, j]
        cols = np.arange(l)
        rl = T[2, cols].copy(); mrl = mT[2, cols].copy()
        rl1 = cw * T[0, cols] + sw * T[1, cols]
        mrl1 = float(abs(cw)) * mT[0, cols] + mcw * _f(T[0, cols]) + float(abs(sw)) * mT[1, cols] + msw * _f(T[1, cols])
        v0 = np.zeros(n, LD); m0 = np.zeros(n); v1 = np.zeros(n, LD); m1 = np.zeros(n)
        v0[:l] = rl; m0[:l] = mrl; v1[:l] = rl1; m1[:l] = mrl1
        v0[l], v0[l + 1] = blk[0, 0], blk[0, 1]; m0[l], m0[l + 1] = mblk[0, 0], mblk[0, 1]
        v1[l], v1[l + 1] = blk[1, 0], blk[1, 1]; m1[l], m1[l + 1] = mblk[1, 0], mblk[1, 1]
        self.aug[l] = (v0, m0); self.aug[l + 1] = (v1, m1)
        # rows 0-2 gain the new columns: P[k, l] = P[l, k]
        self.T[:, l] = v0[:3]; self.T[:, l + 1] = v1[:3]
        self.mT[:, l] = m0[:3]; self.mT[:, l + 1] = m1[:3]
        self.L = L + 1

    def _end(self, m, z, R):
        status = 0
        if m == 0 or self.matches == 0:
            self.y[:3] = self.xp; self.my[:3] = self.mxp
            self.pose = self.y[:3].copy(); self.mpose = self.my[:3].copy()
            self.pose[2], wc = normalize_radian(self.pose[2]); self.mpose[2] += float(wc)
        if self.extra:
            self.depth += DEPTH_AUGMENT
        for i in self.extra:
            if self.L >= self.cap:
                status = 2
                break
            self._augment(z[i], R[i])
        if self.L > self.cap - self.headroom:                          # Robot.cpp:893-904
            self.L = 0
            self.y[3:] = 0; self.my[3:] = 0
            self.T[:, 3:] = 0; self.mT[:, 3:] = 0
            self.base = np.zeros((0, 0)); self.aug = {}
            self._clear_terms()
        return status

    def scan(self, u, z, R):
        """One Robot::localize with odometry u.  Returns (status, j_out)."""
        z = np.asarray(z, np.float64).reshape(-1, 2); R = np.asarray(R, np.float64).reshape(-1, 4)
        m = z.shape[0]
        self.predict(u)
        jout = np.full(m, -1, np.int32)
        for i in range(m):
            if self.L == 0:
                self.extra.append(i)
                continue
            j, k, rec = self._first_fit(z[i], R[i])
            if j < 0:
                self.extra.append(i)
                continue
            self.matched.add(j); self.matches += 1
            self._update(j, k, rec)
            jout[i] = j
        return self._end(m, z, R), jout

    def gate_d2(self, j, z, R):
        """d2 of one (line, landmark) pair against the current state (after a predict)."""
        js, d2, rec = self.gates(z, R)
        return d2[int(np.nonzero(js == j)[0][0])]

    @property
    def min_margin(self):
        return min(self.margins) if self.margins else math.inf


def worst_ratio(x, ref, mag):
    """max |x - ref| / (u mag) over the entries (0 where both sides agree exactly; inf where mag is 0 and they
    differ)."""
    x = np.asarray(x, np.float64).astype(LD)
    err = np.abs(x - ref).astype(np.float64)
    mag = np.asarray(mag, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / (U * mag))
    return float(r.max()) if r.size else 0.0


def check(x, ref, mag, C, what=""):
    """Acceptance rule: |x - ref| <= C u mag, componentwise.  Returns the worst err / (u mag)."""
    w = worst_ratio(x, ref, mag)
    assert w <= C, "%s: worst |x - ref| / (u mag) = %.3g > C = %d" % (what, w, C)
    return w


def normwise_ok(x, ref, tol=1e-9):
    """The suite's older measure: max |dP| / max |P|."""
    ref = np.asarray(ref, np.float64)
    return float(np.abs(np.asarray(x, np.float64) - ref).max() / max(np.abs(ref).max(), 1e-300)) < tol


# ---- start states for the componentwise tests ------------------------------------------------------------------
def spread_state(L, cap, seed, pose=(0.3, -0.2, 0.1), pose_scale=1e-2, decades=(-5.0, -1.0)):
    """An exactly symmetric SPD state of L landmarks in a filter of capacity cap: landmarks (alfa, r) with map_scenario
    geometry, P = D (A A' + I) D with A of rank 6 and the landmark entries of D spread over `decades` (P then covers
    twice as many decades).  Returns (y[n], P[n, n], world (L, 2))."""
    rng = np.random.default_rng(seed)
    n, nl = 3 + 2 * cap, 3 + 2 * L
    world = np.empty((L, 2))
    world[:, 0] = np.mod(rng.uniform(-math.pi, math.pi, L) + math.pi, 2 * math.pi) - math.pi
    world[:, 1] = rng.uniform(2.0, 8.0, L)
    y = np.zeros(n)
    y[:3] = pose
    y[3:nl:2] = world[:, 0]; y[4:nl:2] = world[:, 1]
    A = rng.standard_normal((nl, 6)) / math.sqrt(6.0)
    M = A @ A.T + np.eye(nl)
    M = np.triu(M) + np.triu(M, 1).T
    D = np.empty(nl)
    D[:3] = pose_scale
    D[3:] = np.repeat(10.0 ** rng.uniform(decades[0], decades[1], L), 2)
    Pl = np.triu(D[:, None] * M * D[None, :])
    P = np.zeros((n, n))
    P[:nl, :nl] = Pl + np.triu(Pl, 1).T
    return y, P, world


def predicted_pose(pose, u):
    """Robot.cpp:148 (the truth for lines generated without noise in the pose)."""
    x, yy, th = pose
    a = th + u[2] / 2.0
    return (x + u[0] * math.cos(a), yy + u[0] * math.sin(a), th + u[2])


def lines_for(world, pose, ids, rng, n_unmatched=0, noise=0.05):
    """Observed lines (z (m, 2), R (m, 4)) of landmarks `ids` seen from `pose`, with noise `noise` x the declared
    std, followed by `n_unmatched` lines 3 m beyond a landmark (they match nothing and are appended)."""
    sa, sr = 2e-3, 5e-3
    ids = list(ids)
    extra = rng.choice(len(world), n_unmatched) if n_unmatched else []
    wl = np.array([world[i] for i in ids] + [world[i] + (0.0, 3.0) for i in extra]).reshape(-1, 2)
    x, yy, th = pose
    z = np.empty_like(wl)
    z[:, 0] = wl[:, 0] - th
    z[:, 0] = np.mod(z[:, 0] + math.pi, 2 * math.pi) - math.pi
    z[:, 1] = wl[:, 1] - (x * np.cos(wl[:, 0]) + yy * np.sin(wl[:, 0]))
    z += rng.standard_normal(z.shape) * np.array([sa, sr]) * noise
    R = np.zeros((len(z), 4)); R[:, 0] = sa * sa; R[:, 3] = sr * sr
    return z, R
