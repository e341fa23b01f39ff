"""Scalar NumPy twin of the device L-BFGS of mfgp_gpr_batched_lbfgs (include/mfgp.h): SciPy's L-BFGS-B
(scipy.optimize.minimize(method="L-BFGS-B")) on an unbounded problem, written out.

- Direction: the two-loop recursion over the last m pairs (s, y) with H0 = dr / y^T y of the newest pair, where every
  s^T y is the directional-derivative difference `dr` of the accepted step (as L-BFGS-B stores it); d = -g with an
  empty memory.  z = x + d and d = z - x from then on; the trial point is z when stp == 1 and t + stp d otherwise.
- Step: stp = min(1 / ||d||, 1e10) on iteration 0, 1 afterwards; stpmax = 1e10.
- Line search: MINPACK-2 dcsrch / dcstep (ported below from the published Fortran, as scipy.optimize._dcsrch is) with
  ftol = 1e-3, gtol = 0.9, xtol = 0.1, stpmin = 0, one evaluation per call.  g^T d >= 0 at the start, or more than maxls
  evaluations, fails the search: x, f, g are restored; a non-empty memory is cleared and the iteration restarts; an empty
  one stops with "abnormal".
- After an accepted step, in SciPy's order: nit += 1; nit >= maxiter; nfev > maxfun; ||g||_inf <= gtol;
  (f_old - f) <= ftol max(|f_old|, |f|, 1).  Then the memory update, skipped when dr <= eps * ddum.
- The one deliberate deviation from SciPy: a trial point whose objective or gradient is not finite (a covariance that is
  not positive definite) counts as an evaluation and against maxls, and the search restarts from the same base point with
  a fresh dcsrch at 0.1 x the failed step and stpmax = 0.5 x the failed step.  A start point that fails stops at once
  with "not_pd".
"""
import numpy as np

EPS = np.finfo(float).eps
STATUS = ("pgtol", "ftol", "maxiter", "maxfun", "abnormal", "not_pd")  # codes 1..6 of include/mfgp.h
DEFAULTS = dict(m=10, maxiter=15000, maxfun=15000, maxls=20, ftol=2.220446049250313e-09, gtol=1e-5)
LS_FTOL, LS_GTOL, LS_XTOL, STPMAX = 1e-3, 0.9, 0.1, 1e10


def dcstep(stx, fx, dx, sty, fy, dy, stp, fp, dp, brackt, stpmin, stpmax):
    """MINPACK-2 dcstep: a safeguarded cubic / quadratic step and the update of the interval [stx, sty]."""
    sgnd = np.sign(dp) * np.sign(dx)
    if fp > fx:  # higher function value: the minimum is bracketed
        theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp
        s = max(abs(theta), abs(dx), abs(dp))
        gamma = s * np.sqrt((theta / s) ** 2 - (dx / s) * (dp / s))
        if stp < stx:
            gamma = -gamma
        p = (gamma - dx) + theta
        q = ((gamma - dx) + gamma) + dp
        stpc = stx + (p / q) * (stp - stx)
        stpq = stx + ((dx / ((fx - fp) / (stp - stx) + dx)) / 2.0) * (stp - stx)
        stpf = stpc if abs(stpc - stx) <= abs(stpq - stx) else stpc + (stpq - stpc) / 2.0
        brackt = True
    elif sgnd < 0.0:  # derivatives of opposite sign: bracketed
        theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp
        s = max(abs(theta), abs(dx), abs(dp))
        gamma = s * np.sqrt((theta / s) ** 2 - (dx / s) * (dp / s))
        if stp > stx:
            gamma = -gamma
        p = (gamma - dp) + theta
        q = ((gamma - dp) + gamma) + dx
        stpc = stp + (p / q) * (stx - stp)
        stpq = stp + (dp / (dp - dx)) * (stx - stp)
        stpf = stpc if abs(stpc - stp) > abs(stpq - stp) else stpq
        brackt = True
    elif abs(dp) < abs(dx):  # same sign, the derivative magnitude decreases
        theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp
        s = max(abs(theta), abs(dx), abs(dp))
        gamma = s * np.sqrt(max(0.0, (theta / s) ** 2 - (dx / s) * (dp / s)))
        if stp > stx:
            gamma = -gamma
        p = (gamma - dp) + theta
        q = (gamma + (dx - dp)) + gamma
        r = p / q
        if r < 0.0 and gamma != 0.0:
            stpc = stp + r * (stx - stp)
        elif stp > stx:
            stpc = stpmax
        else:
            stpc = stpmin
        stpq = stp + (dp / (dp - dx)) * (stx - stp)
        if brackt:
            stpf = stpc if abs(stpc - stp) < abs(stpq - stp) else stpq
            if stp > stx:
                stpf = min(stp + 0.66 * (sty - stp), stpf)
            else:
                stpf = max(stp + 0.66 * (sty - stp), stpf)
        else:
            stpf = stpc if abs(stpc - stp) > abs(stpq - stp) else stpq
            stpf = min(stpmax, max(stpmin, stpf))
    else:  # same sign, the derivative magnitude does not decrease
        if brackt:
            theta = 3.0 * (fp - fy) / (sty - stp) + dy + dp
            s = max(abs(theta), abs(dy), abs(dp))
            gamma = s * np.sqrt((theta / s) ** 2 - (dy / s) * (dp / s))
            if stp > sty:
                gamma = -gamma
            p = (gamma - dp) + theta
            q = ((gamma - dp) + gamma) + dy
            stpf = stp + (p / q) * (sty - stp)
        elif stp > stx:
            stpf = stpmax
        else:
            stpf = stpmin
    if fp > fx:
        sty, fy, dy = stp, fp, dp
    else:
        if sgnd < 0.0:
            sty, fy, dy = stx, fx, dx
        stx, fx, dx = stp, fp, dp
    return stx, fx, dx, sty, fy, dy, stpf, brackt


class Dcsrch:
    """MINPACK-2 dcsrch as a resumable state machine: start(stp, f0, g0) then step(stp, f, g) after each evaluation.
    Both return (stp, task) with task "FG" (evaluate at stp), "CONV", "WARN" or "ERROR".  The attribute names are those
    of scipy.optimize._dcsrch.DCSRCH."""

    def __init__(self, ftol=LS_FTOL, gtol=LS_GTOL, xtol=LS_XTOL, stpmin=0.0, stpmax=STPMAX):
        self.ftol, self.gtol, self.xtol, self.stpmin, self.stpmax = ftol, gtol, xtol, stpmin, stpmax

    def start(self, stp, f, g):
        if stp < self.stpmin or stp > self.stpmax or g >= 0.0:
            return stp, "ERROR"
        self.brackt, self.stage = False, 1
        self.finit, self.ginit = f, g
        self.gtest = self.ftol * g
        self.width = self.stpmax - self.stpmin
        self.width1 = self.width / 0.5
        self.stx, self.fx, self.gx = 0.0, f, g
        self.sty, self.fy, self.gy = 0.0, f, g
        self.stmin, self.stmax = 0.0, stp + 4.0 * stp
        return stp, "FG"

    def step(self, stp, f, g):
        ftest = self.finit + stp * self.gtest
        if self.stage == 1 and f <= ftest and g >= 0.0:
            self.stage = 2
        task = "FG"
        if self.brackt and (stp <= self.stmin or stp >= self.stmax):
            task = "WARN"  # rounding errors prevent progress
        if self.brackt and self.stmax - self.stmin <= self.xtol * self.stmax:
            task = "WARN"  # xtol test satisfied
        if stp == self.stpmax and f <= ftest and g <= self.gtest:
            task = "WARN"  # stp = stpmax
        if stp == self.stpmin and (f > ftest or g >= self.gtest):
            task = "WARN"  # stp = stpmin
        if f <= ftest and abs(g) <= self.gtol * -self.ginit:
            task = "CONV"
        if task != "FG":
            return stp, task
        if self.stage == 1 and f <= self.fx and f > ftest:  # the modified function psi
            gt = self.gtest
            stx, fxm, gxm, sty, fym, gym, stp, self.brackt = dcstep(
                self.stx, self.fx - self.stx * gt, self.gx - gt, self.sty, self.fy - self.sty * gt, self.gy - gt,
                stp, f - stp * gt, g - gt, self.brackt, self.stmin, self.stmax)
            self.stx, self.sty = stx, sty
            self.fx, self.fy = fxm + stx * gt, fym + sty * gt
            self.gx, self.gy = gxm + gt, gym + gt
        else:
            (self.stx, self.fx, self.gx, self.sty, self.fy, self.gy, stp, self.brackt) = dcstep(
                self.stx, self.fx, self.gx, self.sty, self.fy, self.gy, stp, f, g, self.brackt, self.stmin, self.stmax)
        if self.brackt:
            if abs(self.sty - self.stx) >= 0.66 * self.width1:
                stp = self.stx + 0.5 * (self.sty - self.stx)
            self.width1 = self.width
            self.width = abs(self.sty - self.stx)
            self.stmin, self.stmax = min(self.stx, self.sty), max(self.stx, self.sty)
        else:
            self.stmin = stp + 1.1 * (stp - self.stx)
            self.stmax = stp + 4.0 * (stp - self.stx)
        stp = min(self.stpmax, max(self.stpmin, stp))
        if (self.brackt and (stp <= self.stmin or stp >= self.stmax)) or \
                (self.brackt and self.stmax - self.stmin <= self.xtol * self.stmax):
            stp = self.stx
        return stp, "FG"


def _finite(f, g):
    return bool(np.isfinite(f)) and bool(np.all(np.isfinite(g)))


def minimize(fg, x0, m=10, maxiter=15000, maxfun=15000, maxls=20, ftol=DEFAULTS["ftol"], gtol=1e-5, trace=None):
    """fg(x) -> (f, g); a non-finite f or g marks a failed point.  Returns dict(x, f, g, nit, nfev, status, iterates),
    iterates = [x0, x_1, ...] the accepted points.  `trace` (a list) receives (x, stp, stpmax) of every trial."""
    x = np.array(x0, dtype=np.float64)
    f, g = fg(x)
    nfev, nit = 1, 0
    iterates = [x.copy()]

    def done(status, x, f, g):
        return dict(x=x, f=f, g=g, nit=nit, nfev=nfev, status=status, iterates=iterates)

    if not _finite(f, g):
        return done("not_pd", x, np.nan, g)
    if np.abs(g).max() <= gtol:
        return done("pgtol", x, f, g)
    S, Y, DR = [], [], []
    while True:
        # ---- direction: two-loop recursion ----
        q = -g
        if S:
            al = []
            for s, y, dr in zip(reversed(S), reversed(Y), reversed(DR)):
                a = (s @ q) / dr
                al.append(a)
                q = q - a * y
            q = q * (DR[-1] / (Y[-1] @ Y[-1]))
            for (s, y, dr), a in zip(zip(S, Y, DR), reversed(al)):
                b = (y @ q) / dr
                q = q + (a - b) * s
        z = x + q
        d = z - x
        stp = min(1.0 / np.sqrt(d @ d), STPMAX) if nit == 0 else 1.0
        t, r, fold = x.copy(), g.copy(), f
        gd = g @ d
        gdold = gd
        ls = Dcsrch()
        ifun = 0
        fail = gd >= 0.0
        if not fail:
            stp, task = ls.start(stp, f, gd)
            fail = task == "ERROR"
        while not fail:
            ifun += 1
            if ifun > maxls:
                fail = True
                break
            x = z.copy() if stp == 1.0 else stp * d + t
            if trace is not None:
                trace.append((x.copy(), stp, ls.stpmax))
            f, g = fg(x)
            nfev += 1
            if not _finite(f, g):  # restart the search from the base point, short of the failed step
                bad = stp
                ls = Dcsrch(stpmax=0.5 * bad)
                stp, task = ls.start(0.1 * bad, fold, gdold)
                fail = task == "ERROR"
                continue
            gd = g @ d
            stp, task = ls.step(stp, f, gd)
            if task in ("CONV", "WARN"):
                break
            fail = task == "ERROR"
        if fail:
            x, g, f = t, r, fold
            if not S:
                nit += 1
                return done("abnormal", x, f, g)
            S, Y, DR = [], [], []
            continue
        nit += 1
        iterates.append(x.copy())
        if nit >= maxiter:
            return done("maxiter", x, f, g)
        if nfev > maxfun:
            return done("maxfun", x, f, g)
        if np.abs(g).max() <= gtol:
            return done("pgtol", x, f, g)
        if (fold - f) <= ftol * max(abs(fold), abs(f), 1.0):
            return done("ftol", x, f, g)
        y = g - r
        if stp == 1.0:
            dr, ddum, s = gd - gdold, -gdold, d
        else:
            dr, ddum, s = (gd - gdold) * stp, -gdold * stp, stp * d
        if dr <= EPS * ddum:
            continue
        S.append(s)
        Y.append(y)
        DR.append(dr)
        if len(S) > m:
            S.pop(0)
            Y.pop(0)
            DR.pop(0)
