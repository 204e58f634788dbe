"""numpy / scipy restatement of the library's GCRO-DR ("Krylov Method" = "GCRODR"; Parks, de Sturler, Mackey, Johnson,
Maiti, SIAM J. Sci. Comput. 28(5), 2006, Algorithm 2, in real arithmetic) -- test infrastructure only.

It follows the GMRES restatement of oracle/krylov.py (two passes of classical Gram-Schmidt, Givens least squares, the
same residual tests and scalings) with the recycled space of the library:
  * a cycle with kc recycled columns runs m - kc Arnoldi steps of (I - C C') A^ on v0 = (I - C C') r / beta', where A^
    is A M^-1 (right), M^-1 A (left) or A; the least-squares right-hand side is [C' r; beta' e1], and the first kc
    columns of Ghat are D = diag(1 / ||u_i||) (U enters scaled);
  * at the end of every cycle of more than k columns, the harmonic Ritz problem Ghat' Ghat z = theta Ghat' (What' Vhat) z
    is solved with scipy.linalg.eig(A, B) (QZ, independent of the library's Cholesky reduction), the k smallest |theta|
    are kept (a complex pair whole), and Ghat P = Q R gives C = What Q, U = Vhat P R^-1;
  * a solve given U0 (and C0 = A^ U0 with orthonormal columns, or None to rebuild it) first sets x += [M^-1] U C' r.
"""
import numpy as np
import scipy.linalg as sl

from oracle.krylov import _scale

RANK_TOL = 1e-12


def _qr_pos(X):
    Q, R = np.linalg.qr(X)
    s = np.where(np.diag(R) < 0, -1.0, 1.0)
    return Q * s, R * s[:, None]


def _cholesky_ok(A):
    """the library's test (dense_eig.cpp, hy_cholesky): every pivot of A = L L' above n eps max_i A_ii"""
    n = A.shape[0]
    floor = n * np.finfo(float).eps * np.abs(np.diag(A)).max()
    L = np.zeros_like(A)
    for j in range(n):
        s = A[j, j] - L[j, :j] @ L[j, :j]
        if not s > floor:
            return False
        L[j, j] = np.sqrt(s)
        L[j + 1:, j] = (A[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return True


def _harmonic(Gh, WV, k, kmax, gaps=None, reduction="qz"):
    """P (real columns) for the k smallest |theta| of Gh'Gh z = theta Gh'WV z, or None (A numerically singular).
    gaps (a list, optional) receives the relative gap of the selection: (t_out - t_in) / t_in, t_in the largest kept
    |theta| and t_out the smallest |theta| left out (inf when nothing is left out).
    reduction: "qz" (scipy.linalg.eig(A, B), the default), or the standard problem L^-1 B L^-T w = mu w with L from
    "normal" (numpy's Cholesky factor of A = Gh'Gh) or "qr" (L' = R of the Householder QR Gh = Q R, A not formed).
    The two alternatives measure how sensitive the harmonic Ritz vectors of a given cycle are to the way the problem
    is solved."""
    A = Gh.T @ Gh
    B = Gh.T @ WV
    n = A.shape[0]
    if not _cholesky_ok(A):
        return None
    if reduction == "qz":
        th, Z = sl.eig(A, B)
    else:
        if reduction == "normal":
            L = np.linalg.cholesky(A)
        else:                                   # L' = R of Gh = Q R
            R = np.linalg.qr(Gh, mode="r")
            R = R * np.where(np.diag(R) < 0, -1.0, 1.0)[:, None]
            L = R.T
        S = sl.solve_triangular(L, sl.solve_triangular(L, B.T, lower=True).T, lower=True)
        mu, Wv = sl.eig(S)
        with np.errstate(divide="ignore"):
            th = 1.0 / mu
        Z = sl.solve_triangular(L.T, Wv, lower=False)
    mod = np.where(np.isfinite(th), np.abs(th), np.inf)
    order = list(np.argsort(mod, kind="stable"))
    sel = order[:k]

    def partner(i):
        if th[i].imag == 0 or not np.isfinite(th[i]):
            return i
        d = np.abs(th - np.conj(th[i]))
        d[i] = np.inf
        return int(np.argmin(d))

    for i in list(sel):
        j = partner(i)
        if j not in sel:
            if len(sel) + 1 > kmax:
                sel.remove(i)
            else:
                sel.append(j)
    if gaps is not None:
        t_in = max(mod[i] for i in sel) if sel else 0.0
        out = [mod[i] for i in range(len(th)) if i not in sel]
        t_out = min(out) if out else np.inf
        gaps.append((t_out - t_in) / t_in if t_in > 0 else np.inf)
    cols = []
    done = set()
    for i in sel:
        if i in done:
            continue
        z = Z[:, i]
        if partner(i) != i:
            cols += [z.real, z.imag]
            done.update((i, partner(i)))
        else:
            cols.append(z.real)
            done.add(i)
    return np.array(cols).T if cols else None


def gcrodr(apply_A, b, x0, apply_M=None, side="Right", tol=1e-8, max_iters=1000, num_blocks=300, num_recycled=5,
           max_restarts=20, explicit_test=False, imp_scaling="Norm of Preconditioned Initial Residual",
           exp_scaling="Norm of Initial Residual", U0=None, C0=None, info=None, reduction="qz"):
    """returns x, iters, converged, history, U, C (U, C: the recycled space for the next solve, or None).
    info (a dict, optional) receives "cycle_ends", the history length at the end of every cycle, and "gaps", for every
    new recycled space the relative gap of its selection (see _harmonic) and the index of the cycle that chose it."""
    if info is not None:
        info["cycle_ends"], info["gaps"] = [], []
    b = np.asarray(b, dtype=np.float64)
    x = np.array(x0, dtype=np.float64, copy=True)
    left = apply_M is not None and side == "Left"
    right = apply_M is not None and side == "Right"
    m = max(1, min(num_blocks, max_iters))
    k = num_recycled
    assert 1 <= k < m
    kmax = min(k + 1, m - 1)

    def prec(r):
        return apply_M(r) if left else r

    def ahat(v):
        if right:
            return apply_A(apply_M(v))
        if left:
            return apply_M(apply_A(v))
        return apply_A(v)

    r0_true = b - apply_A(x)
    pr0 = prec(r0_true)
    imp_scale = _scale(imp_scaling, b, r0_true, pr0) or 1.0
    exp_scale = _scale(exp_scaling, b, r0_true, pr0) or 1.0
    r = pr0
    beta = np.linalg.norm(r)
    history = [beta / imp_scale]
    U, Cm = (None, None) if U0 is None else (np.array(U0, dtype=np.float64), None if C0 is None else np.array(C0))
    if U is not None and Cm is None:          # C = A^ U, thin QR C = Q R, U <- U R^-1
        Cm = np.array([ahat(u) for u in U.T]).T
        Q, R = _qr_pos(Cm)
        Cm, U = Q, U @ np.linalg.inv(R)
    if U is not None:                         # x += [M^-1] U C' r
        upd = U @ (Cm.T @ r)
        x = x + (apply_M(upd) if right else upd)
        rt = b - apply_A(x)
        r = prec(rt)
        beta = np.linalg.norm(r)
    iters = 0
    converged = False
    for restart in range(max_restarts + 1):
        if beta == 0.0 or (beta / imp_scale <= tol and not explicit_test):
            converged = True
            break
        kc = 0 if U is None else U.shape[1]
        H = np.zeros((m + 1, m))
        G = np.zeros((m + 1, m))
        cs, sn, g = np.zeros(m), np.zeros(m), np.zeros(m + 1)
        W = []
        if kc:
            d = 1.0 / np.linalg.norm(U, axis=0)
            c = Cm.T @ r
            v0 = r - Cm @ c
            bp = np.linalg.norm(v0)
            g[:kc] = c
            g[kc] = bp
            H[:kc, :kc] = np.diag(d)
            cs[:kc] = 1.0
            W = list(Cm.T) + [v0 / bp]
        else:
            g[0] = beta
            W = [r / beta]
        k_done = kc
        for j in range(kc, m):
            if iters >= max_iters:
                break
            w = ahat(W[j])
            Bm = np.array(W[:j + 1])
            h = Bm @ w
            w = w - Bm.T @ h
            h2 = Bm @ w
            w = w - Bm.T @ h2
            h = h + h2
            hn = np.linalg.norm(w)
            breakdown = not (hn > 1e-300) or hn <= 1e-15 * np.linalg.norm(h)
            H[:j + 1, j] = h
            H[j + 1, j] = 0.0 if breakdown else hn
            G[:j + 2, j] = H[:j + 2, j]
            W.append(np.zeros_like(w) if breakdown else w / hn)
            for i in range(kc, j):
                t = cs[i] * H[i, j] + sn[i] * H[i + 1, j]
                H[i + 1, j] = -sn[i] * H[i, j] + cs[i] * H[i + 1, j]
                H[i, j] = t
            dd = np.hypot(H[j, j], H[j + 1, j])
            cs[j] = H[j, j] / dd
            sn[j] = H[j + 1, j] / dd
            H[j, j] = dd
            H[j + 1, j] = 0.0
            g[j + 1] = -sn[j] * g[j]
            g[j] = cs[j] * g[j]
            iters += 1
            k_done = j + 1
            rel = abs(g[j + 1]) / imp_scale
            history.append(rel)
            if rel <= tol or breakdown:
                break
        if k_done > kc:
            y = sl.solve_triangular(np.triu(H[:k_done, :k_done]), g[:k_done])
            V = np.array(W[kc:k_done]).T
            upd = V @ y[kc:]
            if kc:
                upd = upd + U @ (d * y[:kc])
            x = x + (apply_M(upd) if right else upd)
        if k_done > kc and k_done > k:        # the new recycled space
            mt, pD = k_done, k_done - kc
            Gh = np.zeros((mt + 1, mt))
            Gh[:kc, :kc] = np.diag(d) if kc else np.zeros((0, 0))
            Gh[:, kc:] = G[:mt + 1, kc:mt]
            Wm = np.array(W[:mt + 1]).T
            WV = np.zeros((mt + 1, mt))
            WV[kc:, kc:] = np.eye(mt + 1 - kc, pD)
            if kc:
                WV[:, :kc] = (Wm.T @ U) * d
            g_ = []
            P = _harmonic(Gh, WV, k, kmax, g_, reduction)
            if info is not None and g_:
                info["gaps"].append((len(info["cycle_ends"]), g_[0]))
            Uold = U
            U = Cm = None              # failure: no space, the next cycle is a plain GMRES cycle
            if P is not None:
                Q, R = _qr_pos(Gh @ P)
                if np.abs(np.diag(R)).min() > RANK_TOL * np.abs(np.diag(R)).max():
                    Ytil = np.array(W[kc:kc + pD]).T @ P[kc:]      # Vhat P, Vhat = [U D | v_0 .. v_(pD-1)]
                    if kc:
                        Ytil = Ytil + (Uold * d) @ P[:kc]
                    U = Ytil @ np.linalg.inv(R)
                    Cm = Wm @ Q
        if info is not None:
            info["cycle_ends"].append(len(history))
        rt = b - apply_A(x)
        r = prec(rt)
        beta = np.linalg.norm(r)
        if history[-1] <= tol:
            if not explicit_test or np.linalg.norm(rt) / exp_scale <= tol:
                converged = True
                break
        if iters >= max_iters:
            break
    return x, iters, converged, history, U, Cm
