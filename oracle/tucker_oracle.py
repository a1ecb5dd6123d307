"""CPU oracle for the Tucker-fit half of the hot path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
leg may import this; the product (nlml_hpe_b200/) never does.

Parity status: PINNED for the fixed-iteration fit -- `sgd_reference_form` and
`sgd_batched` are checked in tests/test_oracle.py against outputs of the real
reference (`TD_Tester.optimize_with_sgd`, `TD_Tester.objective_torch` + autograd)
generated in the build container by tests/golden/make_golden.py and committed under
tests/golden/.  The reference has no golden vectors of its own (SURVEY.md section 4).
Parity UNPINNED for the scipy-Powell search (`powell_fit`): scipy is an unpinned
third-party dependency (TD_Tester.py:191-194) and only the optimum is compared.

What is restated (all file:line into /root/reference):
  cos_feature           TD_Tester.py:105-107  (func_torch)  / :25-28 (func)
  objective             TD_Tester.py:110-125  (objective_torch)
  sgd_reference_form    TD_Tester.py:127-159  (optimize_with_sgd): zero init :130, loss :139,
                        backward :145, joint clip_grad_norm_(max_norm=1) :150, p -= lr*grad :153-154
  sgd_batched           the same recurrence with the gradient of :110-125 written out by hand
                        (NOT TD_Tester.compute_gradient, whose u_id part :97 is wrong and dead)
  powell_fit            TD_Tester.py:162-199 (Test) with the objective of :31-58
  newton_terms, lm_fit  float64 checker of the converged solver (SURVEY.md section 8f row 1): same objective
                        (:110-125), same start (:164); compared with Powell at the optimum only
"""
from __future__ import annotations

import numpy as np
import torch


def cos_feature(w, row):
    """a*cos(b*w+c)+d, TD_Tester.py:105-107."""
    return row[0] * torch.cos(row[1] * w + row[2]) + row[3]


def objective(p, W, x, rows_y, rows_p, rows_r):
    """0.5*||x - W x1 u x2 f_y x3 f_p x4 f_r||^2, TD_Tester.py:110-125."""
    f_y = torch.stack([cos_feature(p[0], r) for r in rows_y])
    f_p = torch.stack([cos_feature(p[1], r) for r in rows_p])
    f_r = torch.stack([cos_feature(p[2], r) for r in rows_r])
    x_hat = torch.einsum("ijklm,i,j,k,l->m", W, p[3:], f_y, f_p, f_r)
    return 0.5 * ((x - x_hat) ** 2).sum()


def sgd_reference_form(W, x, rows_y, rows_p, rows_r, lr=0.001, iters=3000, clip=1.0):
    """One sample, autograd, exactly the recurrence of TD_Tester.py:127-159.

    All inputs are converted to float32 torch tensors as the (commented) caller does
    (TD_Tester.py:170-174).  Returns p f32 [3+R_id] (radians + identity coefficients).
    """
    W = torch.as_tensor(np.asarray(W), dtype=torch.float32)
    x = torch.as_tensor(np.asarray(x), dtype=torch.float32)
    rows = [torch.as_tensor(np.asarray(r), dtype=torch.float32) for r in (rows_y, rows_p, rows_r)]
    p = torch.zeros(3 + W.shape[0], dtype=torch.float32, requires_grad=True)
    for _ in range(iters):
        if p.grad is not None:
            p.grad.zero_()
        objective(p, W, x, *rows).backward()
        torch.nn.utils.clip_grad_norm_(p, max_norm=clip)
        with torch.no_grad():
            p -= lr * p.grad
    return p.detach().numpy().copy()


def _features_and_derivs(w, rows, dtype=np.float32):
    """w [N]; rows [R,4] -> (c, dc) [N,R] each, in dtype."""
    a, b, c, d = rows[:, 0], rows[:, 1], rows[:, 2], rows[:, 3]
    arg = b[None, :] * w[:, None] + c[None, :]
    val = a[None, :] * np.cos(arg) + d[None, :]
    der = -(a * b)[None, :] * np.sin(arg)
    return val.astype(dtype), der.astype(dtype)


def gradient_batched(P, W, X, rows_y, rows_p, rows_r, dtype=np.float32):
    """Gradient of `objective` w.r.t. p for a batch, direct (residual) form, computed in dtype (float32: the
    reference's arithmetic; float64: a check on how well a float32 result is conditioned).

    r = x_hat - x ; dL/dz = W2 r ; chain rule through z = u (x) c_y (x) c_p (x) c_r.
    P [N,3+R_id], X [N,F] -> G [N,3+R_id], loss [N], both dtype.
    """
    W = np.asarray(W, dtype=dtype)
    r_id, r_y, r_p, r_r, F = W.shape
    W2 = W.reshape(-1, F)
    X = np.asarray(X, dtype=dtype)
    rows_y, rows_p, rows_r = (np.asarray(r, dtype=dtype) for r in (rows_y, rows_p, rows_r))
    P = np.asarray(P, dtype=dtype)
    cy, dcy = _features_and_derivs(P[:, 0], rows_y, dtype)
    cp, dcp = _features_and_derivs(P[:, 1], rows_p, dtype)
    cr, dcr = _features_and_derivs(P[:, 2], rows_r, dtype)
    u = P[:, 3:]
    z = np.einsum("ni,nj,nk,nl->nijkl", u, cy, cp, cr).reshape(len(P), -1).astype(dtype)
    res = z @ W2 - X
    gz = (res @ W2.T).reshape(len(P), r_id, r_y, r_p, r_r).astype(dtype)
    G = np.empty_like(P)
    G[:, 0] = np.einsum("nijkl,ni,nj,nk,nl->n", gz, u, dcy, cp, cr)
    G[:, 1] = np.einsum("nijkl,ni,nj,nk,nl->n", gz, u, cy, dcp, cr)
    G[:, 2] = np.einsum("nijkl,ni,nj,nk,nl->n", gz, u, cy, cp, dcr)
    G[:, 3:] = np.einsum("nijkl,nj,nk,nl->ni", gz, cy, cp, cr)
    return G.astype(dtype), (0.5 * (res * res).sum(1)).astype(dtype)


def sgd_batched(W, X, rows_y, rows_p, rows_r, lr=0.001, iters=3000, clip=1.0, P0=None, dtype=np.float32):
    """Batched restatement of TD_Tester.py:127-159 with the hand-written gradient, in dtype (float32 = the reference).

    clip_grad_norm_ semantics (:150): g *= min(1, clip / (||g||_2 + 1e-6)), norm over all
    3+R_id components jointly; update (:153-154): p -= lr * g.  Returns P [N,3+R_id] in dtype.
    """
    X = np.asarray(X, dtype=dtype)
    n = X.shape[0]
    P = np.zeros((n, 3 + W.shape[0]), dtype=dtype) if P0 is None else np.array(P0, dtype=dtype)
    lr_, clip_, eps_ = dtype(lr), dtype(clip), dtype(1e-6)
    for _ in range(iters):
        G, _ = gradient_batched(P, W, X, rows_y, rows_p, rows_r, dtype)
        norm = np.sqrt((G * G).sum(1, dtype=dtype)).astype(dtype)
        coef = np.minimum(clip_ / (norm + eps_), dtype(1.0)).astype(dtype)
        G = (G * coef[:, None]).astype(dtype)
        P = (P - lr_ * G).astype(dtype)
    return P


def powell_fit(W, x, rows_y, rows_p, rows_r):
    """scipy Powell over the float64 objective of TD_Tester.py:31-58, as Test() does (:191-199).

    Returns (yaw, pitch, roll) in degrees and the identity coefficients.  parity unpinned.
    """
    from scipy.optimize import minimize

    W = np.asarray(W, dtype=np.float32)
    x = np.asarray(x, dtype=np.float32)
    rows = [np.asarray(r, dtype=np.float64) for r in (rows_y, rows_p, rows_r)]

    def f(p):
        fs = [np.array([r[0] * np.cos(r[1] * p[k] + r[2]) + r[3] for r in rows[k]]).astype(np.float32)
              for k in range(3)]
        x_hat = np.einsum("ijklm,i,j,k,l->m", W, p[3:], *fs)
        return 0.5 * np.sum((x - x_hat) ** 2)

    res = minimize(f, np.zeros(3 + W.shape[0]), method="Powell")
    return np.degrees(res.x[:3]), res.x[3:]


def _objective_f64(p, W2, x, rows):
    """TD_Tester.py:110-125 in float64 for one sample (functional form, for torch.func)."""
    fs = [r[:, 0] * torch.cos(r[:, 1] * p[k] + r[:, 2]) + r[:, 3] for k, r in enumerate(rows)]
    z = torch.einsum("i,j,k,l->ijkl", p[3:], *fs).reshape(-1)
    res = x - z @ W2
    return 0.5 * (res * res).sum()


def newton_terms(P, W, X, rows_y, rows_p, rows_r):
    """Loss, gradient and exact Hessian of the objective (TD_Tester.py:110-125) at P, float64, batched
    (torch.func).  P [N,3+R_id], X [N,F] -> L [N], G [N,NP], H [N,NP,NP]."""
    W = torch.as_tensor(np.asarray(W), dtype=torch.float64)
    W2 = W.reshape(-1, W.shape[-1])
    rows = [torch.as_tensor(np.asarray(r), dtype=torch.float64) for r in (rows_y, rows_p, rows_r)]
    P = torch.as_tensor(np.asarray(P), dtype=torch.float64)
    X = torch.as_tensor(np.asarray(X), dtype=torch.float64)
    f = lambda p, x: _objective_f64(p, W2, x, rows)
    L = torch.func.vmap(f)(P, X)
    G = torch.func.vmap(torch.func.grad(f))(P, X)
    H = torch.func.vmap(torch.func.hessian(f))(P, X)
    return L.numpy(), G.numpy(), H.numpy()


def lm_fit(W, X, rows_y, rows_p, rows_r, max_evals=200, lambda0=1e-3, down=5.0, up=4.0, angle_cap=0.15,
           step_tol=1e-10, diag_floor=1.0, lambda_min=1e-5):
    """Converged fit: float64 restatement of csrc/tucker_math.h tucker_lm_solve (damped Newton with the exact
    Hessian, Marquardt scaling, capped angle step, from p = 0 as TD_Tester.py:164).  parity unpinned against the
    reference's scipy Powell search (TD_Tester.py:191-194): same objective, same start, compared at the optimum.
    Returns P f64 [N,3+R_id], final loss [N], evaluations [N]."""
    X = np.asarray(X, dtype=np.float64)
    n, NP = X.shape[0], 3 + np.asarray(W).shape[0]
    P = np.zeros((n, NP))
    L, G, H = newton_terms(P, W, X, rows_y, rows_p, rows_r)
    lam = np.full(n, lambda0)
    active = np.ones(n, bool)
    evals = np.ones(n, int)
    eye = np.eye(NP)
    for _ in range(4 * max_evals):
        idx = np.nonzero(active)[0]
        if idx.size == 0:
            break
        diag = np.abs(np.einsum("nii->ni", H[idx])) + diag_floor
        A = H[idx] + lam[idx, None, None] * diag[:, :, None] * eye
        ok = np.all(np.linalg.eigvalsh(A) > 0, axis=1)
        lam[idx[~ok]] *= up
        active[idx[~ok][lam[idx[~ok]] > 1e12]] = False
        idx, A = idx[ok], A[ok]
        if idx.size == 0:
            continue
        D = np.linalg.solve(A, G[idx][:, :, None])[:, :, 0]
        ma = np.abs(D[:, :3]).max(1)
        capped = ma > angle_cap
        D = D * np.where(capped, angle_cap / np.maximum(ma, 1e-300), 1.0)[:, None]
        step = np.abs(D).max(1)
        Pn = P[idx] - D
        done = (step < step_tol) & (lam[idx] < 1.0)
        P[idx[done]] = Pn[done]
        active[idx[done]] = False
        idx, Pn, capped = idx[~done], Pn[~done], capped[~done]
        if idx.size == 0:
            continue
        Ln, Gn, Hn = newton_terms(Pn, W, X[idx], rows_y, rows_p, rows_r)
        evals[idx] += 1
        acc = Ln <= L[idx]
        a = idx[acc]
        P[a], L[a], G[a], H[a] = Pn[acc], Ln[acc], Gn[acc], Hn[acc]
        dn = a[~capped[acc]]
        lam[dn] = np.maximum(lam[dn] / down, lambda_min)
        rj = idx[~acc]
        lam[rj] *= up
        active[rj[lam[rj] > 1e12]] = False
        active[evals >= max_evals] = False
    return P, L, evals
