"""The one-off original analysis on the device (SURVEY.md section 8f, rank 1): the cross-block matrix M (K x p), its
SVD and the latent scores, for `PLS(..., analysis="device")`.

The reference builds M on the host and calls LAPACK on it (pls_classes.py:258-266 mct, 576-586 rb, 854-866 cst,
1131-1143 csb, 1441-1489 mb / cmb; class_functions.py:98-123 `_run_pls`, 126-162 `_run_pls_contrast`).  Here M is never the operand of a
factorisation: every method's M is `Coef^T W` for a fixed coefficient matrix `Coef` (rows x K) and a data matrix W
already on the device (X itself, or its block z-scored copy Z for the behaviour methods), so

    M M^T = Coef^T (W W^T) Coef            K x K, from the Gram matrix the permutation test needs anyway
    [U, s^2] = eig(M M^T)                  the Jacobi kernel (one warp up to K = 32, one CTA up to K = 112)
    V = W^T (Coef U diag(1/s))             one pass over W (salience kernel)
    X_latent = X V                         one pass over X (xv kernel)

Differences from the host path, all inherent to going through the Gram matrix:
  * the sign of each latent variable is fixed by convention (largest-magnitude entry of the design-side vector
    positive) instead of by LAPACK's internals -- the pair (U_k, V_k) may be the negative of the host path's;
  * singular values below 1e-7 of the largest, or at the rounding level of the Gram matrix (8 eps N |Coef|^2 max G_ii
    on the eigenvalue), are set to exactly 0 with a zero brain-side vector (the host path sees ~1e-13 noise there,
    which the permutation test's own 1e-12 threshold zeroes as well);
  * relative accuracy of s_k is ~1e-16 (s_1 / s_k)^2 rather than 1e-16 (s_1 / s_k).
The contrast methods have no SVD at all (U = contrasts), so their device path agrees with the host path to rounding.

A voxel-sharded engine (shard="voxels", mct / cst) holds only its columns of X: G is all-reduced (Engine.G), every
projection runs on the rank's slice and is gathered to p rows (`_project_x`), X V is all-reduced (Engine.xv).
"""
import numpy as np
import torch

from . import class_functions as cf

NULL_RTOL = 1e-7


def _eigh_desc(eng, B):
    """Eigen-decomposition of a small symmetric PSD device matrix: eigenvalues descending, vectors in columns (host)."""
    ev, U = eng.sym_eig(B[None])          # warp-level Jacobi up to K = 32, CTA-level up to 112 (csrc/split.cu)
    ev, U = eng.to_host(ev, U)
    return ev[0], U[0]


def _fix_signs(U):
    """Largest-magnitude entry of every column positive (first one on ties)."""
    j = np.argmax(np.abs(U), axis=0)
    sg = np.sign(U[j, np.arange(U.shape[1])])
    sg[sg == 0] = 1.0
    return U * sg


def _project(eng, W, coef):
    """W^T coef (p x K) for a device matrix W (rows x p) and host / device coefficients (rows x K)."""
    n = int(W.shape[0])
    ident = np.arange(n, dtype=np.int32)[None]
    coef = eng.to_device(coef, torch.float64)
    K = int(coef.shape[1])
    step = max(1, min(K, (150 * 1024 // 8 - n) // max(n, 1)))       # the kernel stages rows x K coefficients in smem
    if step >= K:
        return eng.salience(coef, ident, M=W)[0]
    return torch.cat([eng.salience(coef[:, k0:k0 + step].contiguous(), ident, M=W)[0] for k0 in range(0, K, step)],
                     dim=1)


def _project_x(eng, coef):
    """X^T coef (p x K) on every rank: the projection of this rank's columns, gathered when X is voxel-sharded (an
    engine without the `voxel_sharded` flag holds the whole of X)."""
    P = _project(eng, eng.X, coef)
    return eng.gather_voxels(P) if getattr(eng, "voxel_sharded", False) else P


def _svd_through_gram(eng, W, Gw, coef, project=None):
    """U (K x K), s (K,), V (p x K, device) of M = coef^T W given Gw = W W^T; `project(c)` = W^T c when W is not
    held as one matrix."""
    C = eng.to_device(coef, torch.float64)
    B = eng.quad_form(Gw, C)
    B = 0.5 * (B + B.T)
    ev, U = _eigh_desc(eng, B)
    U = _fix_signs(U)
    # eigenvalues at the rounding level of the Gram matrix are null latent variables
    Ch = np.asarray(coef, dtype=float)
    tau = 8.0 * np.finfo(float).eps * Ch.shape[0] * np.linalg.norm(Ch, 2) ** 2 * float(torch.diagonal(Gw).max())
    live = ev > max(NULL_RTOL ** 2 * max(float(ev.max()), 0.0), tau)
    s = np.sqrt(np.maximum(ev, 0.0))
    s = np.where(live, s, 0.0)
    inv = np.where(live, 1.0 / np.where(live, s, 1.0), 0.0)
    cv = np.asarray(coef) @ (U * inv)
    V = _project(eng, W, cv) if project is None else project(cv)
    return U, s, V


def task(eng, cond_order, mctype):
    """mct (pls_classes.py:258-266): X_means, X_mc, U, s, V (device), X_latent, Tvsc_orig."""
    A = cf._centring_operator(cond_order, mctype)
    Abar = cf._cell_mean_operator(cond_order)
    U, s, V = _svd_through_gram(eng, None, eng.G, A.T, project=lambda c: _project_x(eng, c))
    both = _project_x(eng, np.concatenate([Abar.T, A.T], axis=1))               # one pass: cell means and M
    K = A.shape[0]
    X_means, X_mc = both[:, :K].T.contiguous(), both[:, K:].T.contiguous()
    XL = eng.xv(V)
    X_means, X_mc, Vh, XL = eng.to_host(X_means, X_mc, V, XL)
    return dict(X_means=X_means, X_mc=X_mc, U=U, s=s, V=Vh, V_dev=V, X_latent=XL, Tvsc_orig=Abar @ XL)


def contrast_task(eng, cond_order, contrasts):
    """cst (pls_classes.py:854-866): R = cell means, U = contrasts, V = (C^T R)^T un-normalised, s = its column norms."""
    Abar = cf._cell_mean_operator(cond_order)
    E = Abar.T @ contrasts                                                     # N x L
    both = _project_x(eng, np.concatenate([Abar.T, E], axis=1))
    K = Abar.shape[0]
    R, V = both[:, :K].T.contiguous(), both[:, K:].contiguous()
    Ed = eng.to_device(E, torch.float64)
    VtV = eng.to_host(eng.quad_form(eng.G, Ed))                                  # V^T V in N-space
    VtV = 0.5 * (VtV + VtV.T)
    s = np.sqrt(np.maximum(np.diagonal(VtV), 0.0))
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = np.where(s > 0, 1.0 / s, 0.0)
    XL = eng.xv(V * eng.to_device(inv, torch.float64)[None, :])                # X @ normalize(V)
    R, Vh, XL = eng.to_host(R, V, XL)
    return dict(R=R, U=contrasts, s=s, V=Vh, V_dev=V, lvintercorrs=VtV, X_latent=XL, Tvsc_orig=Abar @ XL)


def _behaviour_matrices(eng, cond_order):
    """Block z-scored X (Z, dense, this call only) and the per-engine cache holding Gz = Z Z^T for the permutations."""
    from .bootstrap_permutation import _cell_offsets
    cells = _cell_offsets(cond_order)
    Xc, Z = eng.cell_standardize(cells)
    eng._behaviour = {"key": tuple(int(c) for c in cells), "Xc": Xc, "Gz": eng.gram_of(Z)}
    return Z, eng._behaviour["Gz"]


def behaviour(eng, Y, cond_order):
    """rb (pls_classes.py:576-586): R, U, s, V (device), X_latent."""
    Z, Gz = _behaviour_matrices(eng, cond_order)
    Cy = cf._behaviour_coefficients(Y, cond_order)
    U, s, V = _svd_through_gram(eng, Z, Gz, Cy)
    R = _project(eng, Z, Cy).T.contiguous()
    del Z
    XL = eng.xv(V)
    R, Vh, XL = eng.to_host(R, V, XL)
    return dict(R=R, U=U, s=s, V=Vh, V_dev=V, X_latent=XL)


def contrast_behaviour(eng, Y, cond_order, contrasts):
    """csb (pls_classes.py:1131-1143): R, U = contrasts, V = (C^T R)^T, s = its column norms, lvintercorrs = V^T V."""
    Z, Gz = _behaviour_matrices(eng, cond_order)
    Cy = cf._behaviour_coefficients(Y, cond_order)
    E = Cy @ contrasts
    both = _project(eng, Z, np.concatenate([Cy, E], axis=1))
    del Z
    K = Cy.shape[1]
    R, V = both[:, :K].T.contiguous(), both[:, K:].contiguous()
    Ed = eng.to_device(E, torch.float64)
    VtV = eng.to_host(eng.quad_form(Gz, Ed))
    VtV = 0.5 * (VtV + VtV.T)
    s = np.sqrt(np.maximum(np.diagonal(VtV), 0.0))
    XL = eng.xv(V)
    R, Vh, XL = eng.to_host(R, V, XL)
    return dict(R=R, U=contrasts, s=s, V=Vh, V_dev=V, lvintercorrs=VtV, X_latent=XL)


def multiblock(eng, pls_alg, cond_order, mctype, bscan, Ybscan, contrasts=None):
    """mb / cmb (pls_classes.py:1441-1489, 1799-1856; class_functions.py:454-516): the multiblock matrix (rows
    L2-normalised), U, s, V (device) and X V.  With W = [X; Zb] (Zb = block z-scored bscan rows of X) the
    un-normalised rows are C1^T W, their norms quadratic forms in Gw = W W^T."""
    from .bootstrap_permutation import _multiblock_state, _multiblock_columns
    co = np.asarray(cond_order)
    st = _multiblock_state(eng, co, bscan, keep_zb=True)
    N, Nb, Gw = eng.N, st["Nb"], st["Gw"]
    tcol, bcol, K = _multiblock_columns(co, bscan, Ybscan.shape[1])
    Lop = cf._cell_mean_operator(co) if pls_alg == "cmb" else cf._centring_operator(co, mctype)
    C1 = np.zeros((N + Nb, K))
    C1[:N, tcol] = Lop.T
    C1[N:, bcol] = cf._behaviour_coefficients(Ybscan, co[:, list(bscan)])
    C1d = eng.to_device(C1, torch.float64)
    d2row = eng.to_host(eng.nspace_coef(Gw, C1d[None])[0][0])                  # diag(C1^T Gw C1)
    with np.errstate(divide="ignore", invalid="ignore"):
        rn = np.where(d2row > 0, 1.0 / np.sqrt(np.where(d2row > 0, d2row, 1.0)), 0.0)
    Cn = C1 * rn[None, :]                                          # normalised rows (norm_opt, :503-505)

    def project(c):                                                # W^T c without holding W
        c = np.asarray(c)
        return _project(eng, eng.X, c[:N]) + _project(eng, st["Zb"], c[N:])
    if contrasts is None:
        U, s, V = _svd_through_gram(eng, None, Gw, Cn, project=project)
        both = project(Cn)
        M = both.T.contiguous()
    else:
        U = contrasts
        E = Cn @ contrasts
        both = project(np.concatenate([Cn, E], axis=1))
        M, V = both[:, :K].T.contiguous(), both[:, K:].contiguous()
        Ed = eng.to_device(E, torch.float64)
        VtV = eng.to_host(eng.quad_form(Gw, Ed))
        s = np.sqrt(np.maximum(np.diagonal(0.5 * (VtV + VtV.T)), 0.0))
    XV = eng.xv(V)                                                 # X @ V (un-normalised V)
    st.pop("Zb", None)
    M, Vh, XV = eng.to_host(M, V, XV)
    return dict(multiblock=M, U=U, s=s, V=Vh, V_dev=V, XV=XV, rows_b=st["rows_b"], raw_sq=float(d2row.sum()))
