"""numpy restatement of the saved model (vpca_pca_loadings_* / vpca_pca_model_terms / vpca_score_*, include/vpca.h,
DESIGN.md 3.7), shared by tests/test_model.py and tests/test_model_gpu.py.  The reference has no projection step: this
pins the formula the library documents, not reference output."""
import numpy as np

from oracle import oracle


def np_model(S, X_fit, U, evals):
    """S: fitted N x N Gram; X_fit: N x V fitted cells; U (N x k), evals (k): the fitted PCs.  Returns the model fields
    {loadings L = X_fit^T U, carriers n = column sums of X_fit, eigenvalues, col_sums a = sum_f u_f, rowsum_dots
    b = sum_f (rs_f / N) u_f, matrix_mean, n_fitted}."""
    n = S.shape[0]
    _, row_sums, _ = oracle.np_center(S)
    U = np.asarray(U, np.float64)
    X = np.asarray(X_fit, np.float64)
    return dict(loadings=X.T @ U, carriers=np.asarray(X_fit, np.int64).sum(axis=0).astype(np.int32),
                eigenvalues=np.asarray(evals, np.float64), col_sums=U.sum(axis=0), rowsum_dots=(row_sums / float(n)) @ U,
                matrix_mean=float(row_sums.sum()) / float(n) / float(n), n_fitted=n)


def np_score(model, X_study, model_rows):
    """X_study: M x V_s study cells; model_rows[v]: the model row of study variant v (-1: not in the model).
    y_pc = (((T_pc - (r_p / N) a_c) - b_c) + mean a_c) / lambda_c with T = X L[rows], r = X n[rows] (exact)."""
    rows = np.asarray(model_rows, np.int64)
    keep = rows >= 0
    Xs = np.asarray(X_study, np.int64)[:, keep]
    L = np.asarray(model["loadings"], np.float64)[rows[keep]]
    T = Xs.astype(np.float64) @ L
    r = (Xs @ np.asarray(model["carriers"], np.int64)[rows[keep]]).astype(np.float64)
    a, b = np.asarray(model["col_sums"]), np.asarray(model["rowsum_dots"])
    n = float(model["n_fitted"])
    return (((T - (r / n)[:, None] * a[None, :]) - b[None, :]) + model["matrix_mean"] * a[None, :]) / \
        np.asarray(model["eigenvalues"])[None, :]
