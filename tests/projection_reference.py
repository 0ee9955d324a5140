"""numpy restatement of the projection of held-out samples onto fitted PCs (vpca_project_pca, include/vpca.h), shared by
tests/test_projection.py and tests/test_projection_gpu.py.  The reference has no projection step: this pins the formula
the library documents, not reference output."""
import numpy as np

from oracle import oracle


def np_project(S, X, U, evals):
    """S: fitted N x N Gram; X: M x N cross counts (variants each projected sample shares with each fitted one); U (N x k),
    evals (k): the fitted PCs.  The reference's centring (VariantsPca.scala:199-223) applied to the new rows with the
    fitted statistics, same operation order:  c_pf = ((X_pf - rowMean_p) - rowSums_f / N) + matrixMean,
    rowMean_p = (sum_f X_pf) / N; then y_pc = (sum_f c_pf u_fc) / lambda_c.  Returns (C_x, Y)."""
    n = S.shape[0]
    _, row_sums, _ = oracle.np_center(S)
    matrix_mean = float(row_sums.sum()) / float(n) / float(n)     # integer-valued partial sums: exact in any order
    rs = np.asarray(X, np.int64).sum(axis=1).astype(np.float64)    # exact (foldLeft(0D) of :206 on the new row)
    Cx = ((np.asarray(X, np.float64) - (rs / float(n))[:, None]) - (row_sums / float(n))[None, :]) + matrix_mean
    return Cx, (Cx @ np.asarray(U, np.float64)) / np.asarray(evals, np.float64)[None, :]
