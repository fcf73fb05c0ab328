"""fp64 ground truth of GP.predict (TEST INFRASTRUCTURE ONLY): the textbook GP prediction with the explicit n x n
covariance, in the notation of oracle/gp_oracle.py.  A plain module (no tests)."""
from typing import Sequence, Tuple

import torch

from oracle.gp_oracle import variances

Tensor = torch.Tensor


def predict(X: Tensor, Vs: Sequence[Tensor], Vs_new: Sequence[Tensor], lvs: Tensor) -> Tuple[Tensor, Tensor]:
    """Posterior mean and variance of the noise-free latents at new rows (the GP prediction of train_gppvae.py:223-261,
    with its variance), through the textbook forms with the explicit n x n covariance
    K = sum_i v_i V_i V_i^T + vn I and the cross-covariance K*t = sum_i v_i V*_i V_i^T:

        mean = K*t K^-1 X  (m x L),    var = diag(K** - K*t K^-1 Kt*)  (m x 1, one value shared by the L columns)."""
    with torch.no_grad():
        vs = variances(lvs)
        n, L = X.shape
        K = vs[-1] * torch.eye(n, dtype=X.dtype)
        Kst = torch.zeros(Vs_new[0].shape[0], n, dtype=X.dtype)
        Kss = torch.zeros(Vs_new[0].shape[0], 1, dtype=X.dtype)
        for i, (Vi, Vn) in enumerate(zip(Vs, Vs_new)):
            K = K + vs[i] * Vi.mm(Vi.t())
            Kst = Kst + vs[i] * Vn.mm(Vi.t())
            Kss = Kss + vs[i] * (Vn * Vn).sum(1, keepdim=True)
        A = torch.linalg.solve(K, torch.cat([X, Kst.t()], 1))
        return Kst.mm(A[:, :L]), Kss - (Kst * A[:, L:].t()).sum(1, keepdim=True)
