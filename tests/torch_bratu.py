"""The Bratu problem written as device callables in plain torch (test and benchmark helper).

``res`` restates P(u) = L u + alpha D u + lambda e^u with torch elementwise ops in the reference's operation order
(DESIGN.md section 5, oracle/gnk_oracle.py:BratuOracle.operator); ``jac`` returns the CSR Jacobian
-(L + alpha D + lambda diag(e^u)) as a torch sparse CSR tensor: the index pattern is fixed and built once, the values
are new at every call.  Only torch.exp differs from the host's exp, so trajectories agree with the reference's to the
bounds the native path is held to, not bit for bit."""
import numpy as np
import scipy.sparse as sp
import torch


class TorchBratu:
    def __init__(self, pb, oracle, y, device, index_dtype=torch.int64):
        """pb: the package's BratuPdeProblem (its host matrices give the pattern and L + alpha D), oracle: the
        BratuOracle of the same grid (the constants of the residual)"""
        self.m, self.c_lap, self.c_adv, self.lam = oracle.m, oracle.c_lap, oracle.c_adv, oracle.lam
        self.n = self.m * self.m
        self.y = torch.as_tensor(np.asarray(y, dtype=np.float64), device=device)
        # L + alpha D as StencilJacobian.tocsr adds them; the diagonal is stored for every row
        LD = sp.csr_array(pb.laplace2d + pb.ALPHA * pb.partial_diff_x)
        LD.sort_indices()
        self.crow = torch.as_tensor(LD.indptr.astype(np.int64), device=device).to(index_dtype)
        self.col = torch.as_tensor(LD.indices.astype(np.int64), device=device).to(index_dtype)
        self.ld_val = torch.as_tensor(LD.data, device=device)
        rows = np.repeat(np.arange(self.n), np.diff(LD.indptr))
        self.diag_pos = torch.as_tensor(np.nonzero(LD.indices == rows)[0], device=device)
        self.jac_calls = 0

    def operator(self, u):
        m, c = self.m, self.c_lap
        U = u.reshape(m, m)
        up, left, right, down = (torch.zeros_like(U) for _ in range(4))
        up[1:, :] = (-c) * U[:-1, :]
        left[:, 1:] = (-c) * U[:, :-1]
        right[:, :-1] = (-c) * U[:, 1:]
        down[:-1, :] = (-c) * U[1:, :]
        lap = up + left
        lap += (4.0 * c) * U
        lap += right
        lap += down
        adv = (-self.c_adv) * U
        adv[:-1, :] += self.c_adv * U[1:, :]
        out = lap + adv
        if self.lam != 0:
            out = out + self.lam * torch.exp(U)
        return out.reshape(-1)

    def res(self, u):
        return self.y - self.operator(u)

    def jac(self, u):
        self.jac_calls += 1
        val = self.ld_val.clone()
        if self.lam != 0:
            val[self.diag_pos] = val[self.diag_pos] + self.lam * torch.exp(u)
        return torch.sparse_csr_tensor(self.crow, self.col, -val, size=(self.n, self.n))
