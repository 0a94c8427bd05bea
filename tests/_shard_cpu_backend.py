"""CPU stand-in for the stages of the fused row-sharded loss (fp64 torch), TEST ONLY: lets the partition /
exchange logic of kccotgan_b200.sharded.ShardedMixedLoss run under gloo without a GPU."""
import math

import torch


class CpuMixedShardBackend:
    """fp64 stand-in for kccotgan_b200.sharded.CudaMixedShardBackend (TEST ONLY): the same five stages on this rank's
    samples, the in-kernel mailbox exchange of the persistent Sinkhorn kernels replaced by all-reduces on `group`.
    Arithmetic follows gan_utils.py:14-17, :34-38, :151-164 and SURVEY Appendix A in the units of sinkhorn_persist.cu
    (log2 domain, cost shifted by the all-reduced minimum)."""

    def __init__(self, B, K, T, J, s, eps, L, row0, Brows, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.B, self.K, self.T, self.J, self.s, self.eps, self.L = B, K, T, J, float(s), float(eps), int(L)
        self.row0, self.Brows, self.group = row0, Brows, group
        self.k = math.log2(math.e) / self.eps
        self.ahat = -math.log2(B)
        self.shift = torch.zeros(3, dtype=torch.float64)

    def _ar(self, t, op):
        if self.dist.is_initialized() and self.dist.get_world_size(self.group) > 1:
            self.dist.all_reduce(t, op=op, group=self.group)
        return t

    def cost_fwd(self, real, fake, h_fake, m_real, h_real, m_fake):
        r0, r1, s = self.row0, self.row0 + self.Brows, self.s
        X, Y = real.double(), fake.double()
        hf, mr, hr, mf = (t.double() for t in (h_fake, m_real, h_real, m_fake))
        self.inputs = (X, Y, hf, mr, hr, mf)

        def block(a_rows, b_all, h_rows, M_all):
            D = ((a_rows[:, None, :] - b_all[None, :, :]) ** 2).sum(-1)
            Ht = h_rows[:, :-1, :].reshape(h_rows.shape[0], -1)
            dM = (M_all[:, 1:, :] - M_all[:, :-1, :]).reshape(M_all.shape[0], -1)
            return s * D + s * Ht @ dM.T
        self.C3 = torch.stack([block(X[r0:r1], Y, hf[r0:r1], mr), block(X[r0:r1], X, hr[r0:r1], mr),
                               block(Y[r0:r1], Y, hf[r0:r1], mf)])
        self.shift.copy_(self.C3.reshape(3, -1).min(dim=1).values)
        return self.shift

    def _chat(self):
        return (self.C3 - self.shift[:, None, None]) * self.k

    def sinkhorn_fwd(self):
        dist = self.dist
        Ch = self._chat()
        B, L = self.B, self.L
        self.u_hist = torch.zeros(3, L + 1, self.Brows, dtype=torch.float64)
        self.v_hist = torch.zeros(3, L + 1, B, dtype=torch.float64)
        ln2 = math.log(2)
        for it in range(L):
            v = self.v_hist[:, it]
            u = self.ahat - torch.logsumexp((v[:, None, :] - Ch) * ln2, dim=2) / ln2
            self.u_hist[:, it + 1] = u
            t = u[:, :, None] - Ch
            m = t.max(dim=1).values
            self._ar(m, dist.ReduceOp.MAX)
            ssum = torch.exp2(t - m[:, None, :]).sum(dim=1)
            self._ar(ssum, dist.ReduceOp.SUM)
            self.v_hist[:, it + 1] = self.ahat - (m + torch.log2(ssum))
        self.nits = L
        pi = torch.exp2(self.u_hist[:, L][:, :, None] + self.v_hist[:, L][:, None, :] - Ch)
        return torch.stack([pi.sum(dim=(1, 2)), (pi * Ch).sum(dim=(1, 2))], dim=1)

    def sinkhorn_bwd(self, g3):
        dist = self.dist
        Ch = self._chat()
        ce = (self.C3 - self.shift[:, None, None]) / self.eps
        n = self.nits
        g = g3.double()[:, None, None]
        pi = g * torch.exp2(self.u_hist[:, n][:, :, None] + self.v_hist[:, n][:, None, :] - Ch)
        Cbar = pi * (1 - ce)
        ubar = (pi * ce).sum(dim=2)
        vbar = (pi * ce).sum(dim=1)
        self._ar(vbar, dist.ReduceOp.SUM)
        for k in range(n, 0, -1):
            uk = self.u_hist[:, k][:, :, None] - self.ahat
            Pv = torch.exp2(uk + self.v_hist[:, k][:, None, :] - Ch)
            Cbar = Cbar + Pv * vbar[:, None, :]
            ub = (ubar if k == n else torch.zeros_like(ubar)) - (Pv * vbar[:, None, :]).sum(dim=2)
            Pu = torch.exp2(uk + self.v_hist[:, k - 1][:, None, :] - Ch)
            Cbar = Cbar + Pu * ub[:, :, None]
            cs = (Pu * ub[:, :, None]).sum(dim=1)
            self._ar(cs, dist.ReduceOp.SUM)
            vbar = -cs
        self.Cbar3 = Cbar
        return Cbar

    def cost_bwd(self, XYcol, YYcol):
        X, Y, hf, mr, hr, mf = self.inputs
        r0, r1, s = self.row0, self.row0 + self.Brows, self.s
        Cxy, Cxx, Cyy = self.Cbar3[0], self.Cbar3[1], self.Cbar3[2]
        XYcol, YYcol = XYcol.double(), YYcol.double()
        Yl = Y[r0:r1]
        # fake rows j: sum_i Cxy[i, j] (y_j - x_i) + sum_c (Cyy[j, c] + Cyy[c, j]) (y_j - y_c)
        w_x = XYcol.T                                        # [Brows, B]: weight of x_i
        w_y = Cyy + YYcol.T                                  # [Brows, B]: weight of y_c
        g_fake = 2 * s * ((w_x.sum(1) + w_y.sum(1))[:, None] * Yl - w_x @ X - w_y @ Y)

        def dM(M):
            return (M[:, 1:, :] - M[:, :-1, :]).reshape(M.shape[0], -1)

        def h_grad(Cb, M):
            out = torch.zeros(self.Brows, self.T, self.J, dtype=torch.float64)
            out[:, :-1, :] = (s * Cb @ dM(M)).reshape(self.Brows, self.T - 1, self.J)
            return out

        def m_grad(Cb, h_rows):
            gd = (s * Cb.T @ h_rows[:, :-1, :].reshape(self.Brows, -1)).reshape(self.B, self.T - 1, self.J)
            out = torch.zeros(self.B, self.T, self.J, dtype=torch.float64)
            out[:, 1:, :] += gd
            out[:, :-1, :] -= gd
            return out
        gh_fake = h_grad(Cxy, mr) + h_grad(Cyy, mf)
        gh_real = h_grad(Cxx, mr)
        gm_real = m_grad(Cxy, hf[r0:r1]) + m_grad(Cxx, hr[r0:r1])
        gm_fake = m_grad(Cyy, hf[r0:r1])
        return g_fake, gh_fake, gm_real, gh_real, gm_fake
