"""numpy stand-in for the library phases of one column-sharded update (TEST DOUBLE).

Implements, on CPU torch tensors, exactly the buffer contract of include/ces_b200.h ("sums", "cuu",
"e_all", "ut_all", "scalars"; rank-major blocks, zero-padded shard columns) so that
ces_b200.engine.run_phases / run_host_phases -- the host orchestration of the collectives -- can be
exercised with gloo and world_size 2 on a machine without a GPU.  It is never imported by the product.
"""
import numpy as np
import torch


class NumpyPhases(object):
    def __init__(self, p, k, J, rank, nranks, y, Gamma, mu, Sigma0, ustar):
        self.p, self.k, self.J, self.rank, self.nranks = p, k, J, rank, nranks
        self.Jl = -(-J // nranks)
        self.ldJ = (self.Jl + 15) // 16 * 16
        self.ldp = (p + 15) // 16 * 16
        lo = min(J, rank * self.Jl)
        self.lo, self.hi = lo, min(J, lo + self.Jl)
        self.cols = self.hi - self.lo
        self.y, self.Gamma, self.mu, self.Sigma0, self.ustar = y, Gamma, mu.reshape(p, 1), Sigma0, ustar.reshape(p, 1)
        self.buf = {
            "sums": torch.zeros(1, k + p, dtype=torch.float64),
            "cuu": torch.zeros(p, self.ldp, dtype=torch.float64),
            "e_all": torch.zeros(nranks * k, self.ldJ, dtype=torch.float64),
            "ut_all": torch.zeros(nranks * p, self.ldJ, dtype=torch.float64),
            "scalars": torch.zeros(1, 16, dtype=torch.float64),
        }

    def buffer(self, name):
        return self.buf[name]

    def bind(self, rule, U, G, xi, switch=1.0, fixed_h=None, peer=False):
        """The phases of ces_b200.engine.run_phases.  ``peer``: add stand-ins for the peer pulls (ces_peer_gather: an
        in-place all-gather of "e_all" / "ut_all" over the default group; ces_peer_gather_wait: nothing to wait for)."""
        self.rule, self.U, self.G, self.xi, self.switch, self.fixed_h = rule, U, G, xi, switch, fixed_h
        ldk = (self.k + 15) // 16 * 16
        self.buf["cpp"] = torch.zeros(self.k, ldk, dtype=torch.float64)
        self.buf["p1"] = torch.zeros(self.p, ldk, dtype=torch.float64)
        self.buf["gram_e"] = torch.zeros(self.k, ldk, dtype=torch.float64)
        self.buf["gram_w"] = torch.zeros(self.k, ldk, dtype=torch.float64)
        return dict({"sums": self.sums, "centre": self.centre, "interact": self.interact, "interact_own": self.interact_own,
                     "interact_rest": self.interact_rest, "drift": self.drift, "update": self.update, "peek": self.peek,
                     "cpp": self.cpp, "resolve": self.resolve, "products": self.products,
                     "finish_factored": self.finish_factored, "spectral": self.spectral}, **self._peer(peer))

    def _peer(self, peer):
        if not peer:
            return {}

        def gather():
            import torch.distributed as dist

            for name, rows in (("e_all", self.k), ("ut_all", self.p)):
                b = self.buf[name]
                dist.all_gather_into_tensor(b, b[self.rank * rows:(self.rank + 1) * rows])
        return {"peer_gather": gather, "peer_wait": lambda: None}

    # ---- the pipelined host step in pieces (ces_host_*; ces_b200.engine.run_host_phases).  Needs a diagonal Gamma: a row
    # chunk of W = Gamma^-1 (G - y) is then a function of the same rows of G only.
    def bind_host(self, rule, U, G, xi, bounds, switch=1.0, peer=False):
        self.rule, self.U, self.G, self.xi, self.switch, self.fixed_h = rule, U, G, xi, switch, None
        self.bounds = list(bounds)
        self.W = np.zeros((self.k, self.cols))
        self.D_own = np.zeros((self.Jl, self.cols))
        self.calls = []
        return dict({"sums_g": self.h_sums_g, "centre_g": self.h_centre_g, "interact_chunk": self.h_interact_chunk,
                     "sums_u": self.h_sums_u, "centre_u": self.h_centre_u, "interact_own": self.h_interact_own,
                     "interact_rest": self.interact_rest, "drift": self.drift, "update": self.update}, **self._peer(peer))

    def _rows(self, c):
        return slice(self.bounds[c], self.bounds[c + 1])

    def h_sums_g(self, c):
        self.calls.append(("sums_g", c))
        self.buf["sums"][0, self._rows(c)] = torch.from_numpy(self.G[self._rows(c)].sum(axis=1))

    def h_centre_g(self, c, interact):
        self.calls.append(("centre_g", c, bool(interact)))
        k, r = self.k, self._rows(c)
        means = self.buf["sums"][0, r].numpy() / self.J
        e_all = self.buf["e_all"].numpy()
        e_all[self.rank * k + r.start:self.rank * k + r.stop] = 0.0
        e_all[self.rank * k + r.start:self.rank * k + r.stop, :self.cols] = self.G[r] - means[:, None]
        self.W[r] = (self.G[r] - self.y[r, None]) / np.diag(self.Gamma)[r, None]
        if interact:
            self.h_interact_chunk(c)

    def h_interact_chunk(self, c):
        self.calls.append(("interact_chunk", c))
        k, r = self.k, self._rows(c)
        if len(self.bounds) > 2:            # several chunks: the own block's D panel accumulates over them
            E = self.buf["e_all"].numpy()[self.rank * k + r.start:self.rank * k + r.stop, :self.Jl]
            self.D_own += (E.T @ self.W[r]) / self.J

    def h_sums_u(self):
        k, c = self.k, self.cols
        E = self.buf["e_all"].numpy()[self.rank * k:(self.rank + 1) * k, :c]
        R = self.G - self.y[:, None]
        S = self.buf["scalars"][0].numpy()
        S[3] = (np.einsum("ij,ij->j", E, E / np.diag(self.Gamma)[:, None]) ** 2).sum()
        S[4] = (np.einsum("ij,ij->j", R, self.W) ** 2).sum()
        self.buf["sums"][0, k:] = torch.from_numpy(self.U.sum(axis=1))

    def h_centre_u(self):
        p, k, c = self.p, self.k, self.cols
        means = self.buf["sums"][0, k:].numpy() / self.J
        Ut = self.U - means[:, None]
        self.Z = np.linalg.solve(self.Sigma0, self.U - self.mu)
        ut_all = self.buf["ut_all"].numpy()
        ut_all[self.rank * p:(self.rank + 1) * p] = 0.0
        ut_all[self.rank * p:(self.rank + 1) * p, :c] = Ut
        S = self.buf["scalars"][0].numpy()
        S[1] = (Ut ** 2).sum()
        S[2] = ((self.U - self.ustar) ** 2).sum()
        alpha = 1.0 / self.J if self.rule == "eks" else 1.0 / (self.J - 1)
        C = alpha * (Ut @ Ut.T)
        if self.rank == 0:
            C = C + 1e-8 * np.eye(p)
        cuu = self.buf["cuu"].numpy()
        cuu[:] = 0.0
        cuu[:, :p] = C

    def h_interact_own(self):
        p, k = self.p, self.k
        self.C = self.buf["cuu"].numpy()[:, :p].copy()
        if len(self.bounds) <= 2:           # single chunk: the whole own block here
            E = self.buf["e_all"].numpy()[self.rank * k:(self.rank + 1) * k, :self.Jl]
            self.D_own = (E.T @ self.W) / self.J
        Ut = self.buf["ut_all"].numpy()[self.rank * p:(self.rank + 1) * p, :self.Jl]
        self.V = Ut @ self.D_own
        self._ssq = (self.D_own ** 2).sum()

    def sums(self):
        s = np.concatenate([self.G.sum(axis=1), self.U.sum(axis=1)])
        self.buf["sums"][0] = torch.from_numpy(s)

    def centre(self):
        p, k, c = self.p, self.k, self.cols
        means = self.buf["sums"][0].numpy() / self.J
        E = self.G - means[:k, None]
        R = self.G - self.y[:, None]
        self.W = np.linalg.solve(self.Gamma, R)
        Ut = self.U - means[k:, None]
        self.Z = np.linalg.solve(self.Sigma0, self.U - self.mu)
        e_all, ut_all = self.buf["e_all"].numpy(), self.buf["ut_all"].numpy()
        e_all[self.rank * k:(self.rank + 1) * k] = 0.0
        e_all[self.rank * k:(self.rank + 1) * k, :c] = E
        ut_all[self.rank * p:(self.rank + 1) * p] = 0.0
        ut_all[self.rank * p:(self.rank + 1) * p, :c] = Ut
        S = self.buf["scalars"][0].numpy()
        S[1] = (Ut ** 2).sum()
        S[2] = ((self.U - self.ustar) ** 2).sum()
        S[3] = (np.einsum("ij,ij->j", E, np.linalg.solve(self.Gamma, E)) ** 2).sum()
        S[4] = (np.einsum("ij,ij->j", R, self.W) ** 2).sum()
        alpha = 1.0 / self.J if self.rule == "eks" else 1.0 / (self.J - 1)
        C = alpha * (Ut @ Ut.T)
        if self.rank == 0:
            C = C + 1e-8 * np.eye(p)
        cuu = self.buf["cuu"].numpy()
        cuu[:] = 0.0
        cuu[:, :p] = C

    def _block(self, s, W):
        """Rank s's block of D = (1/J) E^T W: its ||.||_F^2 into _ssq, its share of V = U~ D into V."""
        p, k = self.p, self.k
        e_all, ut_all = self.buf["e_all"].numpy(), self.buf["ut_all"].numpy()
        D = (e_all[s * k:(s + 1) * k, :self.Jl].T @ W) / self.J
        self._ssq += (D ** 2).sum()
        self.V += ut_all[s * p:(s + 1) * p, :self.Jl] @ D

    def _loops(self, W):
        self.V, self._ssq = np.zeros((self.p, self.cols)), 0.0
        for s in range(self.nranks):
            self._block(s, W)
        return self._ssq

    def interact(self, skip=False):
        self.C = self.buf["cuu"].numpy()[:, :self.p].copy()
        if not skip:
            self.buf["scalars"][0, 0] = self._loops(self.W)

    def interact_own(self):
        self.C = self.buf["cuu"].numpy()[:, :self.p].copy()
        self.V, self._ssq = np.zeros((self.p, self.cols)), 0.0
        self._block(self.rank, self.W)

    def interact_rest(self):
        for i in range(1, self.nranks):
            self._block((self.rank + i) % self.nranks, self.W)
        self.buf["scalars"][0, 0] = self._ssq

    def products(self):
        p, k, c = self.p, self.k, self.cols
        self.C = self.buf["cuu"].numpy()[:, :p].copy()
        E = self.buf["e_all"].numpy()[self.rank * k:(self.rank + 1) * k, :c]
        Ut = self.buf["ut_all"].numpy()[self.rank * p:(self.rank + 1) * p, :c]
        for name, val in (("p1", Ut @ E.T), ("gram_e", E @ E.T), ("gram_w", self.W @ self.W.T)):
            b = self.buf[name].numpy()
            b[:] = 0.0
            b[:, :k] = val

    def finish_factored(self):
        k = self.k
        self.V = (self.buf["p1"].numpy()[:, :k] @ self.W) / self.J
        ssq = (self.buf["gram_e"].numpy()[:, :k] * self.buf["gram_w"].numpy()[:, :k]).sum() / self.J ** 2
        self.buf["scalars"][0, 0] = ssq if self.rank == 0 else 0.0

    def peek(self):
        S = self.buf["scalars"][0].numpy()
        self.h_kept = self.fixed_h if self.fixed_h is not None else 1.0 / (np.sqrt(S[0]) + 1e-8)
        return self.h_kept

    def cpp(self):
        k, c = self.k, self.cols
        E = self.buf["e_all"].numpy()[self.rank * k:(self.rank + 1) * k, :c]
        out = self.buf["cpp"].numpy()
        out[:] = 0.0
        out[:, :k] = (E @ E.T) / self.J

    def spectral(self):
        k = self.k
        lam = np.linalg.eigvals(np.linalg.solve(self.Gamma, self.buf["cpp"].numpy()[:, :k])).real.max()
        self.h_kept = 1.0 / lam
        return lam

    def resolve(self):
        k = self.k
        M = self.h_kept * self.buf["cpp"].numpy()[:, :k] + self.Gamma
        R = self.G - self.y[:, None]
        self._loops(np.linalg.solve(M, R))

    def drift(self):
        p, c = self.p, self.cols
        Ut = self.buf["ut_all"].numpy()[self.rank * p:(self.rank + 1) * p, :c]
        alpha = (p + 1.0) / self.J
        self.T = -self.V - self.C @ self.Z + self.switch * alpha * Ut
        self.buf["scalars"][0, 5] = np.abs(self.T).max() if c else 0.0

    def update(self, keep=False):
        p, c = self.p, self.cols
        S = self.buf["scalars"][0].numpy()
        Ut = self.buf["ut_all"].numpy()[self.rank * p:(self.rank + 1) * p, :c]
        alpha = (p + 1.0) / self.J
        if self.rule == "aldi_constant":
            h = 0.1 / S[5]
            out = self.U + h * self.T + np.sqrt(2 * h) * (np.linalg.cholesky(self.C) @ self.xi)
        else:
            h = self.h_kept if keep else (self.fixed_h if self.fixed_h is not None else 1.0 / (np.sqrt(S[0]) + 1e-8))
            if self.rule == "aldi":
                out = (self.U + h * alpha * Ut - h * self.V - h * (self.C @ self.Z)
                       + np.sqrt(2 * h) * (np.linalg.cholesky(self.C) @ self.xi))
            elif self.rule == "eki":
                out = self.U - h * self.V
            else:
                M = self.Sigma0 + h * self.C
                rhs = self.U - h * self.V + h * (self.C @ np.linalg.solve(self.Sigma0, self.mu))
                out = self.Sigma0 @ np.linalg.solve(M, rhs) + np.sqrt(2 * h) * (np.linalg.cholesky(self.C) @ self.xi)
        self.out, self.hk = out, h
        self.metrics = {"self-bias": S[1] / self.J, "bias": S[2] / self.J, "self-bias-data": S[3] / self.J,
                        "bias-data": S[4] / self.J}
