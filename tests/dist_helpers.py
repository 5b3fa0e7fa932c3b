"""CPU stand-in for the CUDA backend of ``gcs_admm_b200.dist.DistributedADMM`` (tests only):
the x-update is the C oracle's, the edge/dual/residual/control arithmetic is restated in numpy with the
same formulas as the kernels (csrc/gcsadmm.cu edge_frames_kernel in global frames / control_kernel)."""
import ctypes as C

import numpy as np
import torch

from c_oracle import lib as olib


class OracleBackend:
    def __init__(self, lp, max_it=1000, **p):
        self.lp = lp
        L = olib()
        self.nH_own = int(lp.he_off[-1])
        self.nHall = self.nH_own + int(lp.nH_ghost)
        assert self.nHall == 2 * lp.nE
        self.h = L.gcso_create(lp.nV, lp.nE, np.ascontiguousarray(lp.poly_off, np.int32), np.ascontiguousarray(lp.polyA, np.float64).reshape(-1),
                               np.ascontiguousarray(lp.polyb, np.float64), np.ascontiguousarray(lp.he_off, np.int32),
                               np.ascontiguousarray(lp.he_edge, np.int32), np.ascontiguousarray(lp.he_out, np.int32),
                               np.ascontiguousarray(lp.edge_he_tail, np.int32), np.ascontiguousarray(lp.edge_he_head, np.int32),
                               int(lp.src), int(lp.dst), np.ascontiguousarray(lp.cent, np.float64).reshape(-1))
        self.p = dict(rho0=1.0, tau_incr=2.0, tau_decr=2.0, nu=10.0, frac=0.1, eps_abs=1e-4, eps_rel=1e-3, max_it=max_it)
        self.p.update(p)
        self.xc = torch.zeros(self.nHall, 5, dtype=torch.float64)
        self.mu = np.zeros((self.nH_own, 5))
        self.z = np.zeros((lp.nE, 5))
        self.sums = torch.zeros(8, dtype=torch.float64)
        self.rho, self.mu_scale, self.it = self.p["rho0"], 1.0, 0
        self.converged = self.diverged = False
        self.pri_seq, self.dual_seq, self.rho_seq = [0.0], [0.0], [self.rho]

    def vertex_update(self):
        L = olib()
        pad = np.zeros((self.nHall, 5))
        pad[:self.nH_own] = self.mu * self.mu_scale
        L.gcso_set_state(self.h, self.xc.numpy().reshape(-1).copy(), pad.reshape(-1), self.z.reshape(-1).copy(), float(self.rho), int(self.it))
        L.gcso_vertex_update_all(self.h)
        xc, mu, z = np.zeros((self.nHall, 5)), np.zeros((self.nHall, 5)), np.zeros((self.lp.nE, 5))
        L.gcso_get_state(self.h, xc.reshape(-1), mu.reshape(-1), z.reshape(-1))
        self.xc[:self.nH_own] = torch.from_numpy(xc[:self.nH_own])

    def edge_update(self):
        lp, xc = self.lp, self.xc.numpy()
        zn = 0.5 * (xc[lp.edge_he_tail] + xc[lp.edge_he_head])
        w = lp.edge_counted.astype(float)[:, None]
        dz2, z2 = float(np.sum(w * (zn - self.z) ** 2)), float(np.sum(w * zn * zn))
        self.z = zn
        r = zn[lp.he_edge] - xc[:self.nH_own]
        self.mu = self.mu * self.mu_scale + r
        self.sums[:] = torch.tensor([float(np.sum(r * r)), dz2, float(np.sum(xc[:self.nH_own] ** 2)), z2, float(np.sum(self.mu ** 2)), 0.0, 0.0, 0.0], dtype=torch.float64)

    def control(self):
        p, s = self.p, self.sums.numpy()
        self.it += 1
        pri, dual = float(np.sqrt(s[0])), self.rho * float(np.sqrt(2.0 * s[1]))
        scale = 1.0
        if pri >= p["nu"] * dual and self.it < p["frac"] * p["max_it"]:
            self.rho *= p["tau_incr"]; scale = 1.0 / p["tau_incr"]
        elif dual >= p["nu"] * pri and self.it < p["frac"] * p["max_it"]:
            self.rho *= 1.0 / p["tau_decr"]; scale = p["tau_incr"]
        self.mu_scale = scale
        eps_pri = np.sqrt(self.lp.n_x_global) * p["eps_abs"] + p["eps_rel"] * max(np.sqrt(s[2]), np.sqrt(2 * s[3]))
        eps_dual = np.sqrt(self.lp.n_mu_global) * p["eps_abs"] + p["eps_rel"] * scale * np.sqrt(s[4])
        self.pri_seq.append(pri); self.dual_seq.append(dual); self.rho_seq.append(self.rho)
        if pri < eps_pri and dual < eps_dual:
            self.converged = True

    def status(self):
        return dict(iterations=self.it, converged=self.converged, diverged=self.diverged, rho=self.rho)
