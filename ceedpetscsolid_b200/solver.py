"""Newton-Krylov-p-multigrid harness: the PETSc pieces the reference configures in
/root/reference/elasticity.c:378-603 and drives in :632-676, restated so that the operator
apply can be turned into "SNES solve time" without PETSc (SURVEY.md 8(f) rows 2-4, App. H):

  outer KSP      preconditioned CG, natural norm sqrt(r.z), rtol 1e-10, zero initial guess  (:504-507)
  PC             PCMG multiplicative V-cycle, 3 pre + 3 post smoothing steps per level      (:588-590)
  smoother       Chebyshev + point-Jacobi; lambda_max estimated by a few CG steps on the
                 Jacobi-preconditioned level operator, interval [0.1, 1.1] * lambda_max     (:539-552)
  coarse level   p = 1 operator ASSEMBLED by colouring its (linear) action                   (src/misc.c:151-183)
                 reference: GAMG on the AIJ matrix; here: Jacobi-PCG on the assembled ELL matrix
  SNES           Newton with load increments, warm start, rtol 1e-8                          (:595-601,:637-673)

Differences from PETSc that are inherent (SURVEY App. E.9, hard part 11): GAMG and PETSc's noisy-rhs PRNG
are not reproducible outside PETSc; the eigen-estimate rhs here is a seeded deterministic vector, the
coarse solve is Jacobi-PCG, the line search is a backtracking search on |F|.  Iteration counts are therefore
compared between the GPU operators and the CPU oracle under THIS harness (tests/test_gpu_solver.py).

The algorithms are written once over a small "level operations" interface; vectors are torch
tensors.  On CUDA tensors every vector operation is a libceed_b200.so kernel; on CPU tensors
(oracle runs) torch/numpy is used.
"""
import math
import time

import numpy as np
import torch

from .ceed import b2, lib

# --------------------------------------------------------------------------- vector kernels


class Vec:
    """BLAS-1 on torch tensors; CUDA tensors go through libceed_b200.so kernels."""

    def __init__(self, dist=None):
        self.dist = dist
        self._scratch = None
        self.weights = {}   # vector length -> weight vector (shared-dof layouts count every dof once)
        self._wtmp = {}

    def set_weight(self, n, w):
        """Inner-product weight (1 / number of ranks holding the dof) for the vectors of length n.  The weights are
        looked up by vector length: two DMs of the SAME length with DIFFERENT interface multiplicities cannot share one
        Vec -- refused here instead of silently taking the last one registered."""
        old = self.weights.get(int(n))
        if old is not None and old is not w and not torch.equal(old, w):
            raise ValueError(f"Vec.set_weight: two different dot-product weights for vectors of length {n}; "
                             "give the second DM its own Vec")
        self.weights[int(n)] = w

    def _weighted(self, a):
        w = self.weights.get(a.numel())
        if w is None:
            return a
        t = self._wtmp.get(a.numel())
        if t is None:
            t = self._wtmp[a.numel()] = torch.empty_like(a)
        self.pmult(t, a, w)
        return t

    def dot(self, a, b):
        if a.is_cuda:
            if self._scratch is None:
                self._scratch = torch.zeros(1, dtype=torch.float64, device=a.device)
            w = self.weights.get(a.numel())
            if w is None:
                b2(lib.b200_vec_dot(a.data_ptr(), b.data_ptr(), a.numel(), self._scratch.data_ptr()))
            else:   # (w .* a) . b in one pass, same rounding as the separate product
                b2(lib.b200_vec_dot_weighted(w.data_ptr(), a.data_ptr(), b.data_ptr(), a.numel(), self._scratch.data_ptr()))
            s = self._scratch
        else:
            s = torch.dot(self._weighted(a), b).reshape(1)
        if self.dist is not None and self.dist.get_world_size() > 1:
            s = s.clone()
            self.dist.all_reduce(s)
        return float(s.item())

    @staticmethod
    def axpy(y, alpha, x):  # y += alpha x
        if y.is_cuda:
            b2(lib.b200_vec_axpy(y.data_ptr(), float(alpha), x.data_ptr(), y.numel()))
        else:
            y.add_(x, alpha=float(alpha))

    @staticmethod
    def aypx(y, alpha, x):  # y = x + alpha y
        if y.is_cuda:
            b2(lib.b200_vec_aypx(y.data_ptr(), float(alpha), x.data_ptr(), y.numel()))
        else:
            y.mul_(float(alpha)).add_(x)

    @staticmethod
    def axpby(z, a, x, b, y):  # z = a x + b y
        if z.is_cuda:
            b2(lib.b200_vec_axpby(z.data_ptr(), float(a), x.data_ptr(), float(b), y.data_ptr(), z.numel()))
        else:
            torch.add(x * float(a), y, alpha=float(b), out=z)

    @staticmethod
    def pmult(w, x, y):  # w = x .* y
        if w.is_cuda:
            b2(lib.b200_vec_pointwise_mult(w.data_ptr(), x.data_ptr(), y.data_ptr(), w.numel()))
        else:
            torch.mul(x, y, out=w)

    @staticmethod
    def scale(x, a):
        if x.is_cuda:
            b2(lib.b200_vec_scale(x.data_ptr(), float(a), x.numel()))
        else:
            x.mul_(float(a))

    @staticmethod
    def copy(dst, src):
        dst.copy_(src)

    @staticmethod
    def zero(x):
        x.zero_()


# --------------------------------------------------------------------------- Krylov / smoothers


def pcg(V, A, b, x, M=None, rtol=1e-10, atol=1e-50, maxit=10000, work=None, hist=None):
    """Preconditioned CG with the natural norm sqrt(r.z) (KSPCG + KSP_NORM_NATURAL, elasticity.c:504-507).
    x is the initial guess and the result.  A(x, y): y = A x.  M(r, z): z = M^-1 r (None: identity).
    Returns (iterations, converged_reason, final natural residual norm)."""
    r, z, p, Ap = work if work is not None else [torch.zeros_like(b) for _ in range(4)]
    A(x, Ap)
    V.axpby(r, 1.0, b, -1.0, Ap)
    if M is None:
        V.copy(z, r)
    else:
        M(r, z)
    rz = V.dot(r, z)
    r0 = math.sqrt(abs(rz))
    if hist is not None:
        hist.append(r0)
    if r0 <= atol or r0 == 0.0:
        return 0, "atol", r0
    V.copy(p, z)
    for it in range(1, maxit + 1):
        A(p, Ap)
        pAp = V.dot(p, Ap)
        if pAp <= 0:
            return it, "indefinite", math.sqrt(abs(rz))
        alpha = rz / pAp
        V.axpy(x, alpha, p)
        V.axpy(r, -alpha, Ap)
        if M is None:
            V.copy(z, r)
        else:
            M(r, z)
        rz_new = V.dot(r, z)
        rn = math.sqrt(abs(rz_new))
        if hist is not None:
            hist.append(rn)
        if rn <= max(rtol * r0, atol):
            return it, "rtol", rn
        V.aypx(p, rz_new / rz, z)
        rz = rz_new
    return maxit, "maxit", math.sqrt(abs(rz))


def _guarded_ratio(num, den):
    """num / den of two scalars of a sync-free Krylov loop; 0 when the iteration has converged exactly or broken down
    (0/0), so the iterates freeze instead of turning into NaN (same rule as guarded_ratio in csrc/b200_runtime.cu)."""
    num, den = float(num), float(den)
    if den == 0.0:
        return 0.0
    a = num / den
    return a if math.isfinite(a) else 0.0


def jacobi_pcg_nosync(V, A, dinv, b, x, work, rtol, maxit, check_every=10):
    """Jacobi-preconditioned CG from a zero initial guess whose scalars (r.z, p.Ap) stay on the DEVICE:
    the loop enqueues kernels without waiting for them and looks at the residual norm only every
    `check_every` iterations (one host sync per check instead of two per iteration).  Used for the
    coarse-level solve, where an iteration is a few microseconds of device work.  Same arithmetic on
    CPU tensors (oracle runs), so iteration counts agree between the two.  Returns iterations run."""
    r, z, p, Ap = work
    dev = b.device
    if not hasattr(V, "_sc") or V._sc.device != dev:
        V._sc = torch.zeros(4, dtype=torch.float64, device=dev)  # [rz_a, rz_b, pAp, spare]
    sc = V._sc
    multi = V.dist is not None and V.dist.get_world_size() > 1

    def ddot(a_, b_, slot):
        out = sc[slot:slot + 1]
        if a_.is_cuda:
            w = V.weights.get(a_.numel())
            if w is None:
                b2(lib.b200_vec_dot(a_.data_ptr(), b_.data_ptr(), a_.numel(), out.data_ptr()))
            else:
                b2(lib.b200_vec_dot_weighted(w.data_ptr(), a_.data_ptr(), b_.data_ptr(), a_.numel(), out.data_ptr()))
        else:
            out.copy_(torch.dot(V._weighted(a_), b_).reshape(1))
        if multi:
            V.dist.all_reduce(out)
        return out

    x.zero_()
    V.copy(r, b)
    V.pmult(z, dinv, r)
    V.copy(p, z)
    cur, nxt = 0, 1
    ddot(r, z, cur)
    r0 = math.sqrt(abs(float(sc[cur].item())))
    if r0 == 0.0:
        return 0
    it = 0
    while it < maxit:
        for _ in range(check_every):
            A(p, Ap)
            ddot(p, Ap, 2)
            if x.is_cuda:
                b2(lib.b200_pcg_update(x.data_ptr(), r.data_ptr(), z.data_ptr(), p.data_ptr(), Ap.data_ptr(),
                                       dinv.data_ptr(), x.numel(), sc[cur:cur + 1].data_ptr(), sc[2:3].data_ptr()))
            else:
                a = _guarded_ratio(sc[cur], sc[2])
                x.add_(p, alpha=a)
                r.add_(Ap, alpha=-a)
                torch.mul(dinv, r, out=z)
            ddot(r, z, nxt)
            if p.is_cuda:
                b2(lib.b200_vec_aypx_dev(p.data_ptr(), z.data_ptr(), p.numel(), sc[nxt:nxt + 1].data_ptr(),
                                         sc[cur:cur + 1].data_ptr()))
            else:
                p.mul_(_guarded_ratio(sc[nxt], sc[cur])).add_(z)
            cur, nxt = nxt, cur
            it += 1
        rn = math.sqrt(abs(float(sc[cur].item())))  # the only host sync of this block of iterations
        if not math.isfinite(rn) or rn <= rtol * r0:
            break
    return it


def estimate_lambda_max(V, A, dinv, n, device, its=10, seed=0):
    """Largest eigenvalue of D^-1 A from `its` CG (Lanczos) steps with a deterministic rhs
    (KSPChebyshevEstEigSet + noisy rhs, elasticity.c:540-545; PETSc's PRNG is not reproducible here)."""
    # deterministic "noisy" rhs generated ON the device with exact integer arithmetic (identical on CPU
    # and GPU): a multiplicative hash of the dof index, two xorshift-multiply rounds, mapped to [-0.5, 0.5)
    cache = V.__dict__.setdefault("_eig_rhs", {})
    key = (n, seed, str(device))
    if key not in cache:  # generated once per level (it does not depend on the operator), copied afterwards
        h = torch.arange(n, dtype=torch.int64, device=device)
        h = (h * 2654435761 + 1234567 * (seed + 1)) & 0xFFFFFFFF
        h = ((h ^ (h >> 15)) * 2246822519) & 0xFFFFFFFF
        h = ((h ^ (h >> 13)) * 3266489917) & 0xFFFFFFFF
        h = h ^ (h >> 16)
        b0 = h.to(torch.float64) / 4294967296.0 - 0.5
        del h
        fix = getattr(V, "consistent", {}).get(n)
        if fix is not None:  # shared-dof / masked layouts: consistent interface copies, zero Dirichlet entries
            fix(b0)
        cache[key] = b0
    b = cache[key].clone()
    r, z, p, Ap = b, torch.empty_like(b), torch.empty_like(b), torch.empty_like(b)   # r starts as (and overwrites) b
    V.pmult(z, dinv, r)
    V.copy(p, z)
    alphas, betas = [], []
    if b.is_cuda:
        # all scalars stay on the device (rz_0..rz_its, pAp_0..pAp_its-1); ONE host sync at the end
        sc = torch.zeros(2 * its + 1, dtype=torch.float64, device=device)
        multi = V.dist is not None and V.dist.get_world_size() > 1

        def ddot(a_, b_, slot):
            out = sc[slot:slot + 1]
            a_ = V._weighted(a_)
            b2(lib.b200_vec_dot(a_.data_ptr(), b_.data_ptr(), a_.numel(), out.data_ptr()))
            if multi:
                V.dist.all_reduce(out)

        ddot(r, z, 0)
        for k in range(its):
            A(p, Ap)
            ddot(p, Ap, its + 1 + k)
            b2(lib.b200_pcg_update(None, r.data_ptr(), z.data_ptr(), p.data_ptr(), Ap.data_ptr(), dinv.data_ptr(),
                                   r.numel(), sc[k:k + 1].data_ptr(), sc[its + 1 + k:its + 2 + k].data_ptr()))
            ddot(r, z, k + 1)
            b2(lib.b200_vec_aypx_dev(p.data_ptr(), z.data_ptr(), p.numel(), sc[k + 1:k + 2].data_ptr(), sc[k:k + 1].data_ptr()))
        h = sc.cpu().numpy()
        for k in range(its):
            rz, pAp, rz_new = h[k], h[its + 1 + k], h[k + 1]
            if not (np.isfinite(rz) and np.isfinite(pAp) and np.isfinite(rz_new)) or pAp <= 0 or rz == 0:
                break
            alphas.append(rz / pAp)
            betas.append(rz_new / rz)
            if rz_new == 0:
                break
    else:
        rz = V.dot(r, z)
        for _ in range(its):
            A(p, Ap)
            pAp = V.dot(p, Ap)
            if pAp <= 0 or rz == 0:
                break
            alpha = rz / pAp
            V.axpy(r, -alpha, Ap)
            V.pmult(z, dinv, r)
            rz_new = V.dot(r, z)
            beta = rz_new / rz
            alphas.append(alpha)
            betas.append(beta)
            V.aypx(p, beta, z)
            rz = rz_new
            if rz_new == 0:
                break
    k = len(alphas)
    T = np.zeros((k, k))
    for i in range(k):
        T[i, i] = 1.0 / alphas[i] + (betas[i - 1] / alphas[i - 1] if i > 0 else 0.0)
        if i + 1 < k:
            T[i, i + 1] = T[i + 1, i] = math.sqrt(betas[i]) / alphas[i]
    return float(np.linalg.eigvalsh(T).max())


class ChebyshevJacobi:
    """KSPCHEBYSHEV + PCJACOBI smoother with eigenvalue interval [0.1, 1.1] * lambda_max (elasticity.c:539-552)."""

    def __init__(self, V, A, n, device, its=3, seed=0):
        self.V, self.A, self.its, self.n, self.device, self.seed = V, A, its, n, device, seed
        self.dinv = None
        self.emax = self.emin = None
        self.r, self.z, self.d, self.Ad = (torch.zeros(n, dtype=torch.float64, device=device) for _ in range(4))

    def setup(self, diag):
        """PCJacobi set-up (MatGetDiagonal -> GetDiag_Ceed) + eigen-estimate; once per Newton step."""
        self.dinv = 1.0 / diag
        lmax = estimate_lambda_max(self.V, self.A, self.dinv, self.n, self.device, seed=self.seed)
        self.emin, self.emax = 0.1 * lmax, 1.1 * lmax

    def apply(self, b, x, zero_guess):
        V, A = self.V, self.A
        theta, delta = 0.5 * (self.emax + self.emin), 0.5 * (self.emax - self.emin)
        sigma = theta / delta
        rho = 1.0 / sigma
        r, z, d, Ad = self.r, self.z, self.d, self.Ad
        if zero_guess:
            V.copy(r, b)
        else:
            A(x, Ad)
            V.axpby(r, 1.0, b, -1.0, Ad)
        # x_{k+1} = x_k + d_k;  r_{k+1} = r_k - A d_k;  d_{k+1} = rho' rho d_k + (2 rho'/delta) D^-1 r_{k+1}
        if x.is_cuda:
            b2(lib.b200_cheb_init(x.data_ptr(), r.data_ptr(), d.data_ptr(), self.dinv.data_ptr(), 1.0 / theta,
                                  1 if zero_guess else 0, x.numel()))
        else:
            torch.mul(self.dinv, r, out=d)
            d.mul_(1.0 / theta)
            if zero_guess:
                x.copy_(d)
            else:
                x.add_(d)
        for _ in range(self.its - 1):
            A(d, Ad)
            rho_new = 1.0 / (2.0 * sigma - rho)
            c1, c2 = rho_new * rho, 2.0 * rho_new / delta
            if x.is_cuda:
                b2(lib.b200_cheb_step(x.data_ptr(), r.data_ptr(), d.data_ptr(), Ad.data_ptr(), self.dinv.data_ptr(), c1, c2,
                                      x.numel()))
            else:
                r.sub_(Ad)
                torch.mul(self.dinv, r, out=z)
                d.mul_(c1).add_(z, alpha=c2)
                x.add_(d)
            rho = rho_new


# --------------------------------------------------------------------------- coarse level by colouring


def _index_add(dst, idx, src, deterministic):
    """dst[idx[i]] += src[i].  torch's CUDA index_add_ uses FP64 atomics; in deterministic mode the sort-based
    accumulation of torch is used instead (same order every run)."""
    if not (deterministic and dst.is_cuda):
        dst.index_add_(0, idx, src)
        return
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        dst.index_put_((idx.long(),), src, accumulate=True)
    finally:
        torch.use_deterministic_algorithms(prev)


class ColoredCoarseMatrix:
    """FormJacobian (src/misc.c:151-183): the coarse (p = 1) Jacobian, assembled on the LOCAL vector space of the
    rank and stored as a 27-point block stencil on the node lattice (81 values per row dof); the global action is
    P^T A_loc P with the same halo exchange as the matrix-free operator.  Two ways to fill it:

    * colouring, as the reference does: the action on 27 node colours x 3 components = 81 coloured unit vectors --
      exact because the action is linear;
    * `coo`: element matrices from CeedOperatorLinearAssemble (one pass over the Jacobian cache), summed into the
      stencil (MatSetValuesCOO stand-in) -- the same entries up to summation order."""

    def __init__(self, dm, local_apply, coo=None):
        """coo (optional): object with .elem_nodes (nelem x 8 local node ids, torch, on dm.device) and
        .values() -> nelem*576 element-matrix entries in CeedOperatorLinearAssemble layout."""
        self.dm, self.local_apply, self.coo = dm, local_apply, coo
        self.deterministic = bool(getattr(coo, "deterministic", False))
        self.coo_dest = None
        self.N = N = dm.mesh.nodes_per_dim(1)
        n, dev = dm.lsize, dm.device
        k, j, i = np.meshgrid(np.arange(N[2]), np.arange(N[1]), np.arange(N[0]), indexing="ij")
        self.ijk = [a.reshape(-1) for a in (i, j, k)]
        self.svals = torch.zeros((81, n), dtype=torch.float64, device=dev)  # [(o*3 + a)][row], o = (dx+1)+3(dy+1)+9(dz+1)
        self.Xloc = torch.zeros(n, dtype=torch.float64, device=dev)
        self.Yloc = torch.zeros(n, dtype=torch.float64, device=dev)
        self._colouring = None   # built on the first coloured assembly
        self._nbr = None         # CPU mat-vec: neighbour dof table, built on first use

    # ---- colouring (src/misc.c:151-183)
    def _setup_colouring(self):
        N, n, dev = self.N, self.dm.lsize, self.dm.device
        nn = N[0] * N[1] * N[2]
        i, j, k = self.ijk
        mask = np.zeros((81, n), dtype=bool)     # slot (colour, a) of a row exists: that colour's neighbour is inside
        seeds = []
        for color in range(27):
            cc = (color % 3, (color // 3) % 3, color // 9)
            ok = np.ones(nn, bool)
            for d in range(3):
                off = ((cc[d] - self.ijk[d] % 3 + 1) % 3) - 1  # in {-1,0,1}: neighbour of that colour along d
                t = self.ijk[d] + off
                ok &= (t >= 0) & (t < N[d])
            seed_nodes = np.flatnonzero((i % 3 == cc[0]) & (j % 3 == cc[1]) & (k % 3 == cc[2]))
            for a in range(3):
                mask[color * 3 + a] = np.repeat(ok, 3)
                seeds.append(torch.from_numpy((seed_nodes * 3 + a).astype(np.int64)).to(dev))
        # svals[(o*3 + a)][row] = vals[colour(node + d_o)*3 + a][row]; neighbours outside the lattice point at
        # slots that the mask has zeroed
        src = np.zeros((81, n), dtype=np.int64)
        for dz in (-1, 0, 1):
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    o = (dx + 1) + 3 * (dy + 1) + 9 * (dz + 1)
                    color = ((i + dx) % 3) + 3 * ((j + dy) % 3) + 9 * ((k + dz) % 3)
                    for a in range(3):
                        src[o * 3 + a] = np.repeat(color * 3 + a, 3)
        self._colouring = dict(seeds=seeds, mask=torch.from_numpy(mask).to(dev).to(torch.float64),
                               src=torch.from_numpy(src).to(dev),
                               vals=torch.zeros((81, n), dtype=torch.float64, device=dev),
                               x=torch.zeros(n, dtype=torch.float64, device=dev),
                               y=torch.zeros(n, dtype=torch.float64, device=dev))

    def assemble(self):
        """coo: one pass over the Jacobian cache.  Otherwise 81 local operator applies (ApplyJacobianCoarse_Ceed
        without the halo: A_loc itself), colour slots re-indexed by neighbour offset."""
        if self.coo is not None:
            return self._assemble_coo()
        if self._colouring is None:
            self._setup_colouring()
        c = self._colouring
        for s in range(81):
            c["x"].zero_()
            c["x"][c["seeds"][s]] = 1.0
            self.local_apply(c["x"], c["y"])
            c["vals"][s].copy_(c["y"])
        c["vals"].mul_(c["mask"])
        torch.gather(c["vals"], 0, c["src"], out=self.svals)

    def _assemble_coo(self):
        """MatSetValuesCOO stand-in: element-matrix entries summed into the 27-point block stencil."""
        if self.coo_dest is None:
            N, n = self.N, self.dm.lsize
            nodes = self.coo.elem_nodes.long()                                   # (E, 8)
            ijk = (nodes % N[0], (nodes // N[0]) % N[1], nodes // (N[0] * N[1]))
            o = 0
            for d, mul in enumerate((1, 3, 9)):
                o = o + (ijk[d][:, :, None] - ijk[d][:, None, :] + 1) * mul      # (E, col node, row node)
            cb = torch.arange(3, device=nodes.device)
            dest = (o[:, :, None, :, None] * 3 + cb[None, None, :, None, None]) * n \
                + nodes[:, None, None, :, None] * 3 + cb[None, None, None, None, :]
            self.coo_dest = dest.reshape(-1).to(torch.int32 if 81 * n < 2 ** 31 else torch.int64)
        self.svals.zero_()
        _index_add(self.svals.view(-1), self.coo_dest, self.coo.values(), self.deterministic)

    def local_mult(self, xloc, yloc):
        """y_loc = A_loc x_loc (the rank-local, un-assembled matrix)"""
        if xloc.is_cuda:
            b2(lib.b200_stencil27_spmv(self.N[0], self.N[1], self.N[2], self.svals.data_ptr(), xloc.data_ptr(),
                                       yloc.data_ptr()))
            return
        if self._nbr is None:  # [(o*3 + a)][row] -> column dof, or -1 outside the lattice
            N, (i, j, k) = self.N, self.ijk
            nbr = np.full((81, self.dm.lsize), -1, dtype=np.int64)
            for o in range(27):
                dx, dy, dz = o % 3 - 1, (o // 3) % 3 - 1, o // 9 - 1
                ok = (i + dx >= 0) & (i + dx < N[0]) & (j + dy >= 0) & (j + dy < N[1]) & (k + dz >= 0) & (k + dz < N[2])
                col = (i + dx) + N[0] * ((j + dy) + N[1] * (k + dz))
                for a in range(3):
                    nbr[o * 3 + a] = np.repeat(np.where(ok, col * 3 + a, -1), 3)
            self._nbr = torch.from_numpy(nbr)
        yloc.copy_((self.svals * xloc[self._nbr.clamp_min(0)] * (self._nbr >= 0)).sum(0))

    def mult(self, X, Y):
        dm = self.dm
        if dm.masked:  # X is the L-vector with zero Dirichlet entries already
            self.local_mult(X, Y)
            dm.local_to_global(Y, Y)
            return
        dm.zero_and_global_to_local(X, self.Xloc)
        self.local_mult(self.Xloc, self.Yloc)
        dm.local_to_global(self.Yloc, Y)

    def diagonal(self, D):
        """global diagonal: centre-block diagonal of the local stencil, summed over ranks"""
        n = self.dm.lsize
        rows = torch.arange(n, device=self.dm.device)
        slot = 13 * 3 + (rows % 3)                       # centre neighbour (dx=dy=dz=0), same component
        self.Yloc.copy_(self.svals[slot, rows])
        self.dm.local_to_global(self.Yloc, D)
        self.dm.fix_diagonal(D)


class SparseCoarseMatrix:
    """The assembled p = 1 Jacobian on an UNSTRUCTURED mesh (-mesh file.exo): no node lattice, so the matrix is kept
    in ELL form (slot-major, b200_ell_spmv).  Filled from the CeedOperatorLinearAssemble element matrices (device),
    or -- CPU tensors, small oracle-driven tests only -- by probing the local operator with unit vectors."""

    def __init__(self, dm, local_apply, coo=None):
        self.dm, self.local_apply, self.coo = dm, local_apply, coo
        self.deterministic = bool(getattr(coo, "deterministic", False))
        n, dev = dm.lsize, dm.device
        self.Xloc = torch.zeros(n, dtype=torch.float64, device=dev)
        self.Yloc = torch.zeros(n, dtype=torch.float64, device=dev)
        self.dense = None
        if coo is not None:
            nodes = coo.elem_nodes.long()                                        # (E, 8)
            dof = (nodes[:, :, None] * 3 + torch.arange(3, device=nodes.device)[None, None, :]).reshape(-1, 24)
            rows = dof[:, None, :].expand(-1, 24, -1).reshape(-1)                # values layout [e][col][row]
            cols = dof[:, :, None].expand(-1, -1, 24).reshape(-1)
            uniq, inv = torch.unique(rows * n + cols, return_inverse=True)       # sorted by row, then column
            r, c = uniq // n, uniq % n
            start = torch.searchsorted(r, torch.arange(n, device=r.device))
            slot = torch.arange(uniq.numel(), device=r.device) - start[r]
            self.nslots = int(slot.max().item()) + 1
            ell = slot * n + r
            self.cols = torch.full((self.nslots * n,), -1, dtype=torch.int32, device=dev)
            self.cols[ell] = c.to(torch.int32)
            self.vals = torch.zeros(self.nslots * n, dtype=torch.float64, device=dev)
            self.dest = ell[inv]
            self.diag_pos = ell[r == c]                                          # one per row, in row order

    def assemble(self):
        if self.coo is not None:
            self.vals.zero_()
            _index_add(self.vals, self.dest, self.coo.values(), getattr(self, "deterministic", False))
            return
        n, dev = self.dm.lsize, self.dm.device
        if n > 20000:
            raise RuntimeError("SparseCoarseMatrix: probing the operator column by column is for small test meshes; "
                               "use the CeedOperatorLinearAssemble path (assemble='coo')")
        A = torch.zeros((n, n), dtype=torch.float64, device=dev)
        e = torch.zeros(n, dtype=torch.float64, device=dev)
        y = torch.zeros(n, dtype=torch.float64, device=dev)
        for j in range(n):
            e.zero_()
            e[j] = 1.0
            self.local_apply(e, y)
            A[:, j] = y
        self.dense = A

    def local_mult(self, xloc, yloc):
        if self.dense is not None:
            torch.mv(self.dense, xloc, out=yloc)
        elif not xloc.is_cuda:
            n = self.dm.lsize
            c = self.cols.view(self.nslots, n).long()
            yloc.copy_((self.vals.view(self.nslots, n) * xloc[c.clamp_min(0)] * (c >= 0)).sum(0))
        else:
            b2(lib.b200_ell_spmv(self.dm.lsize, self.nslots, self.cols.data_ptr(), self.vals.data_ptr(), xloc.data_ptr(),
                                 yloc.data_ptr()))

    def mult(self, X, Y):
        dm = self.dm
        if dm.masked:
            self.local_mult(X, Y)
            dm.local_to_global(Y, Y)
            return
        dm.zero_and_global_to_local(X, self.Xloc)
        self.local_mult(self.Xloc, self.Yloc)
        dm.local_to_global(self.Yloc, Y)

    def diagonal(self, D):
        if self.dense is not None:
            self.Yloc.copy_(torch.diagonal(self.dense))
        else:
            self.Yloc.copy_(self.vals[self.diag_pos])
        self.dm.local_to_global(self.Yloc, D)
        self.dm.fix_diagonal(D)


class HMultigrid:
    """Geometric h-multigrid on the assembled p = 1 level: the stand-in for GAMG (elasticity.c:569-585).

    Level 0 is the assembled p = 1 matrix; every further level halves the element count per
    axis.  Coarse matrices are Galerkin products A_H = P^T A_h P with trilinear P in index space (on the
    device: one stencil triple-product kernel per level; on CPU tensors: the colouring procedure applied to
    the rank-local P^T A_h P -- the same entries); one V(2,2) cycle with
    Chebyshev/Jacobi smoothing is a fixed linear operator, so the outer CG theory holds, and its cost does
    not grow with the mesh the way Jacobi-PCG iterations do.  Brick partitions stay aligned because every
    brick is coarsened in place; the coarsest level is solved by Jacobi-PCG."""

    def __init__(self, V, fine_matrix, dms, smooth_its=2, coarsest_rtol=1e-2):
        """fine_matrix: ColoredCoarseMatrix of the p = 1 level; dms: LevelDMs of the h-levels, dms[0] = its dm."""
        self.V, self.dms, self.smooth_its, self.coarsest_rtol = V, dms, smooth_its, coarsest_rtol
        self.mats = [fine_matrix]
        for l in range(1, len(dms)):
            self.mats.append(ColoredCoarseMatrix(dms[l], self._galerkin_apply(l)))
        mk = lambda l: torch.zeros(dms[l].nglobal, dtype=torch.float64, device=dms[l].device)
        mkl = lambda l: torch.zeros(dms[l].lsize, dtype=torch.float64, device=dms[l].device)
        L = len(dms)
        self.b, self.x, self.r, self.t, self.diag = ([mk(l) for l in range(L)] for _ in range(5))
        self.lf, self.lf2, self.lc = [mkl(l) for l in range(L)], [mkl(l) for l in range(L)], [mkl(l) for l in range(L)]
        self.smoothers = [ChebyshevJacobi(V, self.mats[l].mult, dms[l].nglobal, dms[l].device, smooth_its, seed=100 + l)
                          for l in range(L - 1)]
        self.cwork = [mk(L - 1) for _ in range(4)]
        self.cdinv = mk(L - 1)
        self.coarsest_its = 0

    # ---- rank-local trilinear transfer between lattice l-1 (fine) and l (coarse)
    def _P(self, l, xc_loc, xf_loc):
        N = self.dms[l].mesh.nodes_per_dim(1)
        if xc_loc.is_cuda:
            b2(lib.b200_lattice_prolong(N[0], N[1], N[2], xc_loc.data_ptr(), xf_loc.data_ptr()))
        else:
            xf_loc.copy_(_lattice_prolong_cpu(N, xc_loc))

    def _PT(self, l, xf_loc, xc_loc):
        N = self.dms[l].mesh.nodes_per_dim(1)
        if xf_loc.is_cuda:
            b2(lib.b200_lattice_restrict(N[0], N[1], N[2], xf_loc.data_ptr(), xc_loc.data_ptr()))
        else:
            xc_loc.copy_(_lattice_restrict_cpu(N, xf_loc))

    def _galerkin_apply(self, l):
        def apply(xc_loc, yc_loc):  # y = P^T A_{l-1,loc} P x on local lattices, no communication
            self._P(l, xc_loc, self.lf[l - 1])
            self.mats[l - 1].local_mult(self.lf[l - 1], self.lf2[l - 1])
            self._PT(l, self.lf2[l - 1], yc_loc)
        return apply

    def setup(self):
        """after the p = 1 matrix has been assembled: Galerkin levels, diagonals, eigen-estimates"""
        for l in range(1, len(self.dms)):
            m = self.mats[l]
            if m.svals.is_cuda:  # direct stencil triple product: same entries as colouring P^T A P, one kernel
                b2(lib.b200_stencil27_galerkin(m.N[0], m.N[1], m.N[2], self.mats[l - 1].svals.data_ptr(), m.svals.data_ptr()))
            else:
                m.assemble()
        for l, m in enumerate(self.mats):
            m.diagonal(self.diag[l])
            if l < len(self.mats) - 1:
                self.smoothers[l].setup(self.diag[l])
        self.cdinv.copy_(1.0 / self.diag[-1])

    def _restrict(self, l, Xf, Xc):  # level l-1 -> l
        dmf, dmc = self.dms[l - 1], self.dms[l]
        src = Xf
        if dmf.dot_weight is not None:  # shared-dof vectors: count every fine dof once across ranks
            src = self.t[l - 1]
            self.V.pmult(src, Xf, dmf.dot_weight)
        dmf.zero_and_global_to_local(src, self.lf[l - 1])
        self._PT(l, self.lf[l - 1], self.lc[l])
        dmc.local_to_global(self.lc[l], Xc)

    def _prolong(self, l, Xc, Xf):  # level l -> l-1 (every copy of a shared dof gets the same value: no exchange)
        dmf, dmc = self.dms[l - 1], self.dms[l]
        dmc.zero_and_global_to_local(Xc, self.lc[l])
        self._P(l, self.lc[l], self.lf[l - 1])
        if Xf.is_cuda:
            b2(lib.b200_gather(Xf.data_ptr(), self.lf[l - 1].data_ptr(), dmf.free_owned_idx.data_ptr(), dmf.nglobal))
        else:
            Xf.copy_(self.lf[l - 1][dmf.free_owned_idx.long()])

    def _cycle(self, l):
        V = self.V
        if l == len(self.dms) - 1:
            self.coarsest_its += jacobi_pcg_nosync(V, self.mats[l].mult, self.cdinv, self.b[l], self.x[l], self.cwork,
                                                   self.coarsest_rtol, 200)
            return
        sm = self.smoothers[l]
        sm.apply(self.b[l], self.x[l], zero_guess=True)
        self.mats[l].mult(self.x[l], self.t[l])
        V.axpby(self.r[l], 1.0, self.b[l], -1.0, self.t[l])
        self._restrict(l + 1, self.r[l], self.b[l + 1])
        self._cycle(l + 1)
        self._prolong(l + 1, self.x[l + 1], self.t[l])
        V.axpy(self.x[l], 1.0, self.t[l])
        sm.apply(self.b[l], self.x[l], zero_guess=False)

    def solve(self, b, x):
        self.b[0].copy_(b)
        self._cycle(0)
        x.copy_(self.x[0])


def _lattice_prolong_cpu(Nc, xc):
    """xf = P xc on CPU tensors (oracle runs): trilinear, fine lattice 2Nc-1 per axis, 3 dofs per node"""
    c = xc.reshape(Nc[2], Nc[1], Nc[0], 3)
    for ax in range(3):
        n = c.shape[ax]
        shp = list(c.shape)
        shp[ax] = 2 * n - 1
        f = torch.zeros(shp, dtype=c.dtype)
        idx_e = [slice(None)] * 4
        idx_o = [slice(None)] * 4
        lo, hi = [slice(None)] * 4, [slice(None)] * 4
        idx_e[ax] = slice(0, None, 2)
        idx_o[ax] = slice(1, None, 2)
        lo[ax], hi[ax] = slice(0, n - 1), slice(1, n)
        f[tuple(idx_e)] = c
        f[tuple(idx_o)] = 0.5 * (c[tuple(lo)] + c[tuple(hi)])
        c = f
    return c.reshape(-1)


def _lattice_restrict_cpu(Nc, xf):
    """xc = P^T xf on CPU tensors"""
    f = xf.reshape(2 * Nc[2] - 1, 2 * Nc[1] - 1, 2 * Nc[0] - 1, 3)
    for ax in range(3):
        n = (f.shape[ax] + 1) // 2
        idx_e, idx_o = [slice(None)] * 4, [slice(None)] * 4
        idx_e[ax], idx_o[ax] = slice(0, None, 2), slice(1, None, 2)
        c = f[tuple(idx_e)].clone()
        odd = f[tuple(idx_o)]
        lo, hi = [slice(None)] * 4, [slice(None)] * 4
        lo[ax], hi[ax] = slice(0, n - 1), slice(1, n)
        c[tuple(lo)] += 0.5 * odd
        c[tuple(hi)] += 0.5 * odd
        f = c
    return f.reshape(-1)


# --------------------------------------------------------------------------- PCMG + Newton


class PMultigrid:
    """PCMG, multiplicative V-cycle, levels[0] = coarsest (p = 1) ... levels[-1] = finest."""

    def __init__(self, V, levels, transfers, coarse_rtol=1e-2, coarse_maxit=500, smooth_its=3, h_dms=None, amg=None):
        """levels: list of objects with .n, .device, .jacobian(X, Y), .diagonal(D), .local_apply(xloc, yloc), .dm
        transfers[l] (l >= 1): object with .prolong(Xc, Yf), .restrict(Xf, Yc) between l-1 and l.
        amg: an amg.SmoothedAggregationAMG of the p = 1 level -> one AMG V-cycle is the coarse solve (coarse_its
        then counts V-cycles)."""
        self.V, self.levels, self.transfers = V, levels, transfers
        self.coarse_rtol, self.coarse_maxit = coarse_rtol, coarse_maxit
        L = len(levels)
        self.smoothers = [None] + [ChebyshevJacobi(V, levels[l].jacobian, levels[l].n, levels[l].device, smooth_its, seed=l)
                                   for l in range(1, L)]
        mk = lambda l: torch.zeros(levels[l].n, dtype=torch.float64, device=levels[l].device)
        self.b = [mk(l) for l in range(L)]
        self.x = [mk(l) for l in range(L)]
        self.r = [mk(l) for l in range(L)]
        self.t = [mk(l) for l in range(L)]
        self.diag = [mk(l) for l in range(L)]
        CoarseMatrix = ColoredCoarseMatrix if getattr(levels[0].dm.mesh, "structured", True) else SparseCoarseMatrix
        coo = getattr(levels[0], "coo", None)
        # the AMG assembles the p = 1 matrix itself (BSR) from the element matrices: no second matrix object then
        self.coarse = None if (amg is not None and coo is not None) else CoarseMatrix(levels[0].dm, levels[0].local_apply,
                                                                                      coo=coo)
        # h_dms: LevelDMs of successively halved meshes below the p = 1 level -> geometric multigrid coarse
        # solve (GAMG stand-in); None -> Jacobi-PCG on the assembled p = 1 matrix
        self.hmg = HMultigrid(V, self.coarse, [levels[0].dm] + list(h_dms)) if h_dms else None
        self.amg = amg
        self.cwork = [mk(0) for _ in range(4)]
        self.cdinv = mk(0)
        self.coarse_its = 0
        self.coarse_solves = 0

    def setup(self):
        """Once per Newton step (SNESComputeJacobian -> FormJacobian + PCSetUp): diagonals, eigen-estimates,
        coarse assembly."""
        for l, lev in enumerate(self.levels):
            lev.diagonal(self.diag[l])
            if l > 0:
                self.smoothers[l].setup(self.diag[l])
        if self.amg is not None:   # assembles the p = 1 matrix itself, in its own (BSR) layout
            self.amg.setup(self.coarse if self.coarse is not None else self.levels[0])
        else:
            self.coarse.assemble()
        self.cdinv.copy_(1.0 / self.diag[0])
        if self.hmg is not None:
            self.hmg.setup()

    def _coarse_solve(self, b, x):
        if self.amg is not None:
            self.amg.solve(b, x)
            self.coarse_solves += 1
            self.coarse_its += 1
            return
        if self.hmg is not None:
            self.hmg.solve(b, x)
            self.coarse_solves += 1
            self.coarse_its = self.hmg.coarsest_its
            return
        its = jacobi_pcg_nosync(self.V, self.coarse.mult, self.cdinv, b, x, self.cwork, self.coarse_rtol,
                                self.coarse_maxit)
        self.coarse_its += its
        self.coarse_solves += 1

    def _cycle(self, l):
        V = self.V
        if l == 0:
            self._coarse_solve(self.b[0], self.x[0])
            return
        sm, lev, tr = self.smoothers[l], self.levels[l], self.transfers[l]
        sm.apply(self.b[l], self.x[l], zero_guess=True)                 # pre-smooth
        lev.jacobian(self.x[l], self.t[l])
        V.axpby(self.r[l], 1.0, self.b[l], -1.0, self.t[l])             # residual
        tr.restrict(self.r[l], self.b[l - 1])
        self._cycle(l - 1)
        tr.prolong(self.x[l - 1], self.t[l])
        V.axpy(self.x[l], 1.0, self.t[l])                               # coarse-grid correction
        sm.apply(self.b[l], self.x[l], zero_guess=False)                # post-smooth

    def apply(self, r, z):
        L = len(self.levels) - 1
        self.b[L].copy_(r)
        self._cycle(L)
        z.copy_(self.x[L])


def newton_solve(V, fine, pc, U, num_increments=10, snes_rtol=1e-8, snes_atol=1e-50, snes_maxit=50, ksp_rtol=1e-10,
                 ksp_maxit=200, log=None, check=None):
    """Load-increment loop + Newton (elasticity.c:637-673).  check (optional): called after every linear solve, at a
    point where the host has just synchronised -- the harness uses it to fail loudly on a timed-out halo exchange.  fine.residual(U, F, load) evaluates
    FormResidual_Ceed at load fraction `load` (and refreshes gradu); the Jacobian operators then
    linearise about that state.  Returns a summary dict (iteration counts as in elasticity.c:684-749)."""
    n, dev = fine.n, fine.device
    F, dU = (torch.zeros(n, dtype=torch.float64, device=dev) for _ in range(2))
    work = [torch.zeros(n, dtype=torch.float64, device=dev) for _ in range(4)]
    total_snes = total_ksp = 0
    per_step = []
    t0 = time.perf_counter()
    fine.residual(U, F, 0.0)  # state (gradu) at the initial iterate, zero boundary load
    for inc in range(1, num_increments + 1):
        load, load_prev = inc / num_increments, (inc - 1) / num_increments
        # Predictor: the boundary increment is first pushed through the tangent at the last converged
        # state, J(U_prev) dU = J(U_prev) [0; du_bc], so the first nonlinear residual is not evaluated
        # on a state where only the Dirichlet nodes have moved (which inverts the boundary layer of
        # elements once du_bc is comparable to the node spacing).  Not in the reference; counted in
        # the KSP totals.
        pc.setup()
        fine.bc_increment_rhs(F, load_prev, load)
        fnorm0 = math.sqrt(V.dot(F, F))  # scale of the increment: reference for the relative tolerance
        dU.zero_()
        k, reason, _ = pcg(V, fine.jacobian, F, dU, M=pc.apply, rtol=ksp_rtol, maxit=ksp_maxit, work=work)
        if check:
            check()
        V.axpy(U, -1.0, dU)
        total_ksp += k
        fine.residual(U, F, load)
        fnorm = math.sqrt(V.dot(F, F))
        if log:
            log(f"  load {load:.2f} predictor: |F| = {fnorm:.3e}  ksp its {k} ({reason})")
        its = 1  # the predictor is a linear solve + update like any Newton iteration
        while its < snes_maxit and fnorm > max(snes_rtol * fnorm0, snes_atol):
            pc.setup()
            dU.zero_()
            k, reason, _ = pcg(V, fine.jacobian, F, dU, M=pc.apply, rtol=ksp_rtol, maxit=ksp_maxit, work=work)
            if check:
                check()
            # backtracking line search on |F| (stand-in for SNES line search "cp", elasticity.c:595-601):
            # full step first, halve while the residual norm does not decrease
            lam, taken = 1.0, 0.0
            for _ in range(6):
                V.axpy(U, -(lam - taken), dU)
                taken = lam
                fine.residual(U, F, load)
                fnew = math.sqrt(V.dot(F, F))
                if math.isfinite(fnew) and fnew < (1.0 - 1e-4 * lam) * fnorm:
                    break
                lam *= 0.5
            fnorm = fnew
            its += 1
            total_ksp += k
            if log:
                log(f"  load {load:.2f} newton {its}: |F| = {fnorm:.3e}  ksp its {k} ({reason})")
            if not math.isfinite(fnorm):
                break
        total_snes += its
        per_step.append((its, fnorm / fnorm0 if fnorm0 else 0.0))
        if not math.isfinite(fnorm) or fnorm > max(snes_rtol * fnorm0, snes_atol):
            break
    if dev.type == "cuda":
        torch.cuda.synchronize()
    converged = len(per_step) == num_increments and all(
        math.isfinite(rel) and rel <= max(snes_rtol, 1e-300) for _, rel in per_step)
    return {"snes_its": total_snes, "ksp_its": total_ksp, "time_s": time.perf_counter() - t0, "converged": converged,
            "per_step": per_step, "coarse_its": pc.coarse_its, "coarse_solves": pc.coarse_solves}
