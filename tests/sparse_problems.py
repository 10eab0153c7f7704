"""User problems with an assembled sparse Jacobian, as the reference's examples write them, for the BK_SPARSE tests:
the Brusselator (examples/brusselator.jl: Fbru!, Jbru_sp) and the Mittelmann problem (examples/mittleman.jl: Fmit!, JFmit),
plus the closed form of the Brusselator's first Hopf point and a host complex twin for codim2.HopfMinAug."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spl

# examples/brusselator.jl:86-87 (n = 500); the parameter tuple (alpha, beta, D1, D2, l), continuation parameter l
BRU_N = 500
BRU_PAR = [2.0, 5.45, 0.008, 0.004, 0.3]
BRU_LENS_L, BRU_LENS_BETA = 4, 1
BRU_LH = 0.5119951013439438      # closed form below, evaluated in NumPy (a dense eigen-solve confirms the crossing)
BRU_OMEGA = 2.139509289533466


def bru_F(x, par):
    """Fbru! (examples/brusselator.jl:26-47), Dirichlet values alpha and beta / alpha"""
    a, b, d1, d2, l = par
    n = len(x) // 2
    h2 = (1.0 / n) ** 2
    c1, c2 = d1 / l**2 / h2, d2 / l**2 / h2
    u, v = x[:n], x[n:]
    lu = -2.0 * u
    lu[:-1] += u[1:]
    lu[1:] += u[:-1]
    lu[0] += a
    lu[-1] += a
    lv = -2.0 * v
    lv[:-1] += v[1:]
    lv[1:] += v[:-1]
    lv[0] += b / a
    lv[-1] += b / a
    uuv = u * u * v
    return np.concatenate([c1 * lu + a - (b + 1) * u + uuv, c2 * lv + b * u - uuv])


def bru_J(x, par):
    """Jbru_sp (examples/brusselator.jl:50-82): spdiagm with offsets 0, +-1, +-n, as a CSC matrix (SparseMatrixCSC)"""
    a, b, d1, d2, l = par
    n = len(x) // 2
    h2 = (1.0 / n) ** 2
    c1, c2 = d1 / l**2 / h2, d2 / l**2 / h2
    u, v = x[:n], x[n:]
    diag = np.concatenate([-2 * c1 - (b + 1) + 2 * u * v, -2 * c2 - u * u])
    off = np.zeros(2 * n - 1)
    off[: n - 1] = c1
    off[n:] = c2
    return sp.diags([diag, off, off, u * u, b - 2 * u * v], [0, 1, -1, n, -n], format="csc")


def bru_steady(par, n=BRU_N):
    """the homogeneous state (alpha, beta / alpha): F = 0 exactly for every l"""
    return np.concatenate([par[0] * np.ones(n), par[1] / par[0] * np.ones(n)])


def bru_hopf(beta=BRU_PAR[1], alpha=BRU_PAR[0], d1=BRU_PAR[2], d2=BRU_PAR[3], n=BRU_N):
    """Hopf point of the homogeneous state in l: mode 1 of the Dirichlet difference Laplacian, mu1 = 4 n^2 sin^2(pi / (2 (n + 1))),
    trace zero at l_H = sqrt((D1 + D2) mu1 / (beta - 1 - alpha^2)), omega^2 = det = (beta - 1 - D1 m)(-alpha^2 - D2 m) + alpha^2 beta,
    m = mu1 / l_H^2"""
    mu1 = 4.0 * n * n * np.sin(np.pi / (2 * (n + 1))) ** 2
    lh = np.sqrt((d1 + d2) * mu1 / (beta - 1 - alpha**2))
    m = mu1 / lh**2
    return lh, np.sqrt((beta - 1 - d1 * m) * (-alpha**2 - d2 * m) + alpha**2 * beta)


def bru_eigvecs(J):
    """right eigenvector of the rightmost complex eigenvalue (positive imaginary part) of J and the matching left one"""
    M = J.toarray()
    vals, vecs = np.linalg.eig(M)
    cand = np.where(vals.imag > 1e-8)[0]
    k = cand[np.argmax(vals[cand].real)]
    valt, vect = np.linalg.eig(M.T)
    kt = int(np.argmin(abs(valt - np.conj(vals[k]))))
    return vals[k], vecs[:, k], vect[:, kt]


# examples/mittleman.jl:58-93: 30 x 30 grid on [-0.5, 0.5]^2, F = Lap u - 10 (u - lambda e^u), continuation in lambda
MIT_N, MIT_L = 30, 0.5


def mit_laplacian(nx=MIT_N, ny=MIT_N, lx=MIT_L, ly=MIT_L):
    """Laplacian2D (examples/mittleman.jl:12-27): corner diagonal -1/h^2"""
    def d2(n, h):
        d = -2.0 * np.ones(n)
        d[0] = d[-1] = -1.0
        return sp.diags([np.ones(n - 1), d, np.ones(n - 1)], [-1, 0, 1]) / h**2
    return (sp.kron(sp.identity(ny), d2(nx, 2 * lx / nx)) + sp.kron(d2(ny, 2 * ly / ny), sp.identity(nx))).tocsc()


class Mittelmann:
    def __init__(self):
        self.lap = mit_laplacian()

    def F(self, u, par):
        return self.lap @ u - 10.0 * (u - par[0] * np.exp(u))

    def J(self, u, par):
        """JFmit: the Laplacian plus the diagonal d phi (examples/mittleman.jl:56-63), the pattern of the Laplacian"""
        return (self.lap + sp.diags(-10.0 * (1.0 - par[0] * np.exp(u)))).tocsc()


class SparseComplexProblem:
    """host cprob of codim2.HopfMinAug over a sparse J(x, par): J(x, p, transpose) -> callable on complex vectors (.M the matrix)"""

    class Jc:
        def __init__(self, M):
            self.M = M

        def __call__(self, z):
            return self.M @ z

    def __init__(self, Jfun, params, lens):
        self.Jfun, self.params, self.lens = Jfun, list(params), lens

    def J(self, x, p, transpose=False):
        q = list(self.params)
        q[self.lens] = p
        M = self.Jfun(np.asarray(x), q).tocsc()
        return self.Jc(M.T.tocsc() if transpose else M)


def sparse_cls(Jc, rhs, a0=0.0, a1=1.0):
    """(a0 I + a1 J) x = rhs by sparse LU, complex a0"""
    M = (a0 * sp.identity(Jc.M.shape[0], dtype=complex) + a1 * Jc.M).tocsc()
    return spl.splu(M).solve(np.asarray(rhs, dtype=complex)), True, 1


def sparse_ls2(J, r1, r2):
    lu = spl.splu(J.tocsc())
    return lu.solve(np.asarray(r1)), lu.solve(np.asarray(r2)), True, (1, 1)
