"""TEST INFRASTRUCTURE — ctypes bindings for the CPU oracle (oracle/_build/libgpirt_oracle.so, the restatement in
gpirt_oracle.cpp) and, when built, for the reference's own sources compiled against stand-in headers
(oracle/_ref/libgpirt_ref.so).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module; nothing under gpirt_b200/ does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(_HERE, "_build", "libgpirt_oracle.so")
REF_SO = os.path.join(_HERE, "_ref", "libgpirt_ref.so")
N_GRID = 1001

# purposes of the addressed RNG (gpo_rng.h)
P_INIT_F_Z, P_INIT_BETA, P_ESS_Z, P_ESS_U, P_FSTAR_Z, P_THETA_U, P_BETA_Z, P_BETA_U = range(8)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_bp = C.POINTER(C.c_uint8)


def build(target="oracle"):
    """Compile the oracle, or with target "ref" the compiled-reference library (needs have_ref_sources())."""
    subprocess.check_call(["make", "-s", "-C", _HERE, target])


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel(order="F") if np.ndim(a) > 1 else np.asarray(a, dtype=np.float64))


def _F(a):
    """column-major float64 copy"""
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


def _p(a):
    return a.ctypes.data_as(_dp) if a is not None else None


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_SO):
            build("oracle")
        L = C.CDLL(ORACLE_SO)
        L.gpo_ll.restype = C.c_double
        L.gpo_ll_bar.restype = C.c_double
        L.gpo_rng_keyed.restype = C.c_void_p
        L.gpo_rng_keyed.argtypes = [C.c_uint64, C.c_int]
        L.gpo_rng_tape.restype = C.c_void_p
        L.gpo_rng_tape.argtypes = [_dp, _bp, C.c_size_t]
        L.gpo_rng_free.argtypes = [C.c_void_p]
        L.gpo_rng_set_sweep.argtypes = [C.c_void_p, C.c_uint32]
        L.gpo_rng_set_stream_map.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint32), C.c_size_t]
        L.gpo_rng_tape_len.restype = C.c_size_t
        L.gpo_rng_tape_len.argtypes = [C.c_void_p]
        L.gpo_rng_tape_pos.restype = C.c_size_t
        L.gpo_rng_tape_pos.argtypes = [C.c_void_p]
        L.gpo_rng_error.argtypes = [C.c_void_p]
        L.gpo_rng_tape_copy.argtypes = [C.c_void_p, _dp, _bp]
        L.gpo_keyed_uniform.restype = C.c_double
        L.gpo_keyed_uniform.argtypes = [C.c_uint64] + [C.c_uint32] * 4
        L.gpo_keyed_normal.restype = C.c_double
        L.gpo_keyed_normal.argtypes = [C.c_uint64] + [C.c_uint32] * 4
        L.gpo_ess.argtypes = [_dp, _dp, _dp, _dp, C.c_int, C.c_uint32, C.c_void_p, _dp, _dp, _dp, _ip]
        L.gpo_draw_f.argtypes = [_dp, _dp, _dp, _dp, C.c_int, C.c_int, C.c_void_p, _dp, _ip]
        L.gpo_draw_fstar.argtypes = [_dp] * 5 + [C.c_int] * 3 + [C.c_void_p, _dp, _dp, _dp]
        L.gpo_draw_theta.argtypes = [_dp] * 4 + [C.c_int] * 4 + [C.c_void_p, _dp, _ip, _dp]
        L.gpo_draw_beta.argtypes = [_dp] * 7 + [C.c_int] * 2 + [C.c_void_p, _dp, _ip]
        L.gpo_mcmc.argtypes = [_dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int, _dp, _dp, _dp, C.c_void_p, C.c_int,
                               _dp, _dp, _dp, _dp, _dp, _dp]
        _lib = L
    return _lib


class Rng:
    """Addressed RNG handle. Rng.keyed(seed) draws Philox variates by address; Rng.tape(vals, kinds) replays."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def keyed(cls, seed, record=False):
        return cls(lib().gpo_rng_keyed(C.c_uint64(seed), int(record)))

    @classmethod
    def tape(cls, vals, kinds):
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        kinds = np.ascontiguousarray(kinds, dtype=np.uint8)
        return cls(lib().gpo_rng_tape(_p(vals), kinds.ctypes.data_as(_bp), vals.size))

    def set_sweep(self, sweep):
        lib().gpo_rng_set_sweep(self.h, sweep)

    def set_item_map(self, items):
        """local item index j of the following calls draws from stream items[j] (global item index); None clears"""
        self._set_map(0, items)

    def set_respondent_map(self, rows):
        """local respondent index i of the following draw_theta calls draws from stream rows[i]; None clears"""
        self._set_map(1, rows)

    def _set_map(self, which, idx):
        a = np.ascontiguousarray([] if idx is None else idx, dtype=np.uint32)
        lib().gpo_rng_set_stream_map(self.h, which, a.ctypes.data_as(C.POINTER(C.c_uint32)), a.size)

    def recorded(self):
        n = lib().gpo_rng_tape_len(self.h)
        vals = np.empty(n, dtype=np.float64)
        kinds = np.empty(n, dtype=np.uint8)
        if n:
            lib().gpo_rng_tape_copy(self.h, _p(vals), kinds.ctypes.data_as(_bp))
        return vals, kinds

    @property
    def error(self):
        return lib().gpo_rng_error(self.h)

    @property
    def pos(self):
        return lib().gpo_rng_tape_pos(self.h)

    def __del__(self):
        try:
            lib().gpo_rng_free(self.h)
        except Exception:
            pass


def keyed_uniform(seed, sweep, purpose, stream, idx):
    return lib().gpo_keyed_uniform(seed, sweep, purpose, stream, idx)


def keyed_normal(seed, sweep, purpose, stream, idx):
    return lib().gpo_keyed_normal(seed, sweep, purpose, stream, idx)


def set_blas_threads(t):
    lib().gpo_set_blas_threads(int(t))


def K(x1, x2):
    x1 = _f64(x1); x2 = _f64(x2)
    out = np.empty((x1.size, x2.size), order="F")
    lib().gpo_K(_p(x1), x1.size, _p(x2), x2.size, _p(out))
    return out


def chol_lower(S):
    S = _F(S).copy(order="F")
    rc = lib().gpo_chol_lower(_p(S), S.shape[0])
    if rc:
        raise np.linalg.LinAlgError("chol(): decomposition failed (info=%d)" % rc)
    return S


def build_cholS(theta):
    theta = _f64(theta)
    L = np.empty((theta.size, theta.size), order="F")
    rc = lib().gpo_build_cholS(_p(theta), theta.size, _p(L))
    if rc:
        raise np.linalg.LinAlgError("chol(): decomposition failed (info=%d)" % rc)
    return L


def ll(f, y):
    f = _f64(f); y = _f64(y)
    return lib().gpo_ll(_p(f), _p(y), f.size)


def ll_bar(f, y, mu):
    f = _f64(f); y = _f64(y); mu = _f64(mu)
    return lib().gpo_ll_bar(_p(f), _p(y), _p(mu), f.size)


def grid():
    ts = np.empty(N_GRID); pr = np.empty(N_GRID)
    n = lib().gpo_grid(_p(ts), _p(pr))
    assert n == N_GRID
    return ts, pr


def linear_mean(x, beta):
    x = _f64(x); beta = _F(beta)
    mu = np.empty((x.size, beta.shape[1]), order="F")
    lib().gpo_linear_mean(_p(x), x.size, _p(beta), beta.shape[1], _p(mu))
    return mu


def ess(f, y, cholS, mu, item, rng, nu=None):
    f = _f64(f); y = _f64(y); mu = _f64(mu); cholS = _F(cholS)
    n = f.size
    out = np.empty(n); nu_out = np.empty(n); nprop = C.c_int(0)
    nu_in = _f64(nu) if nu is not None else None
    rc = lib().gpo_ess(_p(f), _p(y), _p(cholS), _p(mu), n, item, rng.h, _p(nu_in), _p(out), _p(nu_out), C.byref(nprop))
    if rc:
        raise RuntimeError("ess did not terminate")
    return out, nu_out, nprop.value


def draw_f(f, y, cholS, mu, rng):
    f = _F(f); y = _F(y); mu = _F(mu); cholS = _F(cholS)
    n, m = f.shape
    out = np.empty((n, m), order="F"); nprop = np.zeros(m, dtype=np.int32)
    rc = lib().gpo_draw_f(_p(f), _p(y), _p(cholS), _p(mu), n, m, rng.h, _p(out), nprop.ctypes.data_as(_ip))
    if rc:
        raise RuntimeError("ess did not terminate")
    return out, nprop


def draw_fstar(f, theta, theta_star, L, mu_star, rng):
    f = _F(f); theta = _f64(theta); theta_star = _f64(theta_star); L = _F(L); mu_star = _F(mu_star)
    n, m = f.shape; N = theta_star.size
    out = np.empty((N, m), order="F"); s = np.empty(N); mean = np.empty((N, m), order="F")
    rc = lib().gpo_draw_fstar(_p(f), _p(theta), _p(theta_star), _p(L), _p(mu_star), n, m, N, rng.h, _p(out), _p(s), _p(mean))
    if rc:
        raise RuntimeError("dtrtrs failed")
    return out, s, mean


def draw_theta(theta_star, y, theta_prior, fstar, rng, mode=0):
    theta_star = _f64(theta_star); y = _F(y); theta_prior = _f64(theta_prior); fstar = _F(fstar)
    n, m = y.shape; N = theta_star.size
    out = np.empty(n); idx = np.zeros(n, dtype=np.int32); logp = np.empty((n, N), order="F")
    lib().gpo_draw_theta(_p(theta_star), _p(y), _p(theta_prior), _p(fstar), n, m, N, mode, rng.h, _p(out),
                         idx.ctypes.data_as(_ip), _p(logp))
    return out, idx, logp


def draw_beta(beta, theta, y, f, pm, psd, pstep, rng):
    beta = _F(beta); y = _F(y); f = _F(f); pm = _F(pm); psd = _F(psd); pstep = _F(pstep)
    n, m = y.shape
    X = np.asfortranarray(np.column_stack([np.ones(n), _f64(theta)]))
    out = np.empty((2, m), order="F"); acc = np.zeros((2, m), dtype=np.int32, order="F")
    lib().gpo_draw_beta(_p(beta), _p(X), _p(y), _p(f), _p(pm), _p(psd), _p(pstep), n, m, rng.h, _p(out),
                        acc.ctypes.data_as(_ip))
    return out, acc


def mcmc(y, theta_init, sample_iterations, burn_iterations, pm, psd, pstep, rng, theta_cdf_mode=0):
    """gpirtMCMC restatement. Returns dict(theta (S+1,n), beta (2,m,S+1), f (n,m,S+1), IRFs (1001,m), fstar_last, secs)."""
    y = _F(y); theta_init = _f64(theta_init); pm = _F(pm); psd = _F(psd); pstep = _F(pstep)
    n, m = y.shape; S1 = sample_iterations + 1
    th = np.empty((S1, n), order="F"); be = np.empty((2, m, S1), order="F"); f = np.empty((n, m, S1), order="F")
    irf = np.empty((N_GRID, m), order="F"); fl = np.empty((N_GRID, m), order="F"); secs = np.zeros(7)
    rc = lib().gpo_mcmc(_p(y), n, m, _p(theta_init), sample_iterations, burn_iterations, _p(pm), _p(psd), _p(pstep),
                        rng.h, theta_cdf_mode, _p(th), _p(be), _p(f), _p(irf), _p(fl), _p(secs))
    if rc:
        raise RuntimeError("oracle gpirtMCMC failed rc=%d (-1 chol, -2 solve, -3 ess)" % rc)
    return dict(theta=th, beta=be, f=f, IRFs=irf, fstar_last=fl, secs=secs)


# ---------------------------------------------------------------------------------------------------------
# the reference's own sources (compiled against stand-in headers), driven by a replay tape
# ---------------------------------------------------------------------------------------------------------
_ref = None


def have_ref_sources():
    """True where oracle/Makefile finds the reference package's sources (its REF, overridden by GPIRT_REFERENCE)"""
    return subprocess.run(["make", "-s", "-C", _HERE, "have-ref"], capture_output=True).returncode == 0


def have_ref():
    return os.path.exists(REF_SO) or have_ref_sources()


def ref():
    global _ref
    if _ref is None:
        if not os.path.exists(REF_SO):
            build("ref")
        L = C.CDLL(REF_SO)
        L.gpref_ll.restype = C.c_double
        L.gpref_ll_bar.restype = C.c_double
        L.gpref_set_tape.argtypes = [_dp, _bp, C.c_size_t]
        L.gpref_tape_pos.restype = C.c_size_t
        L.gpref_seed.argtypes = [C.c_uint64]
        _ref = L
    return _ref


class RefTape:
    """Context manager: install a (vals, kinds) tape as the compiled reference's R RNG."""

    def __init__(self, vals, kinds):
        self.vals = np.ascontiguousarray(vals, dtype=np.float64)
        self.kinds = np.ascontiguousarray(kinds, dtype=np.uint8)

    def __enter__(self):
        ref().gpref_set_tape(_p(self.vals), self.kinds.ctypes.data_as(_bp), self.vals.size)
        return self

    def __exit__(self, *a):
        self.consumed = ref().gpref_tape_pos()
        self.error = ref().gpref_tape_error()
        ref().gpref_clear_tape()   # back to the self-contained generator (timing runs)
        return False


def ref_K(x1, x2):
    x1 = _f64(x1); x2 = _f64(x2)
    out = np.empty((x1.size, x2.size), order="F")
    ref().gpref_K(_p(x1), x1.size, _p(x2), x2.size, _p(out))
    return out


def ref_ll(f, y):
    f = _f64(f); y = _f64(y)
    return ref().gpref_ll(_p(f), _p(y), f.size)


def ref_ll_bar(f, y, mu):
    f = _f64(f); y = _f64(y); mu = _f64(mu)
    return ref().gpref_ll_bar(_p(f), _p(y), _p(mu), f.size)


def ref_chol_lower(S):
    S = _F(S).copy(order="F")
    if ref().gpref_chol_lower(_p(S), S.shape[0]):
        raise np.linalg.LinAlgError("chol(): decomposition failed")
    return S


def ref_draw_f(f, y, cholS, mu):
    f = _F(f); y = _F(y); mu = _F(mu); cholS = _F(cholS)
    n, m = f.shape
    out = np.empty((n, m), order="F")
    ref().gpref_draw_f(_p(f), _p(y), _p(cholS), _p(mu), n, m, _p(out))
    return out


def ref_draw_fstar(f, theta, theta_star, L, mu_star):
    f = _F(f); theta = _f64(theta); theta_star = _f64(theta_star); L = _F(L); mu_star = _F(mu_star)
    n, m = f.shape; N = theta_star.size
    out = np.empty((N, m), order="F")
    if ref().gpref_draw_fstar(_p(f), _p(theta), _p(theta_star), _p(L), _p(mu_star), n, m, N, _p(out)):
        raise RuntimeError("reference draw_fstar threw")
    return out


def ref_draw_theta(theta_star, y, theta_prior, fstar, mu_star):
    theta_star = _f64(theta_star); y = _F(y); theta_prior = _f64(theta_prior); fstar = _F(fstar); mu_star = _F(mu_star)
    n, m = y.shape; N = theta_star.size
    out = np.empty(n)
    ref().gpref_draw_theta(_p(theta_star), _p(y), _p(theta_prior), _p(fstar), _p(mu_star), n, m, N, _p(out))
    return out


def ref_draw_beta(beta, theta, y, f, pm, psd, pstep):
    beta = _F(beta); y = _F(y); f = _F(f); pm = _F(pm); psd = _F(psd); pstep = _F(pstep)
    n, m = y.shape
    X = np.asfortranarray(np.column_stack([np.ones(n), _f64(theta)]))
    out = np.empty((2, m), order="F")
    ref().gpref_draw_beta(_p(beta), _p(X), _p(y), _p(f), _p(pm), _p(psd), _p(pstep), n, m, _p(out))
    return out


def ref_mcmc(y, theta_init, sample_iterations, burn_iterations, pm, psd, pstep):
    """The reference's gpirtMCMC() itself (src/gpirtMCMC.cpp:5), fed from the installed tape."""
    y = _F(y); theta_init = _f64(theta_init); pm = _F(pm); psd = _F(psd); pstep = _F(pstep)
    n, m = y.shape; S1 = sample_iterations + 1
    th = np.empty((S1, n), order="F"); be = np.empty((2, m, S1), order="F"); f = np.empty((n, m, S1), order="F")
    irf = np.empty((N_GRID, m), order="F"); secs = C.c_double(0)
    rc = ref().gpref_mcmc(_p(y), n, m, _p(theta_init), sample_iterations, burn_iterations, _p(pm), _p(psd), _p(pstep),
                          _p(th), _p(be), _p(f), _p(irf), C.byref(secs))
    if rc:
        raise RuntimeError("reference gpirtMCMC threw (chol(): decomposition failed?)")
    return dict(theta=th, beta=be, f=f, IRFs=irf, secs=secs.value)
