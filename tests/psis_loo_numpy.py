"""The definitions of PSIS-LOO in include/gpirt_b200.h (gpirt_b200_loo) written out in numpy, vectorised over the left-out
units: the reference the device outputs are tested against.  It follows the header, not any version of the loo package."""
import numpy as np

EPS_RANGE = np.finfo(np.float64).eps / 100.0


def tail_len(S):
    return 0 if S <= 0 else int(np.ceil(min(0.2 * S, 3.0 * np.sqrt(S))))


def k_threshold(S):
    if S <= 0:
        return np.nan
    with np.errstate(divide="ignore"):
        return min(1.0 - 1.0 / np.log10(float(S)), 0.7)


def log_sigmoid(a):
    """sigma(a) and log sigma(a) as the device computes them"""
    e = np.exp(-np.abs(a))
    return np.where(a >= 0.0, 1.0, e) / (1.0 + e), -(np.maximum(-a, 0.0) + np.log1p(e))


def _lse(v):
    mx = v.max(axis=1)
    return mx + np.log(np.exp(v - mx[:, None]).sum(axis=1))


def gpdfit(x):
    """x: rows x N, ascending along a row -> (pareto_k adjusted, sigma from the unadjusted k)"""
    N = x.shape[1]
    G = 30 + int(np.floor(np.sqrt(N)))
    xstar = x[:, int(np.floor(N / 4.0 + 0.5)) - 1]
    j = np.arange(1, G + 1, dtype=np.float64)
    theta = 1.0 / x[:, -1:] + (1.0 - np.sqrt(G / (j - 0.5)))[None, :] / (3.0 * xstar[:, None])
    kap = np.mean(np.log1p(-theta[:, :, None] * x[:, None, :]), axis=2)
    lt = N * (np.log(-theta / kap) - kap - 1.0)
    w = np.exp(lt - _lse(lt)[:, None])
    th = np.sum(theta * w, axis=1)
    k = np.mean(np.log1p(-th[:, None] * x), axis=1)
    sigma = -k / th
    khat = k * N / (N + 10.0) + 5.0 / (N + 10.0)
    return np.where(np.isnan(khat), np.inf, khat), sigma


def draw_order_sum(sig):
    """sum along each row in draw order, as the device adds sigma: add.accumulate is sequential (np.sum is pairwise)"""
    return np.cumsum(sig, axis=1)[:, -1]


def psis_loo(ll, sig=None):
    """ll: units x S log-likelihood draws (sig: sigma of each, default exp(ll)) -> dict(elpd, p_loo, k, lpd), per unit"""
    ll = np.atleast_2d(np.asarray(ll, dtype=np.float64))
    cells, S = ll.shape
    if S == 0:
        nan = np.full(cells, np.nan)
        return dict(elpd=nan, p_loo=nan.copy(), k=nan.copy(), lpd=nan.copy())
    sig = np.exp(ll) if sig is None else np.asarray(sig, dtype=np.float64)
    lpd = np.log(draw_order_sum(sig) / S)
    M = tail_len(S)
    rs = np.sort(-ll, axis=1)                   # log ratios, ascending
    mx = rs[:, -1]
    lw = rs - mx[:, None]
    tail = lw[:, S - M:]
    cutoff = lw[:, S - M - 1] if S > M else np.full(cells, -np.inf)
    khat = np.full(cells, np.inf)
    lwt = lw.copy()
    if M >= 5:
        ok = (tail.max(axis=1) - tail.min(axis=1)) >= EPS_RANGE
        if ok.any():
            ec = np.exp(cutoff[ok])
            x = np.exp(tail[ok]) - ec[:, None]
            with np.errstate(all="ignore"):
                kh, sigma = gpdfit(x)
                p = (np.arange(1, M + 1) - 0.5) / M
                sm = np.log(sigma[:, None] * np.expm1(-kh[:, None] * np.log1p(-p)[None, :]) / kh[:, None] + ec[:, None])
            khat[ok] = kh
            fin = np.isfinite(kh)
            rows = np.flatnonzero(ok)[fin]
            lwt[rows, S - M:] = sm[fin]
    lwt = np.where(lwt > 0.0, 0.0, lwt)
    with np.errstate(all="ignore"):
        elpd = _lse(lwt + (-rs)) - _lse(lwt)
    return dict(elpd=elpd, p_loo=lpd - elpd, k=khat, lpd=lpd)


ADVERSARIAL_KINDS = ("logistic", "ties at the cutoff", "all-equal tail", "constant", "Pareto 1.5", "near -700",
                     "x* = 0", "five decades")


def adversarial(S, rs, reps=4):
    """reps x 8 columns of S log-likelihood draws, kind ADVERSARIAL_KINDS[i % 8] in row i, that reach the edges of the
    finish: ties, an all-equal tail, constant columns, k > 1, underflow of exp(ll), x* = 0, a wide spread"""
    cols = []
    M = tail_len(S)
    for rep in range(reps):
        g = rs.standard_normal(S) * (1.0 + rep) + 1.0
        cols.append(log_sigmoid(g)[1])                                     # a logistic cell
        c = log_sigmoid(g)[1]
        if S > M + 1:                                                      # ties at the cutoff, inside and outside the tail
            srt = np.sort(c)
            c[(c >= srt[M - 1]) & (c <= srt[M + 1])] = srt[M]
        cols.append(c)
        c = log_sigmoid(g)[1]
        if S > M:                                                          # an all-equal tail, below a distinct cutoff
            srt = np.sort(c)
            c[c < srt[M]] = srt[0]
        cols.append(c)
        cols.append(np.full(S, -0.25 * (rep + 1)))                         # constant
        u = rs.uniform(size=S)
        cols.append(-np.log((u ** -1.5 - 1.0) / 1.5 + 1.0))                # Pareto ratios, shape 1.5: k > 1
        cols.append(-700.0 - rs.exponential(0.5 + rep, S))                 # ll near -700
        c = -rs.uniform(0.0, 1.0, S)                                       # x* = 0: a quarter of the tail on the cutoff
        if S > M and M >= 4:
            c[:M // 2] = -3.0 - rs.uniform(0.0, 1.0, M // 2)
            c[M // 2:M + 1] = -3.0
        cols.append(c)
        cols.append(np.log(rs.uniform(size=S)) * 10.0 ** rs.uniform(-3, 2))   # spread over five decades
    return np.stack(cols) if S else np.zeros((8 * reps, 0))


def loglik_from_draws(out, y, rs=None):
    """ll (n x m x S) and sigma of every cell and sampling iteration from the stored draws of a thin = 1 run, as the device
    computes them (NaN where y is missing).  rs (a numpy Generator): g is moved by 4 ulps of its terms with random signs,
    the size of the difference between this g and the device's fused g = f + fma(theta, beta1, beta0)"""
    f, th, be = out["f"], out["theta"], out["beta"]
    n, m, S = f.shape[0], f.shape[1], f.shape[2] - 1
    ll = np.full((n, m, S), np.nan)
    sg = np.full((n, m, S), np.nan)
    yo = np.where(np.isnan(y), 1.0, y)
    for s in range(1, S + 1):
        tb = th[s, :][:, None] * be[1, :, s][None, :]
        g = f[:, :, s] + (tb + be[0, :, s][None, :])
        if rs is not None:
            scale = np.abs(f[:, :, s]) + np.abs(tb) + np.abs(be[0, :, s])[None, :]
            g = g + rs.choice([-4.0, 4.0], g.shape) * np.finfo(np.float64).eps * scale
        a = np.where(yo < 0, -g, g)
        sg[:, :, s - 1], ll[:, :, s - 1] = log_sigmoid(a)
    return ll, sg


def aggregate(y, cell):
    """the per-item, per-respondent and total outputs of gpirt_b200_loo from the per-cell reference"""
    S_obs = ~np.isnan(y)
    n, m = y.shape
    e = np.where(S_obs, cell["elpd"].reshape(n, m, order="F"), 0.0)
    p = np.where(S_obs, cell["p_loo"].reshape(n, m, order="F"), 0.0)
    ev = cell["elpd"].reshape(n, m, order="F")[S_obs]
    N = int(S_obs.sum())
    return dict(elpd_loo_item=e.sum(axis=0), elpd_loo_resp=e.sum(axis=1), elpd_loo=ev.sum(), p_loo=p.sum(),
                looic=-2.0 * ev.sum(), se_elpd_loo=np.sqrt(N * np.var(ev, ddof=1)), n_obs=N)
