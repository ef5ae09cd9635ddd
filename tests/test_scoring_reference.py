"""CPU: the restatement of the two scoring stages (oracle/restate/gmm.c, dnn.c), which the GPU scoring tests use as their
checker, held against a float64 numpy statement of the same formulas on shapes that no golden case pins: GMMs at every
feature size the kernels are built for, with irregular mixture counts, NULL densities and empty states; DNNs with widths
that are not multiples of 8 and with a single layer.

Tolerances are bounds derived from the fp32 arithmetic of the restatement, evaluated per element (see the docstrings);
none is a number chosen by trial.  u = 2^-24 is the unit roundoff of fp32 and gamma(n) = n u / (1 - n u) the usual bound
on n accumulated roundings."""
import numpy as np
import pytest

from julius_b200 import desc
from util import LOG_ZERO, dnn_blob, gmm_blob, gmm_frames

U = 2.0 ** -24
INV_LOG_TEN = 0.434294482
LOG_ADDMIN = -13.815510558
# table-driven log-add (addlog.c:39-57, 102-123): log(1 + e^f) tabulated at steps of 15 / 500000 nats, entry chosen by
# rounding; the slope of log(1 + e^f) is at most 1/2 for f <= 0, so one addition is off by at most half a step times
# 1/2, plus the rounding of the table entry (< ln 2 * u) and of the sum (u |y|)
ADDLOG_STEP_ERR = 0.5 * (15.0 / 500000) * 0.5 + np.log(2.0) * U
# a term more than LOG_ADDMIN below the running sum is dropped: it is worth at most e^LOG_ADDMIN = 1e-6 nats
ADDLOG_DROP_ERR = np.exp(LOG_ADDMIN)
# logistic table (calc_dnn.c:342-369): 320001 entries over [-8, 8], step 1/20000, entry chosen by rounding a product of
# two rounded fp32 operations; the chosen entry can be one step away from the exact argument in the worst case, and the
# logistic's slope is at most 1/4: 1/20000 * 1/4 = 1.25e-5, plus the fp32 rounding of the table value
LOGISTIC_ERR = 0.25 / 20000 + U


def gamma(n):
    return n * U / (1 - n * U)


# ---------------------------------------------------------------------------------------------------------------- GMM
def gmm_f64(blob, x):
    """log10 state likelihoods in float64: log10 sum_m w_m N(x; mu_m, var_m) over the valid mixtures (the top -tmix
    Gaussians by Gaussian score under -gprune safe), LOG_ZERO for a state without valid mixtures.  Also returns the
    error bound of the fp32 restatement per element (log10 units):
      Gaussian score  acc = gconst + sum_d (x_d - m_d)^2 iv_d in fp32, sequentially: every term carries 4 roundings
                      (v - m, the square, * iv, and its share of the sum), so |err| <= gamma(D + 4) (|gconst| + sum terms),
                      halved by the * -0.5; + ln w adds u |score|;
      log-sum-exp     is 1-Lipschitz in the max norm of its inputs, so the worst Gaussian error carries over;
                      the M - 1 table additions add ADDLOG_STEP_ERR + u |y| each, dropped terms ADDLOG_DROP_ERR each;
      log10           the conversion in double and the store to float: u |result|."""
    D, S = int(blob["gmm.dim"][0]), int(blob["gmm.n_states"][0])
    off, valid = blob["gmm.state_off"], blob["gmm.valid"].astype(bool)
    mean = blob["gmm.mean"].reshape(-1, D).astype(np.float64)
    iv = blob["gmm.ivar"].reshape(-1, D).astype(np.float64)
    gconst = blob["gmm.gconst"].astype(np.float64)
    lnw = blob["gmm.lnweight"].astype(np.float64)
    method, tmix = int(blob["gmm.gprune_method"][0]), int(blob["gmm.gprune_num"][0])
    xd = x.astype(np.float64)
    terms = (xd[:, None, :] - mean[None]) ** 2 * iv[None]                      # [T, G, D]
    mag = np.abs(gconst)[None] + terms.sum(2)                                    # |gconst| + sum of |terms|
    g = -0.5 * (gconst[None] + terms.sum(2))                                     # Gaussian log score [T, G]
    g_err = 0.5 * gamma(D + 4) * mag + U * np.abs(g)
    T = len(x)
    want = np.full((T, S), LOG_ZERO, np.float64)
    tol = np.zeros((T, S))
    for s in range(S):
        ids = np.arange(off[s], off[s + 1])[valid[off[s]:off[s + 1]]]
        if len(ids) == 0:
            continue
        for t in range(T):
            sel = ids
            if method != 0 and len(ids) > tmix:
                sel = ids[np.argsort(-g[t, ids], kind="stable")[:tmix]]
            a = g[t, sel] + lnw[sel]
            m = a.max()
            lse = m + np.log(np.exp(a - m).sum())
            want[t, s] = lse * INV_LOG_TEN
            n = len(sel)
            tol[t, s] = INV_LOG_TEN * (g_err[t, sel].max() + U * np.abs(a).max()
                                       + (n - 1) * (ADDLOG_STEP_ERR + U * abs(lse) + ADDLOG_DROP_ERR)) + U * abs(want[t, s])
    return want, tol


GMM_SHAPES = [
    # dim, mixture counts per state, states whose slots are all NULL, further NULL slots (global index), gprune
    (25, [1, 3, 6, 2, 0, 5, 4, 1, 17, 2], (3,), (1, 9), (0, 0)),
    (26, [4, 4, 0, 0, 7, 1, 2, 9, 3, 5], (1,), (12,), (0, 0)),
    (38, [16, 16, 16, 16, 1, 3, 63, 2], (), (5, 40), (0, 0)),
    (39, [64, 2, 5, 1, 0, 8, 3], (2,), (70,), (0, 0)),
    (25, [6, 1, 3, 17, 5, 2], (), (7,), (1, 2)),
    (26, [3, 8, 1, 16, 4, 2], (2,), (), (1, 1)),
    (38, [20, 3, 1, 9, 5], (), (25,), (1, 16)),
    (39, [2, 7, 4, 1, 12], (0,), (6,), (1, 4)),
]


@pytest.mark.parametrize("dim,counts,null_states,null_gauss,gprune", GMM_SHAPES)
def test_gmm_restatement_agrees_with_fp64(dim, counts, null_states, null_gauss, gprune, oracle_lib):
    blob = gmm_blob(dim, counts, seed=dim + len(counts), null_states=null_states, null_gauss=null_gauss, gprune=gprune)
    ds = desc.Descriptors(blob)
    x = gmm_frames(blob, 24, seed=dim)
    got = oracle_lib.gmm_score(ds, x)
    want, tol = gmm_f64(blob, x)
    empty = want == LOG_ZERO
    # states without a valid mixture score exactly LOG_ZERO (outprob_state / calc_mix on an empty sum)
    assert np.array_equal(got[empty], want[empty].astype(np.float32))
    err = np.abs(got.astype(np.float64) - want)
    assert (err <= tol).all(), f"max err {err.max():.3e} where the bound is {tol[np.unravel_index(err.argmax(), err.shape)]:.3e}"


# ---------------------------------------------------------------------------------------------------------------- DNN
def logistic_f64(z):
    """the reference's logistic in float64: exact 1/(1+e^-z) inside (-8, 8), the constants of calc_dnn.c:366-367 outside"""
    return np.where(z <= -8.0, 0.000334, np.where(z >= 8.0, 0.999666, 1.0 / (1.0 + np.exp(-np.clip(z, -8, 8)))))


def dnn_f64(blob, x):
    """log10 pseudo-likelihoods in float64 (dnn_calc_outprob: GEMV stack, logistic, log-softmax, / ln 10, - log10 prior)
    and the error bound of the fp32 restatement per element.  Worst-case bounds multiply by ~3 per layer (the row sums
    of |W|) and say nothing at 16 layers, so the errors are treated the way probabilistic rounding error analysis does
    (Higham and Mary, SIAM J. Sci. Comput. 41(5), 2019): every elementary error -- a rounding, a table lookup -- is
    independent, zero-mean and bounded, and a sum of such errors with bounds c_i stays within lambda sqrt(sum c_i^2)
    except with probability 2 exp(-lambda^2 / 2) (Hoeffding).  lambda = 6 here: 3e-8 per element.  The scale
    sqrt(sum c_i^2) is carried per unit, layer by layer:
      GEMV        n + 2 roundings in the accumulation of each product over n inputs (8 FMA lanes + horizontal sum, or a
                  scalar loop): sqrt(n + 2) u (sum_j |w_j h_j| + |b|); the inputs' errors enter weighted by w_j;
      logistic    the largest slope of the reference's logistic on [z - lambda s, z + lambda s] (0 beyond the clamps)
                  times the incoming scale, plus LOGISTIC_ERR for the table (at +-8, where the clamp constants and the
                  table meet, they differ by less than that);
      softmax     log-sum-exp through addlog_array is 1-Lipschitz in the max norm of the logits, adds N - 1 table
                  additions of ADDLOG_STEP_ERR + u |lse|, and drops terms below lse + LOG_ADDMIN, worth at most
                  sum e^(x_i - lse) over those (a one-sided, deterministic error);
      output      (logit - lse) in fp32, * INV_LOG_TEN and - prior in double, stored as float: u |.| each."""
    lam = 6.0
    L = int(blob["dnn.n_layers"][0])
    h = x.astype(np.float64)
    s = np.zeros_like(h)
    for i in range(L):
        n_out, n_in = int(blob[f"dnn.l{i}.out"][0]), int(blob[f"dnn.l{i}.in"][0])
        w = blob[f"dnn.l{i}.w"].reshape(n_out, n_in).astype(np.float64)
        bias = blob[f"dnn.l{i}.b"].astype(np.float64)
        z = h @ w.T + bias
        sz = np.sqrt((s * s) @ (w * w).T + (n_in + 2) * (U * (np.abs(h) @ np.abs(w).T + np.abs(bias))) ** 2)
        if i < L - 1:
            near = np.clip(0.0, z - lam * sz, z + lam * sz)            # the point of the interval closest to 0
            slope = np.where(np.abs(near) >= 8.0, 0.0, logistic_f64(near) * (1.0 - logistic_f64(near)))
            h, s = logistic_f64(z), np.sqrt((slope * sz) ** 2 + LOGISTIC_ERR ** 2)
        else:
            h, s = z, sz
    N = h.shape[1]
    m = h.max(1, keepdims=True)
    lse = m + np.log(np.exp(h - m).sum(1, keepdims=True))
    want = (h - lse) * INV_LOG_TEN - blob["dnn.state_prior"].astype(np.float64)
    e_max = lam * s.max(1, keepdims=True)
    droppable = np.where(h < lse + LOG_ADDMIN + 2 * e_max, np.exp(h - lse), 0.0).sum(1, keepdims=True)
    e_lse = e_max + lam * np.sqrt(N - 1) * (ADDLOG_STEP_ERR + U * np.abs(lse)) + droppable
    tol = INV_LOG_TEN * (lam * s + e_lse + U * np.abs(h - lse)) + 2 * U * np.abs(want)
    return want, tol


DNN_SHAPES = [
    # in_dim, hidden, hidden layers, out_dim
    (117, 100, 2, 61),        # no width a multiple of 8: the scalar GEMV path throughout
    (120, 129, 2, 240),
    (429, 257, 1, 61),
    (117, 129, 0, 3001),      # one layer: the first layer is the output layer
    (120, 100, 15, 240),      # 16 layers, the most a descriptor holds
]


@pytest.mark.parametrize("in_dim,hidden,layers,out_dim", DNN_SHAPES)
def test_dnn_restatement_agrees_with_fp64(in_dim, hidden, layers, out_dim, oracle_lib):
    from julius_b200 import synth
    blob = dnn_blob(in_dim, hidden, layers, out_dim, seed=in_dim + hidden + layers)
    ds = desc.Descriptors(blob)
    x = synth.sample_dnn_input(np.random.default_rng(layers), 6, in_dim)
    x[0] *= 8.0                                   # saturating pre-activations: the clamp at +-8
    got = oracle_lib.dnn_score(ds, x)
    want, tol = dnn_f64(blob, x)
    err = np.abs(got.astype(np.float64) - want)
    assert (err <= tol).all(), f"max err {err.max():.3e} where the bound is {tol[np.unravel_index(err.argmax(), err.shape)]:.3e}"
    # and the bound itself is not vacuous: a few 1e-3 log10 units at most, the sqrt(N) table term of 3001 outputs
    assert tol.max() < 5e-3
