"""Monte-Carlo ensembles / scenario sweeps across GPUs (BASELINE configs[3]).

The workload shards as independent units: every rank (one process per GPU) advances its own replicas
(`Context(n_replicas=R, random_seed=seed0 + rank * R)`) with no data-path collective; the only exchange is the
final reduce of the daily curves -- sum and sum of squares per (day, series).  On GPUs that reduce is ONE ncclAllReduce
on device buffers through the engine's own C-ABI (`Context.moments(reduce=True)` -> rb_reduce_moments); percentile
bands gather the members' rows over the same communicator.  Replaces the reference's broken `run_monte_carlo` process
pool (calc/simulation.py:349-385).  No framework is imported here: a communicator is any object with rank / size /
allreduce / allgather / barrier (reina_b200/comm.py; the CPU tests pass an adapter over a gloo group).
"""
import math

import numpy as np

from .comm import LocalComm


def curve_moments(rows):
    """rows[replica, day, series] -> (sum, sum of squares, n) over the replica axis, float64."""
    x = np.asarray(rows, dtype=np.float64)
    return x.sum(axis=0), (x * x).sum(axis=0), x.shape[0]


def reduce_moments(s1, s2, n, comm=None):
    """All-reduce (sum) of host-side curve moments over the communicator, if there is one."""
    comm = comm or LocalComm()
    if comm.size == 1:
        return s1, s2, n
    t = comm.allreduce(np.concatenate([np.ravel(s1), np.ravel(s2), [float(n)]]), 'sum')
    k = s1.size
    return t[:k].reshape(s1.shape), t[k:2 * k].reshape(s2.shape), int(round(t[-1]))


def mean_std(s1, s2, n):
    mean = s1 / n
    var = np.maximum(s2 / n - mean * mean, 0.0) * (n / max(n - 1, 1))
    return mean, np.sqrt(var)


def percentile_bands(rows, q=(5, 25, 50, 75, 95)):
    """Uncertainty bands of an ensemble: rows[replica, day, series] -> {q: [day, series]} (what the reference's UI would
    draw from run_monte_carlo's reina_<scenario>.csv, calc/simulation.py:365-385)."""
    x = np.asarray(rows, dtype=np.float64)
    p = np.percentile(x, list(q), axis=0)
    return {int(k): p[i] for i, k in enumerate(q)}


def gather_rows(rows, comm=None):
    """All ranks' stats rows on every rank (percentiles need the members, not just the moments)."""
    comm = comm or LocalComm()
    rows = np.ascontiguousarray(rows)
    if comm.size == 1:
        return rows
    out = comm.allgather(rows)                       # [rank, replica, day, series]
    return out.reshape((-1,) + rows.shape[1:])


def seeds_for_rank(seed0, replicas_per_rank, rank):
    """Replica r of rank k uses seed seed0 + k * R + r (Context adds r itself)."""
    return seed0 + rank * replicas_per_rank


def run_ensemble(make_context, days, replicas_per_rank, seed0=0, comm=None):
    """Run this rank's share and return the GLOBAL ensemble mean / std of every raw stats column.

    make_context(n_replicas, random_seed) -> reina_b200.model.Context with interventions added.  `comm` None: the
    engine's own NCCL communicator is joined from the launcher's environment (reina_b200.comm.connect) and the reduce
    runs on the device; any other communicator object reduces the host-side moments."""
    from . import comm as _comm
    rank = comm.rank if comm is not None else _comm.world()[0]
    ctx = make_context(replicas_per_rank, seeds_for_rank(seed0, replicas_per_rank, rank))
    if comm is None:
        comm = _comm.connect(ctx._engine)
    ctx.run(days)
    if isinstance(comm, _comm.EngineComm) and comm.engine is ctx._engine:
        s1, s2, n = ctx.moments(0, days, reduce=True)        # device-side: k_moments + one ncclAllReduce
    else:
        s1, s2, n = reduce_moments(*ctx.moments(0, days), comm=comm)
    mean, std = mean_std(s1, s2, n)
    return dict(mean=mean, std=std, n=n, names=ctx.row_layout(), context=ctx, comm=comm)


_TX_SUMS = ('offspring_hist', 'generation_interval_hist', 'group_closed', 'group_offspring', 'variant_closed',
            'variant_offspring')


def transmission_summary(stats, comm=None):
    """Ensemble transmission statistics from Context.transmission_stats() of every rank (one allreduce, like
    reduce_moments).  With K the total number of replicas, n_r[d] / off_r[d] the infected / offspring of cohort d in
    replica r:

      cohort_R[d]      sum off / sum n, the ratio estimator of the cohort reproduction number (NaN where sum n = 0)
      cohort_R_se[d]   its between-replica standard error by the delta method,
                       SE^2 = sum_r (off_r - R n_r)^2 / (nbar^2 K (K - 1)), nbar = sum n / K
      complete[d]      no agent of the cohort can infect any more (sum open == 0); later cohorts are right-censored
      offspring_mean, offspring_var, dispersion_k   of the closed cases' offspring (bin 64 counts as 64);
                       k = m^2 / (v - m), inf when v <= m (no overdispersion)
      gi_pmf[k], gi_mean                            generation-interval distribution in days
      R_by_group[g], R_by_variant[v]                offspring per closed case
    plus the summed tables and K."""
    comm = comm or LocalComm()
    n = np.asarray(stats['cohort_infected'], dtype=np.float64)
    off = np.asarray(stats['cohort_offspring'], dtype=np.float64)
    parts = [n.sum(0), off.sum(0), (off * off).sum(0), (off * n).sum(0), (n * n).sum(0),
             np.asarray(stats['cohort_open'], dtype=np.float64).sum(0)]
    parts += [np.asarray(stats[k], dtype=np.float64).sum(0) for k in _TX_SUMS]
    flat = np.concatenate(parts + [[float(n.shape[0])]])
    if comm.size > 1:
        flat = comm.allreduce(flat, 'sum')
    out, k = {}, 0
    for name, p in zip(('n', 'off', 'off2', 'offn', 'n2', 'open') + _TX_SUMS, parts):
        out[name] = flat[k:k + p.size]
        k += p.size
    K = int(round(flat[-1]))
    sn, so = out.pop('n'), out.pop('off')
    s2, sxn, sn2 = out.pop('off2'), out.pop('offn'), out.pop('n2')
    with np.errstate(divide='ignore', invalid='ignore'):
        R = np.where(sn > 0, so / sn, np.nan)
        nbar = sn / K
        ss = np.maximum(s2 - 2.0 * R * sxn + R * R * sn2, 0.0)
        se = np.sqrt(ss / (nbar * nbar * K * (K - 1))) if K > 1 else np.full_like(R, np.nan)
        se = np.where(sn > 0, se, np.nan)
        h = out['offspring_hist']
        kk = np.arange(h.size, dtype=np.float64)
        nc = h.sum()
        m = (kk * h).sum() / nc if nc > 0 else np.nan
        v = (((kk - m) ** 2) * h).sum() / (nc - 1) if nc > 1 else np.nan
        disp = m * m / (v - m) if v > m else np.inf
        g = out['generation_interval_hist']
        pmf = g / g.sum() if g.sum() > 0 else np.full_like(g, np.nan)
        r_group = np.where(out['group_closed'] > 0, out['group_offspring'] / out['group_closed'], np.nan)
        r_var = np.where(out['variant_closed'] > 0, out['variant_offspring'] / out['variant_closed'], np.nan)
    return dict(n_replicas=K, cohort_infected=sn, cohort_offspring=so, cohort_open=out['open'], cohort_R=R,
                cohort_R_se=se, complete=out['open'] == 0, offspring_mean=m, offspring_var=v, dispersion_k=disp,
                gi_pmf=pmf, gi_mean=float((np.arange(pmf.size) * pmf).sum()), R_by_group=r_group, R_by_variant=r_var,
                **{name: out[name] for name in _TX_SUMS})


def _spectral_radius(m):
    return float(np.abs(np.linalg.eigvals(m)).max()) if m.size else np.nan


def setting_summary(settings, comm=None):
    """Ensemble transmission by setting and age from Context.transmission_settings() of every rank (one allreduce, like
    transmission_summary).  With K the total number of replicas, x_r[p] the infections at place p (p < 6) in replica r
    and c_r = sum_p x_r[p] its children (agents with an infector):

      share[p]                 sum x[p] / sum c, the share of infections that happened at place p (Context.PLACE_NAMES)
      share_se[p]              its between-replica standard error by the delta method,
                               SE^2 = sum_r (x_r[p] - share[p] c_r)^2 / (cbar^2 K (K - 1)), cbar = sum c / K
      incidence_by_place_mean[d, p], incidence_by_place_std[d, p]   infections per day and place (p = 6: imports and
                               the initial state) over the replicas
      waifw[i, j]              infections of age group j by age group i, all places and replicas (who acquires
                               infection from whom)
      ngm[i, j]                the empirical next-generation matrix: infections in group i per closed case of group j,
                               sum_p pair_closed[p, j, i] / closed_by_group[j] (NaN where a group has no closed case);
                               ngm_by_place[p] the same for the infections at place p, so ngm = sum_p ngm_by_place[p]
      R_by_place[p]            sum pair_closed[p] / sum closed_by_group: offspring per closed case at place p
      rho                      the spectral radius of ngm (NaN columns taken as 0)
      rho_without[p]           the spectral radius of ngm - ngm_by_place[p]

    rho_without is a first-order decomposition: it removes place p's transmissions from the matrix observed in this run
    and holds everything else fixed -- the depletion of susceptibles, who was infected when, and behaviour.  It is not a
    simulated counterfactual; an intervention that closes a place is evaluated by running it.
    Also returned: the summed tables by_day_place, pair_all, pair_closed, closed_by_group, and K."""
    comm = comm or LocalComm()
    P = len(np.asarray(settings['pair_all'])[0])
    bdp = np.asarray(settings['by_day_place'], dtype=np.float64)
    x = bdp[:, :, :P].sum(axis=1)                       # [K_rank, P]
    c = x.sum(axis=1)
    parts = [x.sum(0), (x * x).sum(0), (x * c[:, None]).sum(0), [(c * c).sum()], bdp.sum(0), (bdp * bdp).sum(0)]
    parts += [np.asarray(settings[k], dtype=np.float64).sum(0) for k in ('pair_all', 'pair_closed', 'closed_by_group')]
    flat = np.concatenate([np.ravel(p) for p in parts] + [[float(bdp.shape[0])]])
    if comm.size > 1:
        flat = comm.allreduce(flat, 'sum')
    out, k = [], 0
    for p in parts:
        n = np.size(p)
        out.append(flat[k:k + n].reshape(np.shape(p)))
        k += n
    sx, sx2, sxc, (sc2,), s_bdp, s_bdp2, pair_all, pair_closed, closed = out
    K = int(round(flat[-1]))
    sc = sx.sum()
    with np.errstate(divide='ignore', invalid='ignore'):
        share = sx / sc if sc > 0 else np.full(P, np.nan)
        cbar = sc / K
        ss = np.maximum(sx2 - 2.0 * share * sxc + share * share * sc2, 0.0)
        se = np.sqrt(ss / (cbar * cbar * K * (K - 1))) if K > 1 and sc > 0 else np.full(P, np.nan)
        inc_mean, inc_std = mean_std(s_bdp, s_bdp2, K)
        ngm_by_place = np.where(closed[None, None, :] > 0, pair_closed.transpose(0, 2, 1) / closed[None, None, :], np.nan)
        r_place = pair_closed.sum(axis=(1, 2)) / closed.sum() if closed.sum() > 0 else np.full(P, np.nan)
    ngm = ngm_by_place.sum(axis=0)
    m = np.nan_to_num(ngm)
    m_place = np.nan_to_num(ngm_by_place)
    return dict(n_replicas=K, share=share, share_se=se, incidence_by_place_mean=inc_mean, incidence_by_place_std=inc_std,
                waifw=pair_all.sum(axis=0), ngm=ngm, ngm_by_place=ngm_by_place, R_by_place=r_place,
                rho=_spectral_radius(m), rho_without=np.array([_spectral_radius(m - m_place[p]) for p in range(P)]),
                by_day_place=s_bdp, pair_all=pair_all, pair_closed=pair_closed, closed_by_group=closed)


# ---------------------------------------------------------------- conditioning on observed counts
def systematic_resample(weights, rng):
    """Systematic resampling: how many copies of each replica to keep, counts[r] >= 0 with sum R, for normalised or
    unnormalised weights >= 0 (one uniform from the numpy Generator `rng`)."""
    w = np.asarray(weights, dtype=np.float64)
    if w.ndim != 1 or w.size == 0 or not np.isfinite(w).all() or (w < 0).any() or not w.sum() > 0:
        raise ValueError('weights must be finite, >= 0 and not all 0')
    R = w.size
    cum = np.cumsum(w / w.sum())
    cum[-1] = 1.0
    idx = np.searchsorted(cum, (rng.random() + np.arange(R)) / R, side='right')
    return np.bincount(np.minimum(idx, R - 1), minlength=R)


def assign_slots(counts):
    """The `source` of Context.branch for resampling counts: a replica with counts >= 1 keeps its slot, its extra copies
    fill the slots of the replicas with count 0 in increasing order.  So source[source[j]] == source[j] always."""
    c = np.asarray(counts, dtype=np.int64)
    if c.ndim != 1 or (c < 0).any() or c.sum() != c.size:
        raise ValueError('counts must be >= 0 and sum to their number')
    src = np.arange(c.size)
    src[c == 0] = np.repeat(np.arange(c.size), np.maximum(c - 1, 0))
    return src.astype(np.int32)


def _lgamma(x):
    return np.vectorize(math.lgamma, otypes=[np.float64])(x)


def log_likelihood(mean, observed, model='negbin', dispersion=10.0):
    """log P(observed | model count `mean`) per replica: negative binomial with that mean and dispersion k (variance
    mean + mean^2 / k), or Poisson.  A mean of 0 gives 0 for an observed 0 and -inf otherwise."""
    mu = np.asarray(mean, dtype=np.float64)
    y = float(observed)
    if y < 0 or y != int(y):
        raise ValueError('an observed count must be a non-negative integer, got %r' % observed)
    with np.errstate(divide='ignore', invalid='ignore'):
        if model == 'poisson':
            ll = y * np.log(mu) - mu - math.lgamma(y + 1.0)
        elif model == 'negbin':
            k = float(dispersion)
            if not k > 0:
                raise ValueError('dispersion must be > 0')
            ll = (_lgamma(y + k) - math.lgamma(k) - math.lgamma(y + 1.0) + k * np.log(k / (k + mu))
                  + y * np.log(mu / (k + mu)))
        else:
            raise ValueError("model must be 'negbin' or 'poisson'")
    return np.where(mu > 0, ll, 0.0 if y == 0 else -np.inf)


def _model_counts(ctx, rows, name):
    """Column `name` of stats rows [replica, row]: an ATTRS name summed over the age groups, or a row_layout() column."""
    from ._abi import ATTRS
    G = len(ctx.age_group_labels)
    if name in ATTRS:
        i = ATTRS.index(name)
        return rows[:, i * G:(i + 1) * G].sum(axis=1)
    names = ctx.row_layout()
    if name not in names:
        raise ValueError('unknown observation %r: an ATTRS name or a row_layout() column' % name)
    return rows[:, names.index(name)]


def _logsumexp(x):
    m = x.max()
    return m + math.log(np.exp(x - m).sum()) if np.isfinite(m) else m


def particle_filter(ctx, observations, *, model='negbin', dispersion=10.0, ess_threshold=0.5, seed=0):
    """Sequential importance resampling of the replicas of ONE Context against observed counts.

    observations = {day: {name: count}}: `name` is an ATTRS name summed over the age groups ('in_ward', 'in_icu',
    'dead', 'all_detected', ...) or a row_layout() column.  The observation of day d is compared with stats row d, the
    state before the d-th iterate() (what generate_state() returns at ctx.day == d); the days must not lie before
    ctx.day.  The likelihood of a replica is a negative binomial with mean equal to its count and dispersion k
    (`dispersion`), or Poisson (model='poisson'); several names on one day are independent.  After each observation
    day the weights are updated, and when the effective sample size falls below ess_threshold * R -- and always at the
    last observation -- the replicas are resampled systematically (systematic_resample with a Generator seeded by
    `seed`) and copied on the device with Context.branch (assign_slots): every copy continues with a fresh seed.

    The Context is left at the last observation day, equally weighted, so run(), series(), moments() and
    percentile_bands() give the forecast from there.  The rows of days before it are the paths of the surviving
    replicas' ancestors: for early days few distinct paths remain (they degenerate), so read the past from the filter's
    weights at each day, not from the returned ensemble.  Resampling across GPUs (moving replica state between ranks) is
    not provided: every rank filters its own replicas.

    Returns a dict: log_evidence (the sum over the observation days of the log mean incremental weight), days[k],
    ess[k] (before resampling), resampled[k], ancestors[k, R] (the branch source of step k, the identity where nothing
    was resampled) and loglik[k, R].  Raises ValueError naming the day if no replica can explain an observation (every
    weight zero)."""
    R = ctx.n_replicas
    days = sorted(int(d) for d in observations)
    if days and (days[0] < ctx.day or days[-1] > ctx.max_days):
        raise ValueError('observation days must lie in [ctx.day, max_days] = [%d, %d]' % (ctx.day, ctx.max_days))
    rng = np.random.default_rng(seed)
    logw = np.full(R, -math.log(R))
    out = dict(log_evidence=0.0, days=np.array(days, dtype=np.int64), ess=np.zeros(len(days)),
               resampled=np.zeros(len(days), dtype=bool), ancestors=np.zeros((len(days), R), dtype=np.int32),
               loglik=np.zeros((len(days), R)))
    for k, d in enumerate(days):
        if d > ctx.day:
            ctx.run(d - ctx.day)
        ctx._engine.snapshot()
        ctx._engine.sync()
        ctx._state_day = ctx.day
        rows = ctx._engine.read_stats(d, 1)[:, 0].astype(np.float64)
        ll = np.zeros(R)
        for name, y in observations[d].items():
            ll += log_likelihood(_model_counts(ctx, rows, name), y, model, dispersion)
        post = logw + ll
        total = _logsumexp(post)
        if not np.isfinite(total):
            raise ValueError('particle_filter: no replica can explain the observations of day %d (every weight is 0)' % d)
        out['log_evidence'] += total                  # logw is normalised: log sum_j W_j exp(ll_j)
        logw = post - total
        w = np.exp(logw)
        ess = 1.0 / (w * w).sum()
        src = np.arange(R, dtype=np.int32)
        if ess < ess_threshold * R or k == len(days) - 1:
            src = assign_slots(systematic_resample(w, rng))
            if (src != np.arange(R)).any():
                ctx.branch(src)
            logw = np.full(R, -math.log(R))
            out['resampled'][k] = True
        out['ess'][k], out['ancestors'][k], out['loglik'][k] = ess, src, ll
    return out
