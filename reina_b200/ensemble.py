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

from . import model as _model
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


def migration_plan(counts, n_ranks):
    """The global `source` for resampling counts over n_ranks x R replicas (rank k holds global indices k R .. k R + R - 1)
    that moves the fewest replicas between ranks: a replica with counts >= 1 keeps its slot, a rank's extra copies fill
    that rank's own dropped slots first (in increasing order), and only the remaining dropped slots are filled across
    ranks, with the remaining extra copies, both in increasing global order.  That is sum_k max(0, dropped_k - extras_k)
    moves, the least any plan needs.  source[source[j]] == source[j]; with n_ranks = 1 it is assign_slots(counts)."""
    c = np.asarray(counts, dtype=np.int64)
    if c.ndim != 1 or (c < 0).any() or c.sum() != c.size:
        raise ValueError('counts must be >= 0 and sum to their number')
    if n_ranks < 1 or c.size % n_ranks:
        raise ValueError('%d counts do not split over %d ranks' % (c.size, n_ranks))
    R = c.size // n_ranks
    src = np.arange(c.size)
    holes, extras = [], []
    for k in range(n_ranks):
        ck = c[k * R:(k + 1) * R]
        extra = np.repeat(np.arange(R), np.maximum(ck - 1, 0)) + k * R
        dropped = np.flatnonzero(ck == 0) + k * R
        m = min(extra.size, dropped.size)
        src[dropped[:m]] = extra[:m]
        holes.append(dropped[m:])
        extras.append(extra[m:])
    src[np.concatenate(holes)] = np.concatenate(extras)
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


def _gather(comm, x):
    """[ranks * len(x), ...] of every rank's x (uint32 travels as int32: not every collective backend has uint32)."""
    x = np.ascontiguousarray(x)
    if comm.size == 1:
        return x
    if x.dtype == np.uint32:
        return np.asarray(comm.allgather(x.view(np.int32))).view(np.uint32).reshape((-1,) + x.shape[1:])
    return np.asarray(comm.allgather(x)).reshape((-1,) + x.shape[1:])


def _move_replicas(ctxs, comm, rank, src, seeds, R):
    """Apply the global plan `src` with the global `seeds` to this process's Contexts (ctxs[i] holds global replicas
    (rank + i) R ..): Context.branch for sources on the same Context, copy_replicas_from between the Contexts of this
    process, rb_comm_move_replicas over the engine's own communicator, else host records through comm.sendrecv."""
    from .comm import EngineComm
    N = src.size
    for i, c in enumerate(ctxs):                      # sources on the same Context
        g0 = (rank + i) * R
        loc = np.arange(R, dtype=np.int32)
        same = (src[g0:g0 + R] // R) == (g0 // R)
        loc[same] = src[g0:g0 + R][same] - g0
        if (loc != np.arange(R)).any():
            c.branch(loc, seeds[g0:g0 + R])
    cross = [j for j in range(N) if src[j] // R != j // R]            # increasing global destination order
    if not cross:
        return
    if comm.size == 1:                                # the Contexts of this process
        pairs = {}
        for j in cross:
            pairs.setdefault((j // R, src[j] // R), []).append(j)
        for (kd, ks), js in pairs.items():
            js = np.array(js)
            ctxs[kd].copy_replicas_from(ctxs[ks], src[js] % R, js % R, seeds[js])
        return
    ctx = ctxs[0]
    send = [j for j in cross if src[j] // R == rank]
    recv = [j for j in cross if j // R == rank]
    if isinstance(comm, EngineComm) and comm.engine is ctx._engine:
        ctx._engine.comm_move_replicas([src[j] % R for j in send], [j // R for j in send], [j % R for j in recv],
                                       [src[j] // R for j in recv], seeds[recv])
        ctx._state_day = -1
        return
    if not hasattr(comm, 'sendrecv'):
        raise TypeError('particle_filter: moving replicas between ranks needs the engine\'s own EngineComm or a '
                        'communicator with sendrecv({peer: bytes}) -> {peer: bytes}')
    out = {}
    for j in send:
        out.setdefault(j // R, []).append(src[j] % R)
    payload = {p: ctx.export_replicas(idx).tobytes() for p, idx in out.items()}
    got = comm.sendrecv(payload)
    by_peer = {}
    for j in recv:
        by_peer.setdefault(src[j] // R, []).append(j)
    for p, js in sorted(by_peer.items()):
        js = np.array(js)
        ctx.import_replicas(js % R, np.frombuffer(got[p], dtype=np.uint8).reshape(len(js), -1), seeds[js])


# the range a filtered scale is kept in: the engine accepts (0, 16]
_LOG_SCALE_MIN, _LOG_SCALE_MAX = math.log(1.0 / 16.0), math.log(16.0)


class _FilteredScale:
    """One per-replica log-scale parameter the particle filter estimates along with the state: the prior draw, the
    scales each observation's weights judged, the resampling and the random-walk step, for every global replica.
    `put(ctx, values)` sets one Context's slice (ctxs[i] holds global replicas (rank + i) R ..)."""

    def __init__(self, what, prior, volatility, put, rng, N, n_days):
        median, log_sd = (float(x) for x in prior)
        if not (median > 0 and log_sd >= 0 and volatility >= 0):
            raise ValueError('%s needs median > 0 and log_sd >= 0, and the volatility must be >= 0' % what)
        self.volatility, self.put = volatility, put
        self.log = np.clip(rng.normal(math.log(median), log_sd, N), _LOG_SCALE_MIN, _LOG_SCALE_MAX)
        self.value = np.exp(self.log).astype(np.float32)
        self.judged = np.zeros((n_days, N), dtype=np.float32)

    def resample_and_step(self, src, rng, dt):
        """Follow the resampling (the copies already carry their source's scale on the device), then take the step to
        the next observation (dt days; None after the last).  True when the values changed and must be set."""
        self.log, self.value = self.log[src], self.value[src]
        if dt is None or self.volatility <= 0:
            return False
        self.log = np.clip(self.log + self.volatility * math.sqrt(dt) * rng.standard_normal(self.log.size),
                           _LOG_SCALE_MIN, _LOG_SCALE_MAX)
        self.value = np.exp(self.log).astype(np.float32)
        return True

    def set(self, ctxs, rank, R):
        for i, c in enumerate(ctxs):
            g0 = (rank + i) * R
            self.put(c, self.value[g0:g0 + R])


def particle_filter(ctx, observations, *, model='negbin', dispersion=10.0, ess_threshold=0.5, seed=0, comm=None,
                    transmission_prior=None, transmission_volatility=0.0, severity_prior=None, severity_volatility=0.0):
    """Sequential importance resampling of an ensemble against observed counts: the replicas of ONE Context, of a list
    of Contexts of this process, or of every rank's Context (`comm`, one Context per rank), filtered as ONE set of
    particles.  Global replica g = k R + r is replica r of Context / rank k; every Context holds R replicas.

    observations = {day: {name: count}}: `name` is an ATTRS name summed over the age groups ('in_ward', 'in_icu',
    'dead', 'all_detected', ...) or a row_layout() column.  The observation of day d is compared with stats row d, the
    state before the d-th iterate() (what generate_state() returns at ctx.day == d); the days must not lie before
    ctx.day.  The likelihood of a replica is a negative binomial with mean equal to its count and dispersion k
    (`dispersion`), or Poisson (model='poisson'); several names on one day are independent.  After each observation
    day the log-likelihoods of all replicas are gathered (comm.allgather, or over the list), the weights are updated, and
    when the effective sample size falls below ess_threshold * K R -- and always at the last observation -- the replicas
    are resampled systematically (systematic_resample with a Generator seeded by `seed`, the same on every rank) and
    copied with the plan of migration_plan, which moves the fewest replicas between Contexts.  Every copy continues with
    a fresh seed: Context.branch's rule over the union of every Context's seed history, in global order.  Copies on one
    Context use Context.branch; between Contexts of this process copy_replicas_from; between ranks
    rb_comm_move_replicas when `comm` is the engine's own EngineComm, else host records through comm.sendrecv.  A list
    of Contexts together with a communicator of several ranks is refused.

    The Contexts are left at the last observation day, equally weighted, so run(), series(), moments() and
    percentile_bands() give the forecast from there.  The rows of days before it are the paths of the surviving
    replicas' ancestors: for early days few distinct paths remain (they degenerate), so read the past from the filter's
    weights at each day, not from the returned ensemble.

    Returns a dict, the same on every rank: log_evidence (the sum over the observation days of the log mean incremental
    weight), days[k], ess[k] (before resampling), resampled[k], ancestors[k, K R] (the global source of step k, the
    identity where nothing was resampled), loglik[k, K R] and seeds[k, K R] (every replica's seed from that day on), and
    weights[k, K R] (normalised, before resampling).  Raises ValueError naming the day if no replica can explain an
    observation (every weight zero).

    transmission_prior = (median, log_sd) filters every replica's transmission scale f (Context.set_transmission_scale)
    together with its state.  Before the first observation every global replica draws log f ~ N(log median, log_sd^2)
    from the filter's Generator, in global order, the same on every rank.  At each observation day but the last, after
    the weight update and any resampling (a copy arrives with its source's f), every replica takes a random-walk step
    log f += transmission_volatility * sqrt(d_next - d) * eps, eps ~ N(0, 1), when the volatility is > 0.  log f is kept
    in [log 1/16, log 16].  After the last observation there is no step: the forecast runs with the scales in force.  The
    output then also holds transmission_scale[k, K R], the scales (float32, as set) the weights of day k judged:
    weighted_quantiles(out['transmission_scale'][k], out['weights'][k], q) is the scale's posterior band at that day.
    With transmission_prior None, transmission_scale is None and the Contexts' scales are never touched.

    severity_prior = {name: (median, log_sd)} for any of model.SEVERITY_SCALES ('severe', 'critical', 'fatal') filters
    those severity scales (Context.set_severity_scale) the same way, each with its own prior and the random-walk step
    severity_volatility * sqrt(d_next - d) * eps.  They pin down what the transmission scale alone cannot: `severe` moves
    in_ward, `critical` in_icu and `fatal` dead per infection, so together with all_detected the filter can tell more
    infections from sicker ones.  The Generator draws the transmission scale first (prior and every step, exactly as
    without severity_prior), then severe, critical and fatal, the named ones only; scales not named are never touched.
    The output holds severity_scale = {name: [k, K R] float32}, the scales the weights of day k judged, for the named
    scales; with severity_prior None it is None and no severity call is made."""
    ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
    comm = comm or LocalComm()
    if not ctxs or (len(ctxs) > 1 and comm.size > 1):
        raise ValueError('particle_filter: one Context per rank, or a list of Contexts without a communicator of several ranks')
    R, c0 = ctxs[0].n_replicas, ctxs[0]
    if any(c.n_replicas != R or c.day != c0.day for c in ctxs):
        raise ValueError('particle_filter: the Contexts must hold as many replicas each and be at the same day')
    rank = comm.rank if comm.size > 1 else 0
    N = R * len(ctxs) * comm.size
    days = sorted(int(d) for d in observations)
    if days and (days[0] < c0.day or days[-1] > c0.max_days):
        raise ValueError('observation days must lie in [ctx.day, max_days] = [%d, %d]' % (c0.day, c0.max_days))
    rng = np.random.default_rng(seed)
    logw = np.full(N, -math.log(N))
    out = dict(log_evidence=0.0, days=np.array(days, dtype=np.int64), ess=np.zeros(len(days)),
               resampled=np.zeros(len(days), dtype=bool), ancestors=np.zeros((len(days), N), dtype=np.int32),
               loglik=np.zeros((len(days), N)), seeds=np.zeros((len(days), N), dtype=np.uint32),
               weights=np.zeros((len(days), N)), transmission_scale=None, severity_scale=None)
    if severity_prior is not None and (not severity_prior or set(severity_prior) - set(_model.SEVERITY_SCALES)):
        raise ValueError('severity_prior: a dict over some of %s, not %r' % (_model.SEVERITY_SCALES, sorted(severity_prior)))
    scales = {}                                       # transmission first, then severe, critical, fatal: the draw order
    if transmission_prior is not None:
        scales['transmission'] = _FilteredScale('transmission_prior', transmission_prior, transmission_volatility,
                                                lambda c, v: c.set_transmission_scale(v), rng, N, len(days))
    for name in _model.SEVERITY_SCALES:
        if severity_prior is not None and name in severity_prior:
            scales[name] = _FilteredScale('severity_prior[%r]' % name, severity_prior[name], severity_volatility,
                                          lambda c, v, name=name: c.set_severity_scale(**{name: v}), rng, N, len(days))
    for s in scales.values():
        s.set(ctxs, rank, R)
    hist = None
    for k, d in enumerate(days):
        parts = []
        for c in ctxs:
            if d > c.day:
                c.run(d - c.day)
            c._engine.snapshot()
            c._engine.sync()
            c._state_day = c.day
            rows = c._engine.read_stats(d, 1)[:, 0].astype(np.float64)
            ll = np.zeros(R)
            for name, y in observations[d].items():
                ll += log_likelihood(_model_counts(c, rows, name), y, model, dispersion)
            parts.append(ll)
        ll = _gather(comm, np.concatenate(parts))
        if hist is None:                              # the seed history of every replica, in global order
            hist = _gather(comm, np.concatenate([c._engine.read_seeds() for c in ctxs]))
        post = logw + ll
        total = _logsumexp(post)
        if not np.isfinite(total):
            raise ValueError('particle_filter: no replica can explain the observations of day %d (every weight is 0)' % d)
        out['log_evidence'] += total                  # logw is normalised: log sum_j W_j exp(ll_j)
        logw = post - total
        w = np.exp(logw)
        ess = 1.0 / (w * w).sum()
        out['weights'][k] = w
        for s in scales.values():
            s.judged[k] = s.value
        src = np.arange(N, dtype=np.int32)
        if ess < ess_threshold * N or k == len(days) - 1:
            src = migration_plan(systematic_resample(w, rng), N // R)
            changed = np.flatnonzero(src != np.arange(N))
            seeds = hist[:, d].astype(np.int64)
            seeds[changed] = _model.fresh_seeds(hist, changed.size)
            if changed.size:
                _move_replicas(ctxs, comm, rank, src, seeds.astype(np.uint32), R)
                hist[:, :d] = hist[src, :d]
                hist[:, d:] = seeds.astype(np.uint32)[:, None]
            logw = np.full(N, -math.log(N))
            out['resampled'][k] = True
        out['ess'][k], out['ancestors'][k], out['loglik'][k] = ess, src, ll
        out['seeds'][k] = hist[:, d]
        for s in scales.values():
            if s.resample_and_step(src, rng, days[k + 1] - d if k < len(days) - 1 else None):
                s.set(ctxs, rank, R)
    if 'transmission' in scales:
        out['transmission_scale'] = scales['transmission'].judged
    if severity_prior is not None:
        out['severity_scale'] = {n: scales[n].judged for n in _model.SEVERITY_SCALES if n in scales}
    return out


def weighted_quantiles(values, weights, q):
    """Quantiles of weighted samples along the last axis: for each q, the smallest value whose share of the total weight
    at or below it is >= q (the inverse of the weighted empirical distribution function; with equal weights
    np.quantile(..., method='inverted_cdf')).  values and weights [..., N], weights >= 0 with a positive sum along the last
    axis; q a number or a sequence in [0, 1].  Returns [...] for a number, [len(q), ...] for a sequence: e.g. the 5 / 50 /
    95 % band of a particle filter's transmission scale at every observation day from out['transmission_scale'] and
    out['weights']."""
    x = np.asarray(values, dtype=np.float64)
    if x.ndim == 0 or x.shape[-1] == 0:
        raise ValueError('values need a last axis of at least one sample')
    w = np.broadcast_to(np.asarray(weights, dtype=np.float64), x.shape)
    if not np.isfinite(w).all() or (w < 0).any() or not (w.sum(-1) > 0).all():
        raise ValueError('weights must be finite, >= 0 and not all 0 along the last axis')
    qs = np.asarray(q, dtype=np.float64)
    if ((qs < 0) | (qs > 1)).any():
        raise ValueError('quantiles must lie in [0, 1]')
    order = np.argsort(x, axis=-1, kind='stable')
    xs, cw = np.take_along_axis(x, order, -1), np.cumsum(np.take_along_axis(w, order, -1), axis=-1)
    cw = cw / cw[..., -1:]
    idx = np.stack([np.minimum((cw < qi).sum(-1), x.shape[-1] - 1) for qi in np.atleast_1d(qs)])
    res = np.take_along_axis(np.broadcast_to(xs, idx.shape[:1] + xs.shape), idx[..., None], -1)[..., 0]
    return res[0] if qs.ndim == 0 else res
