"""Reference finite-size Lyapunov exponents (FSLE) of buoy pairs: first-passage state per pair and the exit times
between separation thresholds (test infrastructure only; the product never imports it).

Definitions -- the contract of csrc/st_fsle.cu, sitrack_b200.fsle and DESIGN.md section 14 (Aurell et al. 1997;
Lacorata et al. 2001; LaCasce 2008):

Inputs.    Pairs (nQ,2) i4 buoy indices in the caller's order, a != b, 1 <= nQ < 2^31 (dispersion.check_pairs).
           Thresholds `deltas`: K f8 values, finite, positive, strictly increasing, 2 <= K <= 64; default
           2.0 ** (1 + j/2), j = 0 .. 18 (2 ... 1024 km).  Samples: rows s*n, s = 0, 1, ..., with every = n; row 0 is
           the state handed to set_buoys, masked by the rec_first rule of the engine's _WindowRows; one sample is
           n*rdt/86400 days; sample indices are at most 65535.
Per pair.  At each sample, in f8 and in this order: dy = y_a - y_b, dx = x_a - x_b, r = sqrt(dy*dy + dx*dx).  The
           sample is valid when both masks are != 0 and r is finite (NaN and +-inf end or delay a pair, never binned).
           b = searchsorted(deltas, r, side="right"): the thresholds at or below r, so a tie reaches the threshold.
State.     (nQ,2) i4 {level, anchor}: level -1 not started, -2 ended, 0..K thresholds reached; anchor the sample at
           which the current level was first reached, -1 when unknown.
Update.    At sample t:
             not started, valid:      level = b, anchor = -1, n_start[b] += 1 (a pair starting above delta_j reached
                                      delta_j unseen: its first transition is not timed);
             not started, not valid:  nothing;
             started, not valid:      level = -2; n_censored[level-1] += 1 when anchor >= 0 and level < K;
             started, valid:          L' = max(level, b) (levels never go down: first passages).  If L' > level:
                                      record tau = t - anchor for transition level-1 when level >= 1 and anchor >= 0,
                                      record tau = 0 for transitions level .. L'-2 (thresholds first reached in the
                                      same sample interval: bin 0 shows the sampling limit), then anchor = t and
                                      level = L'.  A pair at level K records nothing more.
           Recording tau for transition j (0..K-2): hist_tau[j][searchsorted(tau_edges, tau, side="right")] += 1,
           sum_tau[j] += tau, sum_tau2[j] += tau^2.  tau_edges: 1..512 f8 edges in samples (check_edges); default
           1, 2, 4, ... 2^16, so bin 0 is tau = 0.
Stats.     Per window, all i8 and exact: n_start (K+1), hist_tau (K-1, len(tau_edges)+1), n (K-1) its row sums,
           sum_tau, sum_tau2, n_censored (K-1).  Window w holds the events of sample w+1, window 0 also those of
           sample 0, so the windows sum to the whole run.  lambda_j = ln(delta_{j+1}/delta_j) / (sample_days *
           sum_tau_j / n_j) [day-1] from the summed windows (sitrack_b200.fsle_lambda).

`sample` is vectorised over pairs; `sample_loop` is a plain per-pair loop that the tests hold it to.
"""
import math

import numpy as np

DEFAULT_DELTAS = np.array([2.0 ** (1 + j / 2) for j in range(19)])                 # 2 ... 1024 km
DEFAULT_TAU_EDGES = np.array([2.0 ** k for k in range(17)])                        # 1, 2, 4, ... 65536 samples


def empty_stats(K, ntau):
    J = K - 1
    return dict(n_start=np.zeros(K + 1, np.int64), hist_tau=np.zeros((J, ntau + 1), np.int64),
                n=np.zeros(J, np.int64), sum_tau=np.zeros(J, np.int64), sum_tau2=np.zeros(J, np.int64),
                n_censored=np.zeros(J, np.int64))


def add_stats(a, b):
    return {k: a[k] + b[k] for k in a}


def new_state(nQ):
    return np.full((nQ, 2), -1, np.int32)


def separation(yx, pairs):
    """(nQ,) f8 r of every pair, in the contract's order."""
    yx = np.asarray(yx, np.float64)
    a, b = np.asarray(pairs, np.int64)[:, 0], np.asarray(pairs, np.int64)[:, 1]
    with np.errstate(all="ignore"):
        dy, dx = yx[a, 0] - yx[b, 0], yx[a, 1] - yx[b, 1]
        return np.sqrt(dy * dy + dx * dx)


def sample(state, yx, m, pairs, t, deltas=DEFAULT_DELTAS, tau_edges=DEFAULT_TAU_EDGES):
    """One sample t of every pair: -> (new state (nQ,2) i4, the stats of its events)."""
    deltas, tau_edges = np.asarray(deltas, np.float64), np.asarray(tau_edges, np.float64)
    K, ntau = deltas.size, tau_edges.size
    p = np.asarray(pairs, np.int64)
    m = np.asarray(m)
    r = separation(yx, pairs)
    valid = (m[p[:, 0]] != 0) & (m[p[:, 1]] != 0) & np.isfinite(r)
    b = np.searchsorted(deltas, r, side="right")
    L, A = np.asarray(state, np.int32)[:, 0].astype(np.int64), np.asarray(state, np.int32)[:, 1].astype(np.int64)
    st = empty_stats(K, ntau)
    start = (L == -1) & valid
    st["n_start"] += np.bincount(b[start], minlength=K + 1)
    started = L >= 0
    end = started & ~valid
    cens = end & (A >= 0) & (L < K)
    st["n_censored"] += np.bincount(L[cens] - 1, minlength=K - 1)
    up = started & valid & (b > L)
    timed = up & (L >= 1) & (A >= 0)
    nz = np.where(up, b - 1 - L, 0).clip(0)                   # zero-tau transitions level .. b-2 per pair
    j = np.r_[L[timed] - 1, np.repeat(L, nz) + (np.arange(nz.sum()) - np.repeat(np.cumsum(nz) - nz, nz))]
    tau = np.r_[t - A[timed], np.zeros(int(nz.sum()), np.int64)]
    np.add.at(st["hist_tau"], (j, np.searchsorted(tau_edges, tau.astype(np.float64), side="right")), 1)
    np.add.at(st["sum_tau"], j, tau)
    np.add.at(st["sum_tau2"], j, tau * tau)
    st["n"] = st["hist_tau"].sum(1)
    L2, A2 = L.copy(), A.copy()
    L2[start], A2[start] = b[start], -1
    L2[end] = -2
    L2[up], A2[up] = b[up], t
    return np.stack([L2, A2], 1).astype(np.int32), st


def sample_loop(state, yx, m, pairs, t, deltas=DEFAULT_DELTAS, tau_edges=DEFAULT_TAU_EDGES):
    """`sample` as a plain loop over pairs, one statement per rule."""
    deltas, tau_edges = [float(d) for d in deltas], [float(e) for e in tau_edges]
    K = len(deltas)
    st = empty_stats(K, len(tau_edges))
    out = np.array(state, np.int32).copy()

    def record(j, tau):
        k = sum(1 for e in tau_edges if e <= tau)
        st["hist_tau"][j, k] += 1
        st["n"][j] += 1
        st["sum_tau"][j] += tau
        st["sum_tau2"][j] += tau * tau

    for i, (a, b) in enumerate(np.asarray(pairs).tolist()):
        level, anchor = int(out[i, 0]), int(out[i, 1])
        dy = float(yx[a][0]) - float(yx[b][0])
        dx = float(yx[a][1]) - float(yx[b][1])
        r = math.sqrt(dy * dy + dx * dx)
        ok = m[a] != 0 and m[b] != 0 and math.isfinite(r)
        nb = sum(1 for d in deltas if d <= r) if ok else -9
        if level == -2:
            continue
        if level == -1:
            if ok:
                level, anchor = nb, -1
                st["n_start"][nb] += 1
        elif not ok:
            if anchor >= 0 and level < K:
                st["n_censored"][level - 1] += 1
            level = -2
        elif nb > level:
            if level >= 1 and anchor >= 0:
                record(level - 1, t - anchor)
            for j in range(level, nb - 1):
                record(j, 0)
            level, anchor = nb, t
        out[i] = level, anchor
    return out, st


def run(rows, masks, pairs, deltas=DEFAULT_DELTAS, tau_edges=DEFAULT_TAU_EDGES, every=1, step=sample):
    """The samples rows[s*every], s = 0 .. S (S = (len(rows)-1) // every): -> (states (S, nQ, 2) after each window,
    the S windows' stats); window w holds sample w+1, window 0 also sample 0."""
    S = (len(rows) - 1) // every
    state = new_state(len(pairs))
    state, first = step(state, rows[0], masks[0], pairs, 0, deltas, tau_edges)
    states, wins = [], []
    for s in range(1, S + 1):
        state, st = step(state, rows[s * every], masks[s * every], pairs, s, deltas, tau_edges)
        if s == 1:
            st = add_stats(first, st)
        states.append(state)
        wins.append(st)
    return np.array(states).reshape(S, len(pairs), 2), wins
