"""Reference buoy connectivity between regions: per-buoy transit state, region-to-region transitions, source-to-region
occupancy and first-arrival times (test infrastructure only; the product never imports it).

Definitions -- the contract of csrc/st_connect.cu, sitrack_b200.connect and DESIGN.md section 16 (DeRepentigny et al.
2016; Newton et al. 2017):

Regions.   A label map `labels` (Nj, Ni) on the T-grid, u8 on the device: 0 = in no region, 1..R regions, 1 <= R <= 31
           the largest label.  A buoy's region is labels[jT, iT] of its host cell, bit 31 of the jT word (the
           discontinued flag) stripped.  The Python side refuses a map of the wrong shape, negative, non-integral or
           larger-than-31 labels and a map without a label >= 1 (masked values become 0); the kernel counts a label
           above R as 0, and so does this reference.
Samples.   Rows s*n, s = 0, 1, ..., with every = n; row 0 is the state handed to set_buoys, masked as the engine's
           _WindowRows.m0; at most 65535 samples.
Valid.     The row mask is != 0 and the cell lies in 1 <= jT <= Nj-2, 1 <= iT <= Ni-2.
State.     Per buoy: status (0 not started, 1 started, 2 ended), src (the region at its start sample), prev (the
           region at the previous sample), start (the start sample) and visited (bit r-1 for each region r entered).
Update.    At sample t, cur = the buoy's region:
             not started, valid:      src = prev = cur, start = t, visited = bit(cur) when cur >= 1; n_start[src] += 1,
                                      count[src][cur] += 1 (not at t = 0);
             not started, not valid:  nothing;
             started, not valid:      ended for good; n_end[src] += 1;
             started, valid:          trans[prev][cur] += 1, count[src][cur] += 1; when cur >= 1 and bit(cur) is not
                                      in visited, a first arrival with tau = t - start (>= 1): n_arrive[src][cur-1],
                                      sum_tau[src][cur-1] += tau, sum_tau2 += tau^2,
                                      hist_tau[src][cur-1][searchsorted(tau_edges, tau, side="right")] += 1, bit set;
                                      then prev = cur.
           A started buoy ends at its first invalid sample, so it was valid at t-1: trans needs no flag.
Stats.     Per window, all i8 and exact.  Events (they sum over windows): n_start, n_end (R+1), trans (R+1, R+1),
           n_arrive, sum_tau, sum_tau2 (R+1, R) (destinations 1..R), hist_tau (R+1, R, len(tau_edges)+1); window w
           holds the events of sample w+1, window 0 also the starts of sample 0.  Snapshot (does not sum): count
           (R+1, R+1) at sample w+1; sample 0's snapshot is diag(n_start), so sample 0 adds no count.  tau_edges: 1..512
           f8 edges in samples; default 1, 2, 4, ... 2^16, so bin 0 is empty.

`sample` is vectorised over buoys; `sample_loop` is a plain per-buoy loop that the tests hold it to.  A state is
(nP, 5) i8 columns [status, src, prev, start, visited].
"""
import numpy as np

DEFAULT_TAU_EDGES = np.array([2.0 ** k for k in range(17)])                        # 1, 2, 4, ... 65536 samples
NAMES = ("n_start", "n_end", "count", "trans", "n_arrive", "sum_tau", "sum_tau2", "hist_tau")


def empty_stats(R, ntau):
    R1 = R + 1
    return dict(n_start=np.zeros(R1, np.int64), n_end=np.zeros(R1, np.int64), count=np.zeros((R1, R1), np.int64),
                trans=np.zeros((R1, R1), np.int64), n_arrive=np.zeros((R1, R), np.int64),
                sum_tau=np.zeros((R1, R), np.int64), sum_tau2=np.zeros((R1, R), np.int64),
                hist_tau=np.zeros((R1, R, ntau + 1), np.int64))


def add_events(a, b):
    """a's and b's events summed, b's count snapshot."""
    return {k: b[k] if k == "count" else a[k] + b[k] for k in a}


def new_state(nP):
    return np.zeros((nP, 5), np.int64)


def regions(labels, R, cells):
    """(nP,) i8 region of each cell (jT bit 31 stripped) and (nP,) bool: the cell lies in the interior."""
    labels = np.asarray(labels)
    Nj, Ni = labels.shape
    c = np.asarray(cells).astype(np.int64)
    jT, iT = (c[:, 0] & 0x7fffffff), c[:, 1]
    inside = (jT >= 1) & (jT <= Nj - 2) & (iT >= 1) & (iT <= Ni - 2)
    lab = np.zeros(c.shape[0], np.int64)
    lab[inside] = labels[jT[inside], iT[inside]]
    lab[lab > R] = 0
    return lab, inside


def sample(state, labels, R, cells, m, t, tau_edges=DEFAULT_TAU_EDGES):
    """One sample t of every buoy: -> (new state, the stats of its events and its count snapshot)."""
    tau_edges = np.asarray(tau_edges, np.float64)
    R1, NB = R + 1, tau_edges.size + 1
    st = empty_stats(R, tau_edges.size)
    S = np.array(state, np.int64, copy=True)
    if t == 0:
        S[:] = 0
    cur, inside = regions(labels, R, cells)
    valid = inside & (np.asarray(m) != 0)
    status, src, prev, start, vis = (S[:, k] for k in range(5))
    bit = np.where(cur >= 1, np.left_shift(1, np.maximum(cur, 1) - 1), 0)
    go = (status == 0) & valid
    end = (status == 1) & ~valid
    cont = (status == 1) & valid
    st["n_start"] += np.bincount(cur[go], minlength=R1)
    st["n_end"] += np.bincount(src[end], minlength=R1)
    if t > 0:
        occ = np.where(go, cur * R1 + cur, src * R1 + cur)[go | cont]
        st["count"] += np.bincount(occ, minlength=R1 * R1).reshape(R1, R1)
    st["trans"] += np.bincount((prev * R1 + cur)[cont], minlength=R1 * R1).reshape(R1, R1)
    arr = cont & (cur >= 1) & ((vis & bit) == 0)
    tau = t - start[arr]
    key = src[arr] * R + cur[arr] - 1
    st["n_arrive"] += np.bincount(key, minlength=R1 * R).reshape(R1, R)
    st["sum_tau"] += _isum(key, tau, R1 * R).reshape(R1, R)
    st["sum_tau2"] += _isum(key, tau * tau, R1 * R).reshape(R1, R)
    b = np.searchsorted(tau_edges, tau.astype(np.float64), side="right")
    st["hist_tau"] += np.bincount(key * NB + b, minlength=R1 * R * NB).reshape(R1, R, NB)
    S[go, 0], S[go, 1], S[go, 2], S[go, 3], S[go, 4] = 1, cur[go], cur[go], t, bit[go]
    S[end, 0] = 2
    S[arr, 4] |= bit[arr]
    S[cont, 2] = cur[cont]
    return S, st


def _isum(key, v, n):
    """Exact integer sums of v per key (np.bincount's weights are f8)."""
    out = np.zeros(n, np.int64)
    np.add.at(out, key, np.asarray(v, np.int64))
    return out


def sample_loop(state, labels, R, cells, m, t, tau_edges=DEFAULT_TAU_EDGES):
    """`sample` as a plain loop over buoys, one statement per rule."""
    labels = np.asarray(labels)
    Nj, Ni = labels.shape
    edges = [float(e) for e in tau_edges]
    st = empty_stats(R, len(edges))
    out = np.array(state, np.int64, copy=True)
    if t == 0:
        out[:] = 0
    for p in range(out.shape[0]):
        status, src, prev, start, vis = (int(v) for v in out[p])
        jT, iT = int(cells[p][0]) & 0x7fffffff, int(cells[p][1])
        ok = int(m[p]) != 0 and 1 <= jT <= Nj - 2 and 1 <= iT <= Ni - 2
        cur = int(labels[jT, iT]) if ok else 0
        if cur > R:
            cur = 0
        if status == 0:
            if ok:
                status, src, prev, start, vis = 1, cur, cur, t, (1 << (cur - 1)) if cur >= 1 else 0
                st["n_start"][src] += 1
                if t > 0:
                    st["count"][src, cur] += 1
        elif status == 1:
            if not ok:
                status = 2
                st["n_end"][src] += 1
            else:
                st["trans"][prev, cur] += 1
                st["count"][src, cur] += 1
                if cur >= 1 and not vis >> (cur - 1) & 1:
                    tau = t - start
                    st["n_arrive"][src, cur - 1] += 1
                    st["sum_tau"][src, cur - 1] += tau
                    st["sum_tau2"][src, cur - 1] += tau * tau
                    st["hist_tau"][src, cur - 1, sum(1 for e in edges if e <= tau)] += 1
                    vis |= 1 << (cur - 1)
                prev = cur
        out[p] = status, src, prev, start, vis
    return out, st


def run(cells, masks, labels, R, tau_edges=DEFAULT_TAU_EDGES, every=1, step=sample):
    """The samples cells[s*every], masks[s*every], s = 0 .. S (S = (len(cells)-1) // every): -> (states (S, nP, 5) after
    each window, the S windows' stats); window w holds sample w+1, window 0 also the starts of sample 0."""
    S = (len(cells) - 1) // every
    nP = np.asarray(cells[0]).shape[0]
    state, first = step(new_state(nP), labels, R, cells[0], masks[0], 0, tau_edges)
    states, wins = [], []
    for s in range(1, S + 1):
        state, st = step(state, labels, R, cells[s * every], masks[s * every], s, tau_edges)
        if s == 1:
            st = add_events(first, st)
        states.append(state)
        wins.append(st)
    return np.array(states).reshape(S, nP, 5), wins
