"""Leave-one-out reference of the tests, written without the library's (k + 1)-search: for every sample i a
brute-force scan over j != i orders the candidates by (d², index) — d² summed left to right without FMA, as the C
oracle and the search kernel form it — keeps the k nearest (then the ball filter), and the C oracle's existing
per-target solve (`oracle_py.krige`) kriges x_i from exactly that neighbour list. max_neighbors == 0: all j != i."""
import numpy as np


def _d2(coords, i):
    d = coords[0] - coords[0][i]
    s = d * d
    for c in coords[1:]:
        e = c - c[i]
        s = s + e * e
    return s


def krige_loo(oracle, spec, want_neighbors=False):
    """Same outputs as ``Context.krige_loo`` (slab of sample indices, neighbour lists in full-sample indices)."""
    from gskrige import ProblemSpec
    n = spec.n_samples
    first = spec.target_first
    count = n - first if spec.target_count < 0 else spec.target_count
    p = dict(spec.params)
    k, radius, nmin = p["max_neighbors"], p["ball_radius"], p["min_neighbors"]
    mean, var = np.full(count, np.nan), np.full(count, np.nan)
    nneigh = np.zeros(count, dtype=np.int32)
    idx = np.full((count, max(k, 1)), -1, dtype=np.int32) if k > 0 else None
    for t in range(count):
        i = first + t
        others = np.delete(np.arange(n), i)
        if k > 0:
            d2 = _d2(spec.coords, i)[others]
            order = others[np.lexsort((others, d2))][:k]        # ascending d², ties by index
            if radius == radius:                               # KBallSearch: dist <= radius, a prefix of the list
                order = order[np.sqrt(_d2(spec.coords, i)[order]) <= radius]
            nb = order
            idx[t, :len(nb)] = nb
        else:
            nb = others
        nneigh[t] = len(nb)
        if len(nb) == 0 or len(nb) < nmin:
            continue
        # the solve on exactly these samples, in this order: a search of all of them returns them as given (same d²,
        # ties by their position, which follows the full index)
        sub = ProblemSpec(coords=[c[nb] for c in spec.coords], values=spec.values[nb],
                          points=[c[i:i + 1] for c in spec.coords],
                          **dict(p, max_neighbors=len(nb) if k > 0 else 0, min_neighbors=1, ball_radius=float("nan")))
        m, v = oracle.krige(sub, search=oracle.SEARCH_BRUTE)
        mean[t], var[t] = m[0], v[0]
    if want_neighbors:
        return mean, var, nneigh, idx
    return mean, var
