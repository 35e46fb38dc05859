"""The host side of locreg_relocalise_staged's contract, shared by its CPU and GPU tests: the selection rule of the cut
and the chain of plain locreg_relocalise calls that a staged call must reproduce bit for bit."""
import numpy as np


def pack_order_scores(scores):
    """The float32 score locreg_pack_score ranks by: NaN and negative scores count as +inf."""
    f = np.asarray(scores, np.float64).astype(np.float32)
    return np.where(np.isnan(f) | (f < 0), np.float32(np.inf), f)


def survivors(scores, alive, keep):
    """The min(keep, len(alive)) hypotheses of `alive` (original indices, ascending; scores aligned with them) with the
    smallest (float32 score, index), returned in ascending original index."""
    alive = np.asarray(alive, np.int64)
    order = np.lexsort((alive, pack_order_scores(scores)))  # primary key last: score, then index
    return np.sort(alive[order[:min(int(keep), len(alive))]])


def chain(handle_for, cloud, hyp, trips, keep):
    """The contract as a host chain: round r is locreg_relocalise (handle_for(trips[r]), a handle whose max_iteration is
    trips[r]) over that round's alive hypotheses, from the poses the previous round left; the cut keeps survivors().
    Returns (best_idx, scores, poses, rounds, alive of every round)."""
    hyp = np.asarray(hyp, np.float64)
    n = len(hyp)
    scores, poses, rounds = np.full(n, np.nan), hyp.copy(), np.zeros(n, np.int32)
    alive = np.arange(n)
    history = []
    best = -1
    for r, t in enumerate(trips):
        history.append(alive)
        _, bi, _, sc, ps = handle_for(int(t)).Relocalise(cloud, poses[alive], want_all=True)
        scores[alive], poses[alive], rounds[alive] = sc, ps, r + 1
        if r + 1 < len(trips):
            alive = survivors(sc, alive, keep[r])
        else:
            best = int(alive[bi])  # positions are in ascending original index: lowest index on ties
    return best, scores, poses, rounds, history
