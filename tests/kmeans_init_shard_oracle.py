"""TEST-ONLY NumPy restatement of hmy_kmeans_init on cells sharded over ranks (a context with n_local < n_global),
built on the single-process oracle of oracle/kmeans_init_oracle.py (same counter-based random numbers, same distances):
per-rank seeding passes, one slot {key, global id, row} per rank summed as an exact all-gather, Lloyd tables
[sums | counts | inertia] summed over ranks, the stop decision voted over ranks.  kmeans_init_sharded runs every rank
in lockstep in one process; kmeans_init_rank is one rank's part over a real all-reduce.  Never imported by the product."""
import numpy as np

from oracle.kmeans_init_oracle import _d2, splitmix64, uniform

# ---- cells sharded over ranks (hmy_kmeans_init on a context with n_local < n_global) ---------------------------------

def _rank_program(Z, lo, n_global, K, seed, rank, world, max_iter, tol):
    """What one rank computes, as a generator: it yields each fp64 buffer the device sums over ranks and receives the
    sum back; it returns (centres, info) of rank 0's kind (every rank computes the same).  Z: this rank's cells
    [lo, lo + len(Z)) of the n_global cells, any scale."""
    Z = np.asarray(Z, dtype=np.float32)
    Zc = Z / np.linalg.norm(Z, axis=1, keepdims=True)
    n, d = Zc.shape
    ids = np.arange(lo, lo + n, dtype=np.uint64)
    C = np.zeros((K, d), dtype=np.float32)
    seeds = np.zeros(K, dtype=np.int64)
    failed = False
    first_id = int(splitmix64(np.uint64(seed)) % np.uint64(n_global))
    mind2 = None
    for c in range(K):
        # k_kmpp_pass_sharded: this rank's winner by (key, global id); local order is global id order
        key, gid, row = np.inf, 0, None
        if c == 0:
            if lo <= first_id < lo + n:
                key, gid, row = 0.0, first_id, Zc[first_id - lo]
        else:
            d2 = _d2(Zc, C[c - 1])
            mind2 = d2 if c == 1 else np.minimum(mind2, d2)
            pos = mind2 > 0
            if pos.any():
                keys = np.full(n, np.inf, dtype=np.float32)
                keys[pos] = (-np.log(uniform(seed, c, ids[pos])) / mind2[pos].astype(np.float64)).astype(np.float32)
                i = int(np.argmin(keys))                        # first index among exact ties = least global id
                key, gid, row = float(keys[i]), lo + i, Zc[i]
        # k_kmpp_publish: one slot per rank, zeros elsewhere; the sum over ranks is an exact all-gather
        slots = np.zeros((world, 2 + d), dtype=np.float64)
        slots[rank, 0] = key
        if row is not None:
            slots[rank, 1] = gid
            slots[rank, 2:] = row
        slots = (yield slots).reshape(world, 2 + d)
        # k_kmpp_pick: least (key, global id) among the ranks that had a candidate
        cand = [w for w in range(world) if slots[w, 0] < np.inf]
        if not cand:
            failed = True                                       # the device reports it after the loop
            continue
        w = min(cand, key=lambda w: (slots[w, 0], slots[w, 1]))
        seeds[c] = int(slots[w, 1])
        C[c] = slots[w, 2:].astype(np.float32)
    if failed:
        raise ValueError("fewer distinct cells than clusters")
    it, inertia, shift = 0, 0.0, 0.0
    for it in range(1, max_iter + 1):
        # k_lloyd_assign on this rank's cells -> table [sums K d | counts K | inertia], summed over ranks
        score = (C * C).sum(axis=1, dtype=np.float32)[None, :] - np.float32(2.0) * (Zc @ C.T)
        lab = np.argmin(score, axis=1)
        sums = np.zeros((K, d), dtype=np.float64)
        np.add.at(sums, lab, Zc.astype(np.float64))
        tab = np.concatenate([sums.ravel(), np.bincount(lab, minlength=K).astype(np.float64),
                              [float((score[np.arange(n), lab].astype(np.float64) + (Zc.astype(np.float64) ** 2).sum(axis=1)).sum())]])
        tab = yield tab
        sums, cnt, inertia = tab[:K * d].reshape(K, d), tab[K * d:K * d + K], float(tab[-1])
        # k_lloyd_update_global: means over the global counts, variance from the global sums
        mean = sums.sum(axis=0) / n_global
        var = (1.0 - float(mean @ mean)) / d
        newC = C.copy()
        nz = cnt > 0
        newC[nz] = (sums[nz] / cnt[nz, None]).astype(np.float32)
        shift = float(((newC.astype(np.float64) - C.astype(np.float64)) ** 2).sum())
        C = newC
        votes = yield np.array([0.0 if shift <= tol * var else 1.0])      # another iteration while any rank votes so
        if float(votes[0]) == 0.0:
            break
    return C, dict(iterations=it, inertia=inertia, last_shift2=shift, seeds=seeds)


def kmeans_init_rank(Z, lo, n_global, K, seed, rank, world, allreduce, max_iter=25, tol=1e-4):
    """One rank's part of the sharded initialisation with a real sum all-reduce: allreduce(fp64 array) -> the sum over
    ranks (every rank must call this with the same arguments except Z / lo / rank)."""
    prog = _rank_program(Z, lo, n_global, K, seed, rank, world, max_iter, tol)
    try:
        buf = next(prog)
        while True:
            buf = prog.send(np.asarray(allreduce(np.ascontiguousarray(buf, dtype=np.float64)), dtype=np.float64))
    except StopIteration as stop:
        return stop.value


def kmeans_init_sharded(Z, K, seed, edges, max_iter=25, tol=1e-4):
    """The sharded initialisation of cells Z split at `edges` (rank r holds [edges[r], edges[r + 1])), all ranks run
    in lockstep in this process and their buffers summed in rank order.  Returns rank 0's (centres, info); with
    exact arithmetic in the exchange the seeds equal kmeans_init's."""
    Z = np.asarray(Z, dtype=np.float32)
    world = len(edges) - 1
    progs = [_rank_program(Z[edges[r]:edges[r + 1]], edges[r], Z.shape[0], K, seed, r, world, max_iter, tol)
             for r in range(world)]
    bufs = [next(p) for p in progs]
    while True:
        total = np.zeros_like(bufs[0])
        for b in bufs:
            total = total + b
        out = []
        for p in progs:
            try:
                out.append(p.send(total.copy()))
            except StopIteration as stop:
                out.append(stop)
        done = [isinstance(o, StopIteration) for o in out]
        if all(done):
            return out[0].value
        assert not any(done), "ranks left the exchange at different steps"
        bufs = out
