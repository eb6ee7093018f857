"""Host side of the Blackwell-native Harmony engine.

Mirrors the public interface of slowkow/harmonypy (``run_harmony`` / ``Harmony``,
harmonypy/harmony.py:49-215 and :218-569): same arguments, same attributes, same
convergence logic, same result layout -- but every pass over the cells is a CUDA kernel
behind the C ABI in ``include/harmony_b200.h``.  What stays in Python is exactly what is
host logic in the reference too: argument normalisation, the sklearn k-means
initialisation, the permutation stream, the loop / convergence bookkeeping.

Differences a caller can observe (all additive):
  * batch membership is kept as integer level codes, not a dense one-hot ``Phi``
    (the ``Phi`` / ``Phi_moe`` properties materialise it on demand);
  * extra keyword arguments ``init_centroids``, ``perm_mode``, ``comm``, ``engine_options``;
  * ``device`` must be a CUDA device (there is no CPU path in this package).
"""
from __future__ import annotations

import logging
from dataclasses import dataclass

import numpy as np
import pandas as pd

from . import _cabi

logger = logging.getLogger("harmonypy_b200")
logger.setLevel(logging.DEBUG)
if not logger.handlers:
    _h = logging.StreamHandler()
    _h.setLevel(logging.DEBUG)
    _h.setFormatter(logging.Formatter("%(asctime)s - %(name)s - %(levelname)s - %(message)s"))
    logger.addHandler(_h)


# ----------------------------------------------------------------------------------------------
# front end (harmony.py:116-173)

@dataclass
class Problem:
    """Normalised inputs of one Harmony run (what harmony.py:116-173 computes)."""
    Z: np.ndarray                 # N x d float32, cells first
    codes: np.ndarray             # V x N int32 level codes
    levels: np.ndarray            # V int32 number of levels per covariate
    level_names: list             # B names in one-hot row order (pd.get_dummies column order)
    Pr_b: np.ndarray              # B float32
    theta: np.ndarray             # B float32
    lamb: np.ndarray              # B+1 float32 (or length-1 zeros when estimated, harmony.py:156)
    lambda_estimation: bool
    sigma: np.ndarray             # K float32
    K: int
    # Pre-sharded input (multi-GPU, large N): Z / codes hold only cells
    # [shard_lo, shard_lo + len(Z)) of n_global cells; Pr_b must be the GLOBAL proportions.
    n_global: int = None
    shard_lo: int = None

    @property
    def N(self):
        return self.Z.shape[0] if self.n_global is None else int(self.n_global)

    @property
    def d(self):
        return self.Z.shape[1]

    @property
    def B(self):
        return int(self.levels.sum())


def _level_codes(meta_data, vars_use):
    """Integer codes per covariate with the level order of ``pd.get_dummies`` (harmony.py:133):
    covariates in the given order, levels sorted (category order for categoricals)."""
    codes, levels, names = [], [], []
    for v in vars_use:
        col = meta_data[v]
        if pd.api.types.is_numeric_dtype(col.dtype) and not isinstance(col.dtype, pd.CategoricalDtype):
            # the reference fails at `describe().loc['unique']` (harmony.py:134) for numeric columns
            raise KeyError("unique")
        cat = pd.Categorical(col)
        if isinstance(col.dtype, pd.CategoricalDtype):
            cat = col.cat.remove_unused_categories().values
        if (cat.codes < 0).any():
            raise ValueError(f"batch covariate {v!r} contains missing values")
        codes.append(np.asarray(cat.codes, dtype=np.int32))
        levels.append(len(cat.categories))
        names.extend(f"{v}_{c}" for c in cat.categories)
    return np.stack(codes), np.asarray(levels, dtype=np.int32), names


def prepare_problem(data_mat, meta_data, vars_use, theta=None, lamb=None, sigma=0.1, nclust=None, tau=0):
    """Argument normalisation of run_harmony (harmony.py:116-173), one-hot replaced by codes."""
    N = meta_data.shape[0]
    if hasattr(data_mat, "values"):
        data_mat = data_mat.values
    data_mat = np.asarray(data_mat)
    if data_mat.shape[1] != N:                                   # :117-118  (d x N wanted there)
        data_mat = data_mat.T
    assert data_mat.shape[1] == N, "data_mat and meta_data do not have the same number of cells"   # :120
    Z = np.ascontiguousarray(data_mat.T, dtype=np.float32)       # cells first for the engine

    if nclust is None:                                            # :123-124
        nclust = int(min(round(N / 30.0), 100))
    nclust = int(nclust)
    if np.ndim(sigma) == 0:                                       # :126-127
        sigma = np.repeat(float(sigma), nclust)
    sigma = np.asarray(sigma, dtype=np.float32)
    assert sigma.shape == (nclust,), "sigma must be a scalar or have one entry per cluster"

    if isinstance(vars_use, str):                                 # :129-130
        vars_use = [vars_use]
    vars_use = list(vars_use)
    codes, phi_n, names = _level_codes(meta_data, vars_use)      # :133-134
    B = int(phi_n.sum())

    def per_level(x, what):
        """scalar | per covariate | per level -> per level (harmony.py:137-147, :157-166)."""
        if isinstance(x, (float, int, np.floating, np.integer)):
            return np.repeat([x] * len(phi_n), phi_n).astype(np.float32)
        x = list(x) if not isinstance(x, np.ndarray) else x
        if len(x) == len(phi_n):
            return np.repeat(np.asarray(x, dtype=np.float32), phi_n).astype(np.float32)
        return np.asarray(x, dtype=np.float32)

    theta = per_level(2 if theta is None else theta, "theta")
    assert len(theta) == B, "each batch variable must have a theta"      # :146-147

    lambda_estimation = False
    if lamb is None:                                              # :151-153
        lamb = np.insert(per_level(1, "lamb"), 0, 0).astype(np.float32)
    elif isinstance(lamb, (float, int, np.floating, np.integer)) and lamb == -1:      # :154-156
        lambda_estimation = True
        lamb = np.zeros(1, dtype=np.float32)
    else:                                                         # :157-166
        lamb = per_level(lamb, "lamb")
        if len(lamb) == B:
            lamb = np.insert(lamb, 0, 0).astype(np.float32)
        assert len(lamb) == B + 1, "each batch variable must have a lambda"

    N_b = np.concatenate([np.bincount(codes[v], minlength=int(phi_n[v])) for v in range(len(phi_n))]).astype(np.float64)
    Pr_b = (N_b / N).astype(np.float32)                           # :169-170
    if tau > 0:                                                   # :172-173
        theta = (theta * (1 - np.exp(-(N_b / (nclust * tau)) ** 2))).astype(np.float32)
    return Problem(Z=Z, codes=codes, levels=phi_n, level_names=names, Pr_b=Pr_b, theta=theta.astype(np.float32),
                   lamb=lamb, lambda_estimation=lambda_estimation, sigma=sigma, K=nclust), vars_use


# Shape limits of the CUDA engine (include/harmony_b200.h, "Limits"); the reference has none, so a run that exceeds
# one fails here with the reason instead of deep inside the library.
ENGINE_LIMITS = dict(max_d=128, max_K=256, max_covariates=8, max_blocks=250)


def check_engine_limits(problem, block_size):
    lim = ENGINE_LIMITS
    if problem.d > lim["max_d"]:
        raise ValueError(f"harmonypy_b200 supports at most {lim['max_d']} PCs (got {problem.d})")
    if not 2 <= problem.K <= lim["max_K"]:
        raise ValueError(f"harmonypy_b200 supports 2..{lim['max_K']} clusters (nclust = {problem.K})")
    if len(problem.levels) > lim["max_covariates"]:
        raise ValueError(f"harmonypy_b200 supports at most {lim['max_covariates']} batch covariates (got {len(problem.levels)})")
    if not 0 < block_size <= 1 or int(np.ceil(1.0 / block_size)) > lim["max_blocks"]:
        raise ValueError(f"block_size must be in [{1.0 / lim['max_blocks']}, 1] (got {block_size})")


def get_device(device=None):
    """harmony.py:35-46, restricted to CUDA: returns the CUDA device index."""
    if device is None:
        return 0
    s = str(device)
    if s in ("cuda", "gpu"):
        return 0
    if s.startswith("cuda:"):
        return int(s.split(":")[1])
    if isinstance(device, (int, np.integer)):
        return int(device)
    raise ValueError(f"harmonypy_b200 runs on CUDA devices only (got device={device!r})")


# ----------------------------------------------------------------------------------------------
# multi-GPU plumbing (cells sharded contiguously over ranks, SURVEY.md section 8e)

class Comm:
    """Sum all-reduce over the ranks of a torch.distributed process group."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.backend = dist.get_backend(group)

    def shard(self, N):
        lo = N * self.rank // self.world
        hi = N * (self.rank + 1) // self.world
        return lo, hi

    def allreduce_numpy(self, arr):
        """In-place sum of a host array (gloo); used by CPU test engines."""
        import torch
        t = torch.from_numpy(arr)
        self.dist.all_reduce(t, group=self.group)
        return arr

    def allreduce_devptr(self, ptr, count, dtype, stream):
        """In-place sum of `count` elements at device pointer `ptr` (nccl), ordered on the engine's `stream`."""
        import torch

        class _Mem:
            pass
        m = _Mem()
        m.__cuda_array_interface__ = {"shape": (int(count),), "typestr": "<f4" if dtype == 0 else "<f8",
                                      "data": (int(ptr), False), "version": 2}
        t = torch.as_tensor(m, device="cuda")
        # the engine's kernels run on `stream`: the collective must be enqueued there too, whatever stream the
        # caller has made current in the meantime
        with torch.cuda.stream(torch.cuda.ExternalStream(int(stream)) if stream else torch.cuda.current_stream()):
            self.dist.all_reduce(t, group=self.group)
        return 0

    def broadcast_array(self, arr, src=0):
        import torch
        t = torch.from_numpy(np.ascontiguousarray(arr))
        if self.backend == "nccl":
            t = t.cuda()
        self.dist.broadcast(t, src=src, group=self.group)
        return t.cpu().numpy()

    def gather_rows(self, local, N, lo=None):
        """All ranks' row blocks -> the full matrix on every rank.  lo: first global row of this rank's block
        (default: the even split of shard(); pre-sharded inputs pass their own offset)."""
        import torch
        out = np.zeros((N,) + local.shape[1:], dtype=local.dtype)
        if lo is None:
            lo = self.shard(N)[0]
        out[lo:lo + local.shape[0]] = local
        t = torch.from_numpy(out)
        if self.backend == "nccl":
            t = t.cuda()
        self.dist.all_reduce(t, group=self.group)
        return t.cpu().numpy()


def _cuda_engine_factory(problem, lo, hi, device_index, comm, options):
    eng = _cabi.Engine(device_index, hi - lo, problem.N, lo, problem.d, problem.K, problem.levels)
    options = dict(options or {})
    eng.want_fused = bool(options.pop("fused", 1))       # host-side switch, not a library option
    for k, v in options.items():
        eng.set_option(k, v)
    if comm is not None and comm.world > 1:
        import torch
        torch.cuda.set_device(device_index)
        eng.set_stream(torch.cuda.current_stream().cuda_stream)
        eng.set_allreduce(comm.allreduce_devptr)
        eng.set_rank(comm.rank, comm.world)
    return eng


# ----------------------------------------------------------------------------------------------

def run_harmony(data_mat, meta_data, vars_use, theta=None, lamb=None, sigma=0.1, nclust=None, tau=0,
                block_size=0.05, max_iter_harmony=10, max_iter_kmeans=20, epsilon_cluster=1e-5,
                epsilon_harmony=1e-4, alpha=0.2, verbose=True, random_state=0, device=None, *,
                init_centroids=None, perm_mode="reference", comm=None, engine_options=None,
                engine_factory=None, init_mode="sklearn"):
    """Run Harmony batch-effect correction on a B200 (drop-in for harmonypy.run_harmony).

    Parameters are those of harmonypy/harmony.py:49-67.  Additional keyword-only arguments:

    init_centroids : (K, d) array, optional
        Skip the sklearn k-means initialisation (harmony.py:369-373) and start from these.
    perm_mode : "reference" | "device"
        "reference": one ``torch.randperm(N)`` per update_R from the CPU generator seeded with
        ``random_state`` (harmony.py:200, :471) -- bit-identical block membership to the
        reference's CPU path.  "device": a keyed pseudo-random permutation evaluated on the GPU
        (no host work per round; use for large N).
    comm : torch.distributed process group (or True for the default group), optional
        Shard the cells over the ranks of the group (one process per GPU).
    init_mode : "sklearn" | "device"
        Where the k-means initialisation of harmony.py:369-373 runs when ``init_centroids`` is not given.
        "sklearn" (default): exactly the reference's call.  "device": k-means++ / Lloyd on the GPU
        (``hmy_kmeans_init``; same algorithm, its own random stream keyed by ``random_state``) -- for sizes
        where sklearn dominates the wall time.  With ``comm`` every rank initialises from its own cells (also
        pre-sharded input, where no rank holds all cells): the ranks exchange one slot per k-means++ step and the
        Lloyd sums, pick exactly the seeds one GPU holding all cells would, and all start from the same centroids.
    """
    problem, vars_use = prepare_problem(data_mat, meta_data, vars_use, theta, lamb, sigma, nclust, tau)
    dev = get_device(device)
    if verbose:
        logger.info(f"Running Harmony (sm_100a CUDA engine on cuda:{dev})")
        logger.info("  Parameters:")
        logger.info(f"    max_iter_harmony: {max_iter_harmony}")
        logger.info(f"    max_iter_kmeans: {max_iter_kmeans}")
        logger.info(f"    epsilon_cluster: {epsilon_cluster}")
        logger.info(f"    epsilon_harmony: {epsilon_harmony}")
        logger.info(f"    nclust: {problem.K}")
        logger.info(f"    block_size: {block_size}")
        logger.info(f"    lamb: dynamic (alpha={alpha})" if problem.lambda_estimation else f"    lamb: {problem.lamb[1:]}")
        logger.info(f"    theta: {problem.theta}")
        logger.info(f"    sigma: {problem.sigma[:5]}..." if problem.K > 5 else f"    sigma: {problem.sigma}")
        logger.info(f"    random_state: {random_state}")
        logger.info(f"  Data: {problem.d} PCs x {problem.N} cells")
        logger.info(f"  Batch variables: {vars_use}")
    np.random.seed(random_state)                                  # harmony.py:199
    return Harmony(problem, alpha, max_iter_harmony, max_iter_kmeans, epsilon_cluster, epsilon_harmony,
                   block_size, verbose, random_state, dev, init_centroids=init_centroids, perm_mode=perm_mode,
                   comm=comm, engine_options=engine_options, engine_factory=engine_factory, init_mode=init_mode)


class Harmony:
    """State object of one run; constructing it runs the algorithm (harmony.py:224-282)."""

    def __init__(self, problem, alpha, max_iter_harmony, max_iter_kmeans, epsilon_kmeans, epsilon_harmony,
                 block_size, verbose, random_state, device, init_centroids=None, perm_mode="reference",
                 comm=None, engine_options=None, engine_factory=None, run=True, init_mode="sklearn"):
        self.problem = problem
        self.device = device
        self.N, self.B, self.d, self.K = problem.N, problem.B, problem.d, problem.K
        self.window_size = 3                                      # harmony.py:258
        self.epsilon_kmeans = epsilon_kmeans
        self.epsilon_harmony = epsilon_harmony
        self.alpha = alpha
        self.lambda_estimation = problem.lambda_estimation
        self.block_size = block_size
        self.max_iter_harmony = max_iter_harmony
        self.max_iter_kmeans = max_iter_kmeans
        self.verbose = verbose
        self.random_state = random_state
        if perm_mode not in ("reference", "device"):
            raise ValueError("perm_mode must be 'reference' or 'device'")
        self.perm_mode = perm_mode
        if init_mode not in ("sklearn", "device"):
            raise ValueError("init_mode must be 'sklearn' or 'device'")
        self.init_mode = init_mode
        self._perm_gen = None

        if comm is True:
            comm = Comm(None)
        elif comm is not None and not isinstance(comm, Comm):
            comm = Comm(comm)
        self.comm = comm
        if problem.shard_lo is not None:
            self._lo, self._hi = int(problem.shard_lo), int(problem.shard_lo) + problem.Z.shape[0]
        else:
            self._lo, self._hi = (0, self.N) if comm is None else comm.shard(self.N)

        self.objective_harmony = []
        self.objective_kmeans = []
        self.objective_kmeans_dist = []
        self.objective_kmeans_entropy = []
        self.objective_kmeans_cross = []
        self.kmeans_rounds = []
        self._last_obj = None

        if engine_factory is None:
            check_engine_limits(problem, block_size)
        factory = engine_factory or _cuda_engine_factory
        self._engine = factory(problem, self._lo, self._hi, device, comm, engine_options)
        if perm_mode == "device" and "seed" not in (engine_options or {}):
            # the device-side permutation follows random_state like the host stream does (harmony.py:200);
            # random_state = 0 is the library's default key
            self._engine.set_option("seed", int(random_state))
        lamb = problem.lamb if not problem.lambda_estimation else None
        self._engine.set_params(problem.Pr_b, problem.theta, problem.sigma, lamb, problem.lambda_estimation,
                                alpha, block_size)
        if comm is not None and comm.world > 1 and getattr(self._engine, "want_fused", False):
            # fused mode: the round kernel exchanges its K x B tables itself through peer-mapped
            # memory; only the 64-byte IPC handles travel through torch.distributed
            try:
                mine = self._engine.comm_export()
            except _cabi.EngineError:
                mine = None                               # e.g. d > 64: stay in staged mode
            handles = [None] * comm.world
            comm.dist.all_gather_object(handles, mine, group=comm.group)
            if all(h is not None for h in handles):
                self._engine.comm_attach(comm.rank, comm.world, handles)
            comm.dist.barrier(group=comm.group)
        self.allocate_buffers()
        # Engines that run one round ahead keep R in tensor memory / registers and store it to HBM only when asked:
        # inside cluster() that is after the rounds the loop can stop at (harmony.py:455-458); stages called one by
        # one (init_cluster, kmeans_round, update_R) always store it.
        self._lazy_R = bool(getattr(self._engine, "lookahead", False))
        if run:
            rounds_follow = self.max_iter_harmony > 0 and self.max_iter_kmeans > 0
            if self._lazy_R and rounds_follow:
                self._engine.set_option("write_r", 0)          # nothing reads R between init and the first round
            self.init_cluster(random_state, init_centroids)
            if self._lazy_R:
                self._engine.set_option("write_r", 1)
            self.harmonize(self.max_iter_harmony, self.verbose)

    # ------------------------------------------------------------------ gathered reads
    def _cells(self, which):
        local = self._engine.get(which)
        if self.comm is None or self.comm.world == 1:
            return local
        return self.comm.gather_rows(local, self.N, self._lo)

    @property
    def Z_corr(self):
        """Corrected embedding (N x d)  -- harmony.py:288-291."""
        return self._cells(_cabi.Z_CORR)

    @property
    def Z_orig(self):
        """Input embedding (N x d)  -- harmony.py:293-296."""
        return self._cells(_cabi.Z_ORIG)

    @property
    def Z_cos(self):
        """Unit-length embedding used for clustering (N x d)  -- harmony.py:298-301."""
        return self._cells(_cabi.Z_COS)

    @property
    def R(self):
        """Soft assignments (N x K)  -- harmony.py:303-306."""
        return self._cells(_cabi.R)

    @property
    def Y(self):
        """Centroids (d x K)  -- harmony.py:308-311."""
        return np.ascontiguousarray(self._engine.get(_cabi.Y).T)

    @property
    def O(self):
        """Observed batch-by-cluster mass (K x B)  -- harmony.py:313-316."""
        return self._engine.get(_cabi.O).astype(np.float32)

    @property
    def E(self):
        """Expected batch-by-cluster mass (K x B)  -- harmony.py:318-321."""
        return self._engine.get(_cabi.E).astype(np.float32)

    @property
    def Phi(self):
        """One-hot batch indicators (N x B), materialised on demand  -- harmony.py:323-326."""
        p = self.problem
        n_loc = p.codes.shape[1]
        out = np.zeros((n_loc, self.B), dtype=np.float32)
        off = 0
        rows = np.arange(n_loc)
        for v in range(len(p.levels)):
            out[rows, off + p.codes[v]] = 1
            off += int(p.levels[v])
        if n_loc != self.N:                                       # pre-sharded input: this rank holds its own rows only
            if self.comm is None:
                raise ValueError("Phi: the problem holds a shard of the cells but no communicator was given")
            return self.comm.gather_rows(out, self.N, self._lo)
        return out

    @property
    def Phi_moe(self):
        """[1 | Phi] (N x (B+1))  -- harmony.py:328-331."""
        return np.hstack([np.ones((self.N, 1), dtype=np.float32), self.Phi])

    @property
    def Pr_b(self):
        return self.problem.Pr_b

    @property
    def theta(self):
        return self.problem.theta

    @property
    def sigma(self):
        return self.problem.sigma

    @property
    def lamb(self):
        return self.problem.lamb

    def result(self):
        """harmony.py:353-355."""
        return self.Z_corr

    def result_local(self):
        """This rank's rows of Z_corr (cells [lo, hi) of the global order), no gather."""
        return self._engine.get(_cabi.Z_CORR)

    # ------------------------------------------------------------------ stages
    def allocate_buffers(self):
        """Upload this rank's cells; the engine owns all device buffers (harmony.py:357-364)."""
        p = self.problem
        if p.shard_lo is not None:
            self._engine.set_data(p.Z, p.codes)
        else:
            self._engine.set_data(p.Z[self._lo:self._hi], p.codes[:, self._lo:self._hi])

    def _record_objective(self, triple):
        """Bookkeeping of compute_objective (harmony.py:396, :413-417)."""
        c0 = 2000.0 / self.N
        err, ent, cross = triple
        self._last_obj = triple
        self.objective_kmeans.append((err + ent + cross) * c0)
        self.objective_kmeans_dist.append(err * c0)
        self.objective_kmeans_entropy.append(ent * c0)
        self.objective_kmeans_cross.append(cross * c0)

    def compute_objective(self):
        """The objective is a by-product of every round on the device; calling this again
        re-records the last value (harmony.py:394-417 recomputes it from the K x N matrices)."""
        if self._last_obj is None:
            raise RuntimeError("no objective yet: call init_cluster first")
        self._record_objective(self._last_obj)

    def init_cluster(self, random_state, init_centroids=None):
        """harmony.py:366-392.  k-means++ / Lloyd initialisation stays with sklearn on the host
        exactly as in the reference (or runs on the device with init_mode="device"; with sharded cells
        that call is collective: every rank makes it); everything after it runs on the device."""
        if init_centroids is None and self.init_mode == "device":
            if self.verbose:
                logger.info("Computing initial centroids on the device (k-means++ / Lloyd)...")
            init_centroids, self.kmeans_init_info = self._engine.kmeans_init(int(random_state), max_iter=25, tol=1e-4)
        if init_centroids is None:
            if self.comm is None or self.comm.rank == 0:
                from sklearn.cluster import KMeans
                if self.problem.shard_lo is not None:
                    raise ValueError("pre-sharded input needs init_centroids or init_mode='device' "
                                     "(no rank holds all cells)")
                Z = self.problem.Z
                Z_cos = Z / np.linalg.norm(Z, axis=1, keepdims=True)
                if self.verbose:
                    logger.info("Computing initial centroids with sklearn.KMeans...")
                model = KMeans(n_clusters=self.K, init="k-means++", n_init=1, max_iter=25,
                               random_state=random_state)           # harmony.py:370-371
                model.fit(Z_cos)
                init_centroids = model.cluster_centers_.astype(np.float32)
                if self.verbose:
                    logger.info("KMeans initialization complete.")
            else:
                init_centroids = np.zeros((self.K, self.d), dtype=np.float32)
            if self.comm is not None and self.comm.world > 1:
                init_centroids = self.comm.broadcast_array(init_centroids, src=0)
        Y0 = np.asarray(init_centroids, dtype=np.float32)
        if Y0.shape == (self.d, self.K) and self.d != self.K:
            Y0 = Y0.T
        assert Y0.shape == (self.K, self.d), "init_centroids must be K x d"
        if getattr(self._engine, "lookahead", False) and self.perm_mode == "reference":
            # the init assignment already groups its sums by the FIRST round's blocks: hand over that permutation
            # (first draw of the stream, harmony.py:471); every round call then carries the next round's
            self._engine.queue_perm(self._next_perm())
        self._record_objective(self._engine.init_from_centroids(Y0))
        self.objective_harmony.append(self.objective_kmeans[-1])  # harmony.py:392

    def _next_perm(self):
        """The reference's permutation stream (harmony.py:200 + :471), or None in device mode."""
        if self.perm_mode == "device":
            return None
        import torch
        if self._perm_gen is None:
            self._perm_gen = torch.Generator(device="cpu")
            self._perm_gen.manual_seed(int(self.random_state))
        return torch.randperm(self.N, generator=self._perm_gen).numpy()

    def kmeans_round(self):
        """One iteration of the body of cluster() (harmony.py:443-453), fused on the device."""
        self._record_objective(self._engine.kmeans_round(self._next_perm()))

    def update_R(self):
        """harmony.py:464-513.  The device round fuses the centroid update, the distances, the
        blockwise R update and the objective; calling update_R alone runs that fused round
        without recording the objective."""
        self._last_obj = self._engine.kmeans_round(self._next_perm())

    def cluster(self):
        """harmony.py:437-462."""
        rounds = 0
        lazy = getattr(self, "_lazy_R", False)
        pending = 0            # rounds enqueued whose objective has not been read yet
        for i in range(self.max_iter_kmeans):
            can_stop = i > self.window_size or i == self.max_iter_kmeans - 1
            if lazy:      # R must be in HBM after every round the loop can end with
                self._engine.set_option("write_r", int(can_stop))
            if lazy and not can_stop:
                # the convergence rule cannot fire after this round (harmony.py:455): no host round trip, the
                # objective is read together with the next one that matters
                self._engine.kmeans_round(self._next_perm(), wait=False)
                pending += 1
            else:
                if pending:
                    self._engine.kmeans_round(self._next_perm(), wait=False)
                    for o in self._engine.objectives(pending + 1):
                        self._record_objective(o)
                    pending = 0
                else:
                    self.kmeans_round()
            rounds = i + 1
            if i > self.window_size and self.check_convergence(0):    # :455-458
                break
        if lazy:
            self._engine.set_option("write_r", 1)
        self.kmeans_rounds.append(rounds)                              # :461
        self.objective_harmony.append(self.objective_kmeans[-1])       # :462

    def check_convergence(self, i_type):
        """harmony.py:515-533 (python floats, unchanged)."""
        if i_type == 0:
            if len(self.objective_kmeans) <= self.window_size + 1:
                return False
            w = self.window_size
            obj_old = sum(self.objective_kmeans[-w - 1:-1])
            obj_new = sum(self.objective_kmeans[-w:])
            return abs(obj_old - obj_new) / abs(obj_old) < self.epsilon_kmeans
        if i_type == 1:
            if len(self.objective_harmony) < 2:
                return False
            obj_old = self.objective_harmony[-2]
            obj_new = self.objective_harmony[-1]
            return (obj_old - obj_new) / abs(obj_old) < self.epsilon_harmony
        return True

    def moe_correct_ridge(self):
        """harmony.py:535-569."""
        self._engine.ridge_correct()

    def harmonize(self, iter_harmony=10, verbose=True):
        """harmony.py:419-435."""
        converged = False
        for i in range(1, iter_harmony + 1):
            if verbose:
                logger.info(f"Iteration {i} of {iter_harmony}")
            self.cluster()
            self.moe_correct_ridge()
            converged = self.check_convergence(1)
            if converged:
                if verbose:
                    logger.info(f"Converged after {i} iteration{'s' if i > 1 else ''}")
                break
        if verbose and not converged:
            logger.info("Stopped before convergence")
        return converged
