"""Muscle-synergy extraction on the GPU: batched NMF by multiplicative updates and by coordinate descent (EXTENSION).

API mirror of the reference's `vaf`, `SynergyRunResult` and `find_synergies`
(src/muscle_synergies/analysis.py:597-667, 670-710, 713-914).  The reference hands the
factorisation to `sklearn.decomposition.NMF(n_components=k, **kwargs)` (:862-863); here the
solver="mu", beta_loss="frobenius", init="random" case runs as ONE CUDA launch for the whole
rank sweep x restarts grid (csrc/ms_nmf.cu), in fp32, with sklearn's initialisation
(`RandomState(seed)`: H drawn first, then W - sklearn/decomposition/_nmf.py:_initialize_nmf)
generated on the host so that a run is comparable to `NMF(solver="mu", init="random",
random_state=seed)` at the same iteration count.  By default every other call (sklearn's default solver="cd",
nndsvd inits, regularisation ...) is forwarded to scikit-learn, exactly as the reference does
(analysis.py:848-864): this stage is an extension, not a replacement of scikit-learn.

`find_synergies(..., engine="gpu")` and `nmf_cd_batched` also run sklearn's default solver="cd" (shuffle=False, no
regularisation) on the GPU, in fp64 (csrc/ms_nmf_cd.cu), with init "nndsvd" / "nndsvda" computed on the device or
sklearn's "random" draws.  Parity claim, against `NMF(solver="cd")` in fp64: from the same init and at the same
iteration count (tol=0), W H, VAF (overall and per muscle) and ||X - W H||_F / ||X||_F agree to 1e-9; run to
convergence with the reference's defaults (tol=1e-6, max_iter=100 000) from the device's NNDSVD init, VAF agrees to
1e-8 and n_iter to max(3, 0.5 %).  Deviation: the device's NNDSVD uses an exact SVD where sklearn uses a randomized
one, so sklearn's random_state has no effect on it; the two inits agree to ~1e-13 relative where sklearn's randomized
SVD is itself accurate (tests/test_nmf_cd_gpu.py).

`NMFModel.transform` and `nmf_transform_batched` fit activations to fixed synergies - sklearn's `NMF.transform`, for
solver "cd" and "mu" - on the GPU in fp64 (csrc/ms_nmf_fixed.cu).  Parity claim, against sklearn's transform of the same
X with the same components_ in fp64: at the same iteration count (tol=0), W H and VAF agree to 1e-9; run to convergence
(tol=1e-6, max_iter=100 000), VAF agrees to 1e-8 and n_iter to max(3, 0.5 %) for "cd" and to one check (10) for "mu"
(tests/test_nmf_transform_gpu.py).  The result is fp64 whatever X's dtype; sklearn's is in X's dtype, fp64 for a DataFrame.

`nmf_beta_batched`, `find_synergies(engine="gpu", solver="mu", beta_loss=...)` and the transform of such a model run
sklearn's multiplicative updates for the β-divergence (beta_loss "kullback-leibler" = 1, "itakura-saito" = 0, or any
float other than 2) on the GPU in fp64 (csrc/ms_nmf_beta.cu).  Parity claim, against sklearn in fp64: from the same init
at the same iteration count (tol=0), W H, VAF and err (sklearn's reconstruction_err_, the square-rooted divergence) agree
to 1e-9; converged, VAF agrees to 1e-8 and n_iter to one check (10) (tests/test_nmf_beta_gpu.py).

`match_synergies_batched` compares synergy sets pair by pair - unit-length synergies, the optimal one-to-one pairing
of `scipy.optimize.linear_sum_assignment(maximize=True)`, the mean matched similarity - on the GPU in fp64
(csrc/ms_synmatch.cu); mean and per-synergy similarity agree with numpy + scipy to 1e-12
(tests/test_synergy_match_gpu.py).
"""
import ctypes
import functools
import threading
import warnings
from collections import OrderedDict
from dataclasses import dataclass, field
from collections.abc import Sequence
from typing import Mapping, Optional, Union

import numpy as np
import pandas

from . import _native as nat


# ---- batched solver ---------------------------------------------------------------------------------
@dataclass
class NMFBatchResult:
    ranks: np.ndarray          # (P,)
    seeds: np.ndarray          # (P,)
    W: Sequence                # P arrays (n, k_p) float32 (mu) / float64 (cd) (views of one packed array, made on access)
    H: Sequence                # P arrays (k_p, m) float32 (mu) / float64 (cd)
    n_iter: np.ndarray         # (P,)
    err: np.ndarray            # (P,)  ||X - W H||_F
    vaf: np.ndarray            # (P, m + 1): overall, then per column


def sklearn_random_init(X: np.ndarray, k: int, seed: int):
    """`_initialize_nmf(X, k, init="random", random_state=seed)` of scikit-learn."""
    avg = np.sqrt(X.mean() / k)
    rng = np.random.RandomState(seed)
    H = avg * rng.standard_normal(size=(k, X.shape[1])).astype(X.dtype, copy=False)
    W = avg * rng.standard_normal(size=(X.shape[0], k)).astype(X.dtype, copy=False)
    np.abs(H, out=H)
    np.abs(W, out=W)
    return W, H


def _unit_draws(n: int, m: int, k: int, seed: int):
    """|standard_normal| draws of sklearn's random init for (seed, k) on an n x m matrix: H first,
    then W.  The init itself is these times sqrt(X.mean() / k) (|a z| == a |z| exactly for a > 0)."""
    rng = np.random.RandomState(seed)
    H = np.abs(rng.standard_normal(size=(k, m)))
    W = np.abs(rng.standard_normal(size=(n, k)))
    return W.ravel(), H.ravel()


_unit_draws_cached = functools.lru_cache(maxsize=1024)(_unit_draws)  # gait-cycle sized problems only
_draw_cache = OrderedDict()  # (n, m, ranks, seeds, device) -> unit draws of the whole batch, on the device


def _batch_draws(torch, n, m, ranks, seeds, dev):
    with _cache_lock:
        return _batch_draws_locked(torch, n, m, ranks, seeds, dev)


def _batch_draws_locked(torch, n, m, ranks, seeds, dev):
    key = (n, m, ranks.tobytes(), seeds.tobytes(), str(dev))
    hit = _draw_cache.get(key)
    if hit is None:
        draws = _unit_draws_cached if n * m <= 1 << 16 else _unit_draws
        parts = [draws(n, m, int(k), int(s)) for k, s in zip(ranks, seeds)]
        hit = (torch.from_numpy(np.concatenate([p[0] for p in parts])).to(dev),
               torch.from_numpy(np.concatenate([p[1] for p in parts])).to(dev))
        if n * m > 1 << 16:
            return hit
        _draw_cache[key] = hit
        while len(_draw_cache) > 8:
            _draw_cache.popitem(last=False)
    else:
        _draw_cache.move_to_end(key)
    return hit


_plan_cache = OrderedDict()  # (n, m, ranks, x_index, device) -> (device problem table, kmax, device ranks, x_index, element -> problem maps)


_cache_lock = threading.Lock()  # the two caches below are process-wide; batches may be launched from several threads


def _batch_plan(torch, lib, n, m, ranks, xi, dev):
    with _cache_lock:
        return _batch_plan_locked(torch, lib, n, m, ranks, xi, dev)


def _batch_plan_locked(torch, lib, n, m, ranks, xi, dev):
    """The device-side description of a sweep (ms_nmf_plan's table, the ranks and matrix indices as int64 tensors), kept
    for the sweeps a caller repeats: a pipeline runs the same one for every trial, and each copy from pageable memory
    would wait for everything queued on the stream - the factorisation of the trial before."""
    key = (n, m, ranks.tobytes(), xi.tobytes(), str(dev))
    hit = _plan_cache.get(key)
    if hit is None:
        table = np.empty(len(ranks) * 32, dtype=np.uint8)
        kmax = int(lib.ms_nmf_plan(n, m, ranks.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                   xi.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), len(ranks), table.ctypes.data))
        nat.check(min(kmax, 0), "ms_nmf_plan")
        r64 = ranks.astype(np.int64)
        problem = np.arange(len(ranks), dtype=np.int64)
        # which problem every element of the packed W / H belongs to (the per-problem scale of the random init is
        # gathered through these; torch.repeat_interleave with device counts would wait for the device to size its output)
        hit = (torch.from_numpy(table).to(dev), kmax, torch.from_numpy(r64).to(dev), torch.from_numpy(xi.astype(np.int64)).to(dev),
               torch.from_numpy(np.repeat(problem, r64 * n)).to(dev), torch.from_numpy(np.repeat(problem, r64 * m)).to(dev))
        _plan_cache[key] = hit
        while len(_plan_cache) > 8:
            _plan_cache.popitem(last=False)
    else:
        _plan_cache.move_to_end(key)
    return hit


_pinned_pool = OrderedDict()  # nbytes -> pinned uint8 tensors not on loan (results travel through them), 32 sizes at most


def _pinned_take(torch, nbytes: int):
    free = _pinned_pool.get(nbytes)
    return free.pop() if free else torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)


def _pinned_give(buf):
    free = _pinned_pool.setdefault(int(buf.numel()), [])
    _pinned_pool.move_to_end(int(buf.numel()))
    if len(free) < 4:
        free.append(buf)
    while len(_pinned_pool) > 32:  # calls on ever new shapes must not keep pinned memory for each
        _pinned_pool.popitem(last=False)


_NEGATIVE_X = "Negative values in data passed to NMF (input X)"
_NNDSVD_DEGENERATE = ("NNDSVD initialisation divides by zero for this X: a singular value it needs is zero, or the "
                      "chosen part of a singular vector pair is empty")


class PendingNMF:
    """A batch whose kernel is queued and whose results are on their way to pinned host memory: `result()` waits
    for the copies and builds the NMFBatchResult.  Lets a caller queue the next trial's GPU work before it
    looks at this one's (pipeline.synergies_for_files)."""

    def __init__(self, torch, stream, ranks, seeds, n, m, device_arrays, keep, checks=()):
        self._ranks, self._seeds, self._n, self._m = ranks, seeds, n, m
        self._keep = keep  # inputs of the kernel: alive until the copies below have run
        self._bufs = []
        # device flags travel with the results: each (message, flag) of `checks`; the first one set is raised
        self._flags = [msg for msg, _ in checks]
        device_arrays = list(device_arrays) + [(flag != 0).to(torch.uint8).reshape(1) for _, flag in checks]
        for t in device_arrays:
            t = t.contiguous()
            buf = _pinned_take(torch, int(t.numel()) * t.element_size())
            buf.view(t.dtype).copy_(t.reshape(-1), non_blocking=True)
            self._bufs.append((buf, t.dtype, tuple(t.shape)))
            self._keep.append(t)
        self._event = torch.cuda.Event()
        self._event.record(stream)
        self._result = None

    def result(self) -> NMFBatchResult:
        if self._result is None:
            self._event.synchronize()
            out = []
            for buf, dtype, shape in self._bufs:
                out.append(buf.view(dtype).numpy().reshape(shape).copy())  # own memory: the pinned buffer goes back
                _pinned_give(buf)
            self._bufs, self._keep = [], []
            raised = [msg for msg, flag in zip(self._flags, out[len(out) - len(self._flags):]) if flag[0]]
            del out[len(out) - len(self._flags):]
            if raised:
                raise ValueError(raised[0])
            self._result = _assemble(self._ranks, self._seeds, self._n, self._m, *out)
        return self._result


class _Factors(Sequence):
    """The factors of a batch, problem after problem in one array: item p is a view, made when it is asked for (a
    trial's batch has 1280 problems and its tables read 64 of them)."""

    def __init__(self, packed: np.ndarray, offsets: np.ndarray, shapes):
        self._packed, self._offsets, self._shapes = packed, offsets, shapes

    def __len__(self):
        return len(self._offsets) - 1

    def __getitem__(self, p):
        if isinstance(p, slice):
            return [self[i] for i in range(*p.indices(len(self)))]
        p = int(p)
        if p < 0:
            p += len(self)
        if not 0 <= p < len(self):
            raise IndexError(p)
        return self._packed[self._offsets[p] : self._offsets[p + 1]].reshape(self._shapes(p))


def _assemble(ranks, seeds, n, m, Wall, Hall, n_iter, err, vafs) -> NMFBatchResult:
    w_off = np.concatenate([[0], np.cumsum(ranks.astype(np.int64) * n)])
    h_off = np.concatenate([[0], np.cumsum(ranks.astype(np.int64) * m)])
    Ws = _Factors(Wall, w_off, lambda p: (n, int(ranks[p])))
    Hs = _Factors(Hall, h_off, lambda p: (int(ranks[p]), m))
    return NMFBatchResult(ranks, seeds, Ws, Hs, n_iter, err, vafs)


# ---- what the NMF entries share: argument checks, X on the device, the initial factors, the launch outputs, the end
def _host_x(X):
    """(X as a float64 (B, n, m) numpy stack, or None for a CUDA X; the (B, n, m) shape).  Touches no device."""
    import torch

    if isinstance(X, torch.Tensor) and X.is_cuda:
        Xh, shape = None, tuple(X.shape) if X.ndim == 3 else (1,) + tuple(X.shape)
    else:
        Xh = X.detach().to("cpu", torch.float64).numpy() if isinstance(X, torch.Tensor) else np.asarray(X, dtype=np.float64)
        Xh = Xh[None] if Xh.ndim == 2 else Xh
        shape = Xh.shape
    if len(shape) != 3 or 0 in shape:
        raise ValueError("X must be a non-empty (n, m) matrix or a (B, n, m) stack")
    return Xh, shape


def _problem_arrays(ranks, seeds, x_index, shape, regime, max_iter, tol):
    """ranks (int32), seeds (int64, -1 where none is given) and x_index (int32) of a batch on an X of `shape` (B, n, m),
    after the argument checks every NMF entry shares.  Touches no device."""
    if regime not in (None, "resident", "stream"):
        raise ValueError(f"regime must be None, 'resident' or 'stream', not {regime!r}")
    if int(max_iter) < 0 or not float(tol) >= 0:
        raise ValueError("max_iter and tol must be non-negative")
    B, _, m = shape
    ranks = np.ascontiguousarray(ranks, dtype=np.int32)
    P = len(ranks)
    xi = np.zeros(P, dtype=np.int32) if x_index is None else np.ascontiguousarray(x_index, dtype=np.int32)
    seeds = np.full(P, -1, dtype=np.int64) if seeds is None else np.ascontiguousarray(seeds, dtype=np.int64)
    if P < 1 or xi.shape != (P,) or len(seeds) != P or xi.min() < 0 or xi.max() >= B:
        raise ValueError("ranks, seeds and x_index must have one entry per problem, and x_index must name a matrix of X")
    if ranks.min() < 1 or ranks.max() > 16 or m > 64:
        raise ValueError(f"ranks must be in 1..16 and X may have at most 64 columns (ranks {ranks.min()}..{ranks.max()}, "
                         f"{m} columns)")
    return ranks, seeds, xi


def _check_init(init, ranks, seeds, shape, names=("nndsvd", "nndsvda", "random"), values=False):
    """Checks `init`: a name of `names`, or one (W, H) pair per problem of the problem's shapes - with values, also
    finite, non-negative and not all zero, as scikit-learn's _check_init.  Touches no device."""
    _, n, m = shape
    if isinstance(init, str):
        if init not in names:
            raise ValueError(f"init must be {', '.join(map(repr, names))} or (W, H) pairs, not {init!r}")
        if init == "random" and (seeds < 0).any():
            raise ValueError("init='random' needs a non-negative seed per problem")
        if init != "random" and int(ranks.max()) > min(n, m):
            raise ValueError(f"init = '{init}' can only be used when n_components <= min(n_samples, n_features)")
        return
    if len(init) != len(ranks):
        raise ValueError("init must give one (W, H) pair per problem")
    for p, (W0, H0) in enumerate(init):
        if np.shape(W0) != (n, ranks[p]) or np.shape(H0) != (ranks[p], m):
            raise ValueError(f"init pair {p} must have shapes {(n, int(ranks[p]))} and {(int(ranks[p]), m)}")
        for A, whom in ((H0, "NMF (input H)"), (W0, "NMF (input W)")) if values else ():  # sklearn's order: H first
            A = np.asarray(A, dtype=np.float64)
            if not np.isfinite(A).all():
                raise ValueError(f"Input contains NaN or infinity (init pair {p}, {whom})")
            if (A < 0).any():
                raise ValueError(f"Negative values in data passed to {whom}")
            if A.max() == 0:
                raise ValueError(f"Array passed to {whom} is full of zeros.")


def _check_x(A, checks, defer=False):
    """Raises the message of the first (message, test) of `checks` whose elementwise test holds somewhere in A (a numpy
    or CUDA stack).  defer: returns the (message, device flag) pairs instead, for PendingNMF to raise - a deferred run
    does not wait for the answer here (it would wait for everything queued before it, the previous trial's
    factorisation included)."""
    if defer:
        return [(msg, test(A).any()) for msg, test in checks]
    for msg, test in checks:
        if bool(test(A).any()):
            raise ValueError(msg)
    return []


def _cuda_lib(entry):
    import torch

    lib = nat.lib()
    if not torch.cuda.is_available():
        raise nat.NativeError(f"{entry} needs a CUDA device; there is no CPU fallback")
    return lib


def _device_x(torch, X, Xh, strided, device=None, host_dtype=np.float64):
    """X as a (B, n, m) stack on the device.  A host X goes up row-major in host_dtype, to `device` (None: the current
    one).  A CUDA X stays on its device, in float64: with `strided` (the kernel reads X through its strides) a view is
    read in place - unless it is a stack whose matrices are not n * m apart, since the problem table addresses matrix b
    at b * n * m - and otherwise it becomes row-major."""
    if Xh is not None:
        dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        return torch.from_numpy(np.ascontiguousarray(Xh, dtype=host_dtype)).to(dev)
    dX = X.detach().to(torch.float64)
    dX = dX[None] if dX.ndim == 2 else dX
    B, n, m = dX.shape
    if not strided or (B > 1 and dX.stride(0) != n * m):
        dX = dX.contiguous()
    return dX


def _init_scale(torch, dX, Xh, d_ranks, d_xi):
    """sqrt(X.mean() / k) of every problem, on the device: the mean numpy takes on the host for a host X (what
    scikit-learn computes), the mean of the row-major copy for a CUDA X (the same, bit for bit, whatever its layout)."""
    if Xh is not None:
        means = torch.from_numpy(np.array([Xh[b].mean() for b in range(len(Xh))])).to(dX.device)
    else:
        means = dX.contiguous().mean(dim=(1, 2))
    return torch.sqrt(means[d_xi] / d_ranks)


def _initial_factors(torch, lib, init, dX, Xh, ranks, seeds, xi, stream):
    """The packed initial W and H (fp64, on X's device), the tensors that must outlive the launch and the (message,
    device flag) checks of the init: "random" (scikit-learn's draws for seeds[p] times sqrt(X.mean() / k)), "nndsvd" /
    "nndsvda" (computed on the device from an exact SVD, one per matrix of the stack) or one (W, H) pair per problem."""
    _, n, m = dX.shape
    dev = dX.device
    if not isinstance(init, str):
        dW = torch.from_numpy(np.concatenate([np.asarray(w, dtype=np.float64).ravel() for w, _ in init])).to(dev)
        dH = torch.from_numpy(np.concatenate([np.asarray(h, dtype=np.float64).ravel() for _, h in init])).to(dev)
        return dW, dH, [], []
    table, kmax, d_ranks, d_xi, w_problem, h_problem = _batch_plan(torch, lib, n, m, ranks, xi, dev)
    if init == "random":
        unit_w, unit_h = _batch_draws(torch, n, m, ranks, seeds, dev)
        avg = _init_scale(torch, dX, Xh, d_ranks, d_xi)
        return unit_w * avg[w_problem], unit_h * avg[h_problem], [], []
    dXc = dX.contiguous()  # the SVD reads row-major matrices
    dW = torch.empty(int(ranks.astype(np.int64).sum()) * n, dtype=torch.float64, device=dev)
    dH = torch.empty(int(ranks.astype(np.int64).sum()) * m, dtype=torch.float64, device=dev)
    work = torch.empty(int(lib.ms_nndsvd_workspace_bytes(m, len(dX))), dtype=torch.uint8, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    nat.check(lib.ms_nndsvd_init(dXc.data_ptr(), n, m, len(dX), table.data_ptr(), len(ranks), kmax,
                                 int(init == "nndsvda"), work.data_ptr(), dW.data_ptr(), dH.data_ptr(),
                                 status.data_ptr(), ctypes.c_void_p(stream.cuda_stream)), "ms_nndsvd_init")
    return dW, dH, [dXc, work], [(_NNDSVD_DEGENERATE, status)]


def _launch_outputs(torch, dev, regime, n, max_rows, P, m, dtype):
    """(resident, n_iter, err, vaf): the regime - resident when n fits the resident kernel's shared memory (regime None),
    or as asked - and the per-problem outputs of the launch."""
    resident = n <= max_rows if regime is None else regime == "resident"
    return (resident, torch.empty(P, dtype=torch.int32, device=dev), torch.empty(P, dtype=dtype, device=dev),
            torch.empty((P, m + 1), dtype=dtype, device=dev))


def _finish(torch, stream, ranks, seeds, n, m, device_arrays, keep, checks, defer):
    """The end of every entry: the PendingNMF of the queued launch under defer, else its result."""
    pending = PendingNMF(torch, stream, ranks, seeds, n, m, device_arrays, keep, checks)
    return pending if defer else pending.result()


_NEGATIVE_CHECK = ((_NEGATIVE_X, lambda A: A < 0),)


def nmf_mu_batched(X, ranks: Sequence[int], seeds: Sequence[int], max_iter: int = 200, tol: float = 1e-4,
                   check_every: int = 10, init=None, device=None, x_index: Optional[Sequence[int]] = None,
                   regime: Optional[str] = None, defer: bool = False) -> Union[NMFBatchResult, PendingNMF]:
    """Runs len(ranks) MU factorisations in one kernel launch.  defer=True returns a PendingNMF right after the
    launch (`.result()` gives the NMFBatchResult).

    X: non-negative (n samples x m muscles), or a stack (B, n, m) of such matrices (e.g. one per
    gait cycle) with x_index[p] naming the matrix of problem p; a numpy array, or a CUDA tensor
    (e.g. the output of `envelope_windows`), which then never leaves the device.  ranks[p], seeds[p]:
    rank and sklearn `random_state` of problem p; `init` optionally gives the initial (W, H) pairs
    instead of the seeds.  regime: None (by size), "resident" or "stream"."""
    import torch

    Xh, shape = _host_x(X)
    ranks, seeds, xi = _problem_arrays(ranks, seeds, x_index, shape, regime, max_iter, tol)
    how = "random" if init is None else init
    _check_init(how, ranks, seeds, shape, names=("random",))
    checks = _check_x(Xh, _NEGATIVE_CHECK) if Xh is not None else []
    lib = _cuda_lib("nmf_mu_batched")
    _, n, m = shape
    P = len(ranks)
    dX = _device_x(torch, X, Xh, strided=False, device=device, host_dtype=np.float32)  # float64 for a CUDA X
    dev = dX.device
    stream = torch.cuda.current_stream(dev)
    with torch.cuda.device(dev):
        if Xh is None:
            checks = _check_x(dX, _NEGATIVE_CHECK, defer)
        # sklearn's init in float64, then the kernel's fp32
        dW, dH = (t.to(torch.float32) for t in _initial_factors(torch, lib, how, dX, Xh, ranks, seeds, xi, stream)[:2])
        dX = dX.to(torch.float32)
        max_rows = int(lib.ms_nmf_resident_max_rows(m, int(ranks.max())))
        resident, d_iter, d_err, d_vaf = _launch_outputs(torch, dev, regime, n, max_rows, P, m, torch.float32)
        if resident:
            # the problem table lives on the device for as long as the sweep is repeated: the launch copies nothing
            # and waits for nothing
            work, kmax_plan = _batch_plan(torch, lib, n, m, ranks, xi, dev)[:2]
            nat.check(
                lib.ms_nmf_mu_batched_planned(
                    dX.data_ptr(), n, m, work.data_ptr(), P, kmax_plan, dW.data_ptr(), dH.data_ptr(), int(max_iter),
                    ctypes.c_float(tol), int(check_every), d_iter.data_ptr(), d_err.data_ptr(), d_vaf.data_ptr(),
                    ctypes.c_void_p(stream.cuda_stream),
                ),
                "ms_nmf_mu_batched_planned",
            )
        else:
            work = torch.empty(int(lib.ms_nmf_stream_workspace_bytes(m, P)), dtype=torch.uint8, device=dev)
            h_ranks = ranks.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
            h_xi = xi.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
            nat.check(
                lib.ms_nmf_mu_stream(
                    dX.data_ptr(), n, m, h_ranks, h_xi, P, dW.data_ptr(), dH.data_ptr(), int(max_iter), ctypes.c_float(tol),
                    int(check_every), work.data_ptr(), d_iter.data_ptr(), d_err.data_ptr(), d_vaf.data_ptr(),
                    ctypes.c_void_p(stream.cuda_stream),
                ),
                "ms_nmf_mu_stream",
            )
        return _finish(torch, stream, ranks, seeds, n, m, [dW, dH, d_iter, d_err, d_vaf], [dX, work], checks, defer)


def nmf_cd_batched(X, ranks: Sequence[int], init="nndsvda", seeds: Optional[Sequence[int]] = None, max_iter: int = 200,
                   tol: float = 1e-4, x_index: Optional[Sequence[int]] = None, regime: Optional[str] = None,
                   defer: bool = False) -> Union[NMFBatchResult, PendingNMF]:
    """Runs len(ranks) factorisations with scikit-learn's coordinate-descent solver (`NMF(solver="cd")`, shuffle=False,
    no regularisation) in fp64, all in one launch.  X, ranks, x_index, regime and defer as for `nmf_mu_batched`.

    init: "nndsvd" / "nndsvda" (computed on the device from an exact SVD, one per matrix of the stack; `seeds` is not
    needed and sklearn's random_state has no counterpart), "random" (sklearn's draws for seeds[p]), or one explicit
    (W, H) pair per problem.  The factors of the result are fp64; its seeds are -1 where no seed was given."""
    import torch

    Xh, shape = _host_x(X)
    ranks, seeds, xi = _problem_arrays(ranks, seeds, x_index, shape, regime, max_iter, tol)
    _check_init(init, ranks, seeds, shape)
    checks = _check_x(Xh, _NEGATIVE_CHECK) if Xh is not None else []
    lib = _cuda_lib("nmf_cd_batched")
    _, n, m = shape
    P = len(ranks)
    dX = _device_x(torch, X, Xh, strided=False)
    dev = dX.device
    table, kmax = _batch_plan(torch, lib, n, m, ranks, xi, dev)[:2]
    stream = torch.cuda.current_stream(dev)
    with torch.cuda.device(dev):
        if Xh is None:
            checks = _check_x(dX, _NEGATIVE_CHECK, defer)
        dW, dH, keep, init_checks = _initial_factors(torch, lib, init, dX, Xh, ranks, seeds, xi, stream)
        max_rows = int(lib.ms_nmf_cd_resident_max_rows(m, kmax))
        resident, d_iter, d_err, d_vaf = _launch_outputs(torch, dev, regime, n, max_rows, P, m, torch.float64)
        keep.append(dX)
        if resident:
            nat.check(lib.ms_nmf_cd_batched_planned(
                dX.data_ptr(), n, m, table.data_ptr(), P, kmax, dW.data_ptr(), dH.data_ptr(), int(max_iter), float(tol),
                d_iter.data_ptr(), d_err.data_ptr(), d_vaf.data_ptr(), ctypes.c_void_p(stream.cuda_stream)),
                "ms_nmf_cd_batched_planned")
        else:
            work = torch.empty(int(lib.ms_nmf_cd_stream_workspace_bytes(m, P)), dtype=torch.uint8, device=dev)
            keep.append(work)
            nat.check(lib.ms_nmf_cd_stream(
                dX.data_ptr(), n, m, table.data_ptr(), P, kmax, dW.data_ptr(), dH.data_ptr(), int(max_iter), float(tol),
                work.data_ptr(), d_iter.data_ptr(), d_err.data_ptr(), d_vaf.data_ptr(), ctypes.c_void_p(stream.cuda_stream)),
                "ms_nmf_cd_stream")
        return _finish(torch, stream, ranks, seeds, n, m, [dW, dH, d_iter, d_err, d_vaf], keep, checks + init_checks,
                       defer)


_BETA_NAMES = {"frobenius": 2.0, "kullback-leibler": 1.0, "itakura-saito": 0.0}
_BETA_ZEROS = ("When beta_loss <= 0 and X contains zeros, the solver may diverge. Please add small values to X, or use a "
               "positive beta_loss.")


def _beta_to_float(beta_loss) -> float:
    """sklearn's _beta_loss_to_float, with its parameter check: a name of _BETA_NAMES or a finite real number."""
    if isinstance(beta_loss, str):
        if beta_loss not in _BETA_NAMES:
            raise ValueError(f"beta_loss must be one of {sorted(_BETA_NAMES)} or a float, not {beta_loss!r}")
        return _BETA_NAMES[beta_loss]
    if isinstance(beta_loss, bool) or not isinstance(beta_loss, (int, float, np.integer, np.floating)) \
            or not np.isfinite(beta_loss):
        raise ValueError(f"beta_loss must be one of {sorted(_BETA_NAMES)} or a float, not {beta_loss!r}")
    return float(beta_loss)


class _BetaLossSolverError(ValueError, NotImplementedError):
    """scikit-learn's ValueError for a solver other than "mu" with beta_loss != 2.  It is also the NotImplementedError
    that find_synergies(engine="gpu") raised for beta_loss != 2 before the β kernels existed, so code that caught that
    keeps working."""


def _beta_solver_error(solver, beta_loss) -> ValueError:
    return _BetaLossSolverError(f"Invalid beta_loss parameter: solver {solver!r} does not handle beta_loss = {beta_loss!r}")


def _zeros_check(beta):
    """sklearn's refusal of zeros in X under beta_loss <= 0 (after its other checks of X)."""
    return ((_BETA_ZEROS, lambda A: A == 0),) if beta <= 0 else ()


def nmf_beta_batched(X, ranks: Sequence[int], beta_loss, init="nndsvda", seeds: Optional[Sequence[int]] = None,
                     max_iter: int = 200, tol: float = 1e-4, x_index: Optional[Sequence[int]] = None,
                     regime: Optional[str] = None, defer: bool = False) -> Union[NMFBatchResult, PendingNMF]:
    """Runs len(ranks) factorisations with scikit-learn's multiplicative updates for the β-divergence
    (`NMF(solver="mu", beta_loss=beta_loss)`, no regularisation) in fp64, all in one launch.

    beta_loss: "kullback-leibler" (1), "itakura-saito" (0) or any float other than 2 (Frobenius runs on
    `nmf_mu_batched` / `nmf_cd_batched`).  X, ranks, init, seeds, x_index, regime and defer as for `nmf_cd_batched`; X
    may also be a strided CUDA view (a channel-major `env.T`), read in place.  A negative X, and a zero in X with
    beta_loss <= 0, raise sklearn's ValueError (under defer, from `.result()` for a CUDA X).  The result's err is
    sklearn's reconstruction_err_, sqrt(2 D_beta(X | W H)); its VAF is the Frobenius one, as `vaf` computes it."""
    import torch

    beta = _beta_to_float(beta_loss)
    if beta == 2.0:
        raise ValueError("beta_loss = 2 (Frobenius) runs on nmf_mu_batched or nmf_cd_batched")
    Xh, shape = _host_x(X)
    ranks, seeds, xi = _problem_arrays(ranks, seeds, x_index, shape, regime, max_iter, tol)
    _check_init(init, ranks, seeds, shape, values=True)
    x_checks = _NEGATIVE_CHECK + _zeros_check(beta)
    checks = _check_x(Xh, x_checks) if Xh is not None else []
    lib = _cuda_lib("nmf_beta_batched")
    _, n, m = shape
    dX = _device_x(torch, X, Xh, strided=True)
    dev = dX.device
    table, kmax = _batch_plan(torch, lib, n, m, ranks, xi, dev)[:2]
    stream = torch.cuda.current_stream(dev)
    with torch.cuda.device(dev):
        if Xh is None:
            checks = _check_x(dX, x_checks, defer)
        dW, dH, keep, init_checks = _initial_factors(torch, lib, init, dX, Xh, ranks, seeds, xi, stream)
        d_iter, d_err, d_vaf, work = _beta_launch(torch, lib, dX, n, m, table, len(ranks), kmax, dW, dH, beta, 1,
                                                  max_iter, tol, regime, stream)
        return _finish(torch, stream, ranks, seeds, n, m, [dW, dH, d_iter, d_err, d_vaf], keep + [dX, work],
                       checks + init_checks, defer)


def _beta_launch(torch, lib, dX, n, m, table, P, kmax, dW, dH, beta, update_H, max_iter, tol, regime, stream):
    """Queues ms_nmf_beta on `stream` (regime None: resident when n fits shared memory); returns the device outputs
    and the workspace, which must outlive the launch."""
    dev = dX.device
    max_rows = int(lib.ms_nmf_beta_resident_max_rows(m, kmax))
    resident, d_iter, d_err, d_vaf = _launch_outputs(torch, dev, regime, n, max_rows, P, m, torch.float64)
    work = torch.empty(0 if resident else int(lib.ms_nmf_beta_workspace_bytes(n, m, P, kmax)), dtype=torch.uint8,
                       device=dev)
    nat.check(lib.ms_nmf_beta(
        dX.data_ptr(), n, m, dX.stride(1), dX.stride(2), table.data_ptr(), P, kmax, dW.data_ptr(), dH.data_ptr(),
        float(beta), int(update_H), int(max_iter), float(tol), 0 if resident else 1,
        work.data_ptr() if not resident else None, d_iter.data_ptr(), d_err.data_ptr(), d_vaf.data_ptr(),
        ctypes.c_void_p(stream.cuda_stream)), "ms_nmf_beta")
    return d_iter, d_err, d_vaf, work


# sklearn's texts for the input checks of NMF.transform (sklearn.utils.validation)
_TRANSFORM_NAN = "Input X contains NaN."
_TRANSFORM_INF = "Input X contains infinity or a value too large for dtype('float64')."
_TRANSFORM_NEGATIVE = "Negative values in data passed to X in NMF."
_SOLVER_CODES = {"cd": 0, "mu": 1}
# the input checks of sklearn's transform, in its order: NaN, infinity, negative values
_TRANSFORM_CHECKS = ((_TRANSFORM_NAN, lambda A: A != A), (_TRANSFORM_INF, lambda A: abs(A) == np.inf),
                     (_TRANSFORM_NEGATIVE, lambda A: A < 0))


def _transform_args(shape, H, solver, beta_loss="frobenius"):
    """Validates the synergies nmf_transform_batched is given for an X of `shape` (B, n, m), without touching a device;
    returns (H list, ranks)."""
    if solver not in _SOLVER_CODES:
        raise ValueError(f"solver must be 'cd' or 'mu', not {solver!r}")
    if _beta_to_float(beta_loss) != 2.0 and solver != "mu":
        raise _beta_solver_error(solver, beta_loss)
    Hs = [np.ascontiguousarray(h, dtype=np.float64) for h in H]
    if not Hs:
        raise ValueError("H must give one (k, m) matrix per problem")
    m = Hs[0].shape[-1] if Hs[0].ndim == 2 else -1
    for p, h in enumerate(Hs):
        if h.ndim != 2 or h.shape[1] != m or not 1 <= h.shape[0] <= 16 or m > 64:
            raise ValueError(f"H[{p}] must be a (k, m) matrix with 1 <= k <= 16 and m <= 64 columns shared by every "
                             f"problem, not {h.shape}")
        if not np.isfinite(h).all() or (h < 0).any():
            raise ValueError(f"H[{p}] must be finite and non-negative")
    if shape[-1] != m:
        raise ValueError(f"X has {shape[-1]} features, but H has {m}")
    return Hs, [h.shape[0] for h in Hs]


def nmf_transform_batched(X, H: Sequence, x_index: Optional[Sequence[int]] = None, solver: str = "cd",
                          max_iter: int = 200, tol: float = 1e-4, regime: Optional[str] = None,
                          defer: bool = False, beta_loss="frobenius") -> Union[NMFBatchResult, PendingNMF]:
    """Fits activations to fixed synergies - scikit-learn's `NMF.transform` (update_H=False, no regularisation) - for a
    batch of problems in one launch, in fp64: problem p fits W_p >= 0 to X[x_index[p]] with H[p] (k_p x m) fixed.

    solver "cd" starts from W = 0, "mu" from sqrt(X.mean() / k_p), as sklearn does; max_iter and tol are sklearn's.
    X: a non-negative (n, m) matrix or a (B, n, m) stack, as a numpy array or a CUDA tensor (which never leaves the
    device; a strided view such as the (samples, channels) `env.T` of a channel-major envelope is read in place).
    A negative or non-finite X raises ValueError (under defer, from `.result()`).  regime: None (by size),
    "resident" or "stream".  beta_loss: "frobenius" (2), or with solver "mu" "kullback-leibler" (1), "itakura-saito"
    (0) or any other float - then err is sklearn's square-rooted β-divergence, and a zero in X with beta_loss <= 0
    raises sklearn's ValueError.  Returns an NMFBatchResult whose H are the given matrices and whose seeds are -1, or a
    PendingNMF when defer=True."""
    return _nmf_transform(X, H, x_index, solver, max_iter, tol, regime, defer, beta_loss=beta_loss)


def _nmf_transform(X, H, x_index, solver, max_iter, tol, regime, defer, device_w=False, beta_loss="frobenius"):
    import torch

    Xh, shape = _host_x(X)
    Hs, ranks = _transform_args(shape, H, solver, beta_loss)
    ranks, seeds, xi = _problem_arrays(ranks, None, x_index, shape, regime, max_iter, tol)
    beta = _beta_to_float(beta_loss)
    x_checks = _TRANSFORM_CHECKS + _zeros_check(beta)
    checks = _check_x(Xh, x_checks) if Xh is not None else []
    lib = _cuda_lib("nmf_transform_batched")
    _, n, m = shape
    P = len(ranks)
    dX = _device_x(torch, X, Xh, strided=True)
    dev = dX.device
    table, kmax, d_ranks, d_xi, w_problem, _ = _batch_plan(torch, lib, n, m, ranks, xi, dev)
    stream = torch.cuda.current_stream(dev)
    with torch.cuda.device(dev):
        if Xh is None:
            checks = _check_x(dX, x_checks, defer)
        if solver == "cd":
            dW = torch.zeros(int(ranks.astype(np.int64).sum()) * n, dtype=torch.float64, device=dev)
        else:
            dW = _init_scale(torch, dX, Xh, d_ranks, d_xi)[w_problem]
        dH = torch.from_numpy(np.concatenate([h.ravel() for h in Hs])).to(dev)
        if beta != 2.0:  # the β-divergence: the same loop as the fit, H fixed
            d_iter, d_err, d_vaf, work = _beta_launch(torch, lib, dX, n, m, table, P, kmax, dW, dH, beta, 0, max_iter,
                                                      tol, regime, stream)
        else:
            max_rows = int(lib.ms_nmf_fixed_h_resident_max_rows(m, kmax))
            resident, d_iter, d_err, d_vaf = _launch_outputs(torch, dev, regime, n, max_rows, P, m, torch.float64)
            work = torch.empty(0 if resident else int(lib.ms_nmf_fixed_h_workspace_bytes(n, m, P, kmax)),
                               dtype=torch.uint8, device=dev)
            nat.check(lib.ms_nmf_fixed_h(
                dX.data_ptr(), n, m, dX.stride(1), dX.stride(2), table.data_ptr(), P, kmax, dW.data_ptr(), dH.data_ptr(),
                _SOLVER_CODES[solver], int(max_iter), float(tol), 0 if resident else 1,
                work.data_ptr() if not resident else None, d_iter.data_ptr(), d_err.data_ptr(), d_vaf.data_ptr(),
                ctypes.c_void_p(stream.cuda_stream)), "ms_nmf_fixed_h")
        if device_w:
            return dW, d_iter
        return _finish(torch, stream, ranks, seeds, n, m, [dW, dH, d_iter, d_err, d_vaf], [dX, work], checks, defer)


# ---- synergy comparison -------------------------------------------------------------------------------
@dataclass
class SynergyMatch:
    """What `match_synergies_batched` returns: numpy arrays, or CUDA tensors for a CUDA H.  kmax is the largest rank
    among the sets; a pair of rank k < kmax has -1 (perm) and NaN (sim) in its columns k .. kmax - 1."""

    mean: object          # (P,) float64: mean matched cosine similarity of each pair
    sim: object = None    # (P, kmax) float64: sim[p, i] = similarity of row i of a and row perm[p, i] of b
    perm: object = None   # (P, kmax) int8: the row of b paired with row i of a


def _match_sets(H):
    """(on_device, list of sets, m) after the shape checks of match_synergies_batched; a set is a 2-D numpy array or
    a 2-D CUDA tensor.  Touches no device."""
    import torch

    if not isinstance(H, (list, tuple)):
        if not (isinstance(H, torch.Tensor) and H.is_cuda):
            H = H.detach().cpu().numpy() if isinstance(H, torch.Tensor) else np.asarray(H)
        if H.ndim != 3:
            raise ValueError(f"H must be a list of (k, m) synergy sets or an (S, k, m) stack, not shape {tuple(H.shape)}")
        if isinstance(H, torch.Tensor):  # a CUDA stack stays one tensor: S can be large
            S, k, m = H.shape
            if S < 1 or not 1 <= k <= 16 or not 1 <= m <= 64:
                raise ValueError(f"H is a stack of {S} sets of rank k = {k} with m = {m} muscles: a synergy set needs "
                                 "1 <= k <= 16 and 1 <= m <= 64")
            return True, H, m
    sets = list(H)
    on_device = any(isinstance(h, torch.Tensor) and h.is_cuda for h in sets)
    out = []
    for s, h in enumerate(sets):
        if not (isinstance(h, torch.Tensor) and h.is_cuda):
            h = h.detach().cpu().numpy() if isinstance(h, torch.Tensor) else np.asarray(h)
        if h.ndim != 2:
            raise ValueError(f"H[{s}] must be a (k, m) synergy set, not shape {tuple(h.shape)}")
        out.append(h)
    if not out:
        raise ValueError("H holds no synergy set")
    m = int(out[0].shape[1])
    for s, h in enumerate(out):
        k = int(h.shape[0])
        if not 1 <= k <= 16:
            raise ValueError(f"H[{s}] has rank k = {k}: a synergy set has 1 <= k <= 16 rows")
        if int(h.shape[1]) != m:
            raise ValueError(f"H[{s}] has m = {h.shape[1]} muscles, H[0] has {m}: every set must have the same m")
    if not 1 <= m <= 64:
        raise ValueError(f"the sets have m = {m} muscles: 1 <= m <= 64 is supported")
    return on_device, out, m


def _match_pairs(pairs, ranks, n_sets):
    """Checks a host (P, 2) pair list against the sets' ranks (an array, or an int for a stack); returns it as int32."""
    pairs = np.asarray(pairs)
    if pairs.ndim != 2 or pairs.shape[1] != 2 or not (pairs.size == 0 or np.issubdtype(pairs.dtype, np.integer)):
        raise ValueError(f"pairs must be a (P, 2) integer array of set indices, not {pairs.dtype} {pairs.shape}")
    if pairs.size and (pairs.min() < 0 or pairs.max() >= n_sets):
        bad = int(np.flatnonzero(((pairs < 0) | (pairs >= n_sets)).any(axis=1))[0])
        raise ValueError(f"pair {bad} = {tuple(pairs[bad].tolist())} names a set H does not have ({n_sets} sets)")
    if not isinstance(ranks, int) and pairs.size:
        ka, kb = ranks[pairs[:, 0]], ranks[pairs[:, 1]]
        if (ka != kb).any():
            bad = int(np.flatnonzero(ka != kb)[0])
            a, b = pairs[bad]
            raise ValueError(f"pair {bad} compares H[{a}] (rank {ka[bad]}) with H[{b}] (rank {kb[bad]}): both sets of a "
                             "pair must have the same rank")
    return np.ascontiguousarray(pairs, dtype=np.int32)


def match_synergies_batched(H, pairs=None, *, similarities: bool = False, permutations: bool = False) -> SynergyMatch:
    """Compares synergy sets pair by pair in one launch, the standard comparison of synergies between gait cycles,
    trials or subjects: each synergy vector (a row of `components_`) is scaled to unit length (a zero row has
    similarity 0 with everything), the k x k matrix S of scalar products is formed, and the rows are paired one to one
    so that the summed similarity is as large as possible - the optimum `scipy.optimize.linear_sum_assignment(S,
    maximize=True)` finds.  fp64 (csrc/ms_synmatch.cu).

    H: a list of (k, m) synergy sets or an (S, k, m) stack, as numpy arrays or CUDA tensors (which never leave the
    device); 1 <= k <= 16, 1 <= m <= 64, finite.  pairs: a (P, 2) array of set indices, both sets of a pair of the same
    rank; None compares every unordered pair a < b, in `np.triu_indices(S, 1)` order, generated on the device (the
    kernel decodes the pair index: no pair list is built).
    Returns a SynergyMatch with `mean` (P,) and, on request, `sim` and `perm` (P, kmax).  Argument errors raise
    ValueError, naming the set or pair, before any native call."""
    import torch

    on_device, sets, m = _match_sets(H)
    stack = isinstance(sets, torch.Tensor)
    n_sets = int(sets.shape[0]) if stack else len(sets)
    if stack:
        ranks, kmax = int(sets.shape[1]), int(sets.shape[1])
    else:
        ranks = np.array([h.shape[0] for h in sets], dtype=np.int64)
        kmax = int(ranks.max())
    pairs_dev = None
    if pairs is None:
        if stack or (ranks == ranks[0]).all():
            pass  # every pair of the triangle has equal ranks
        else:
            raise ValueError("pairs=None compares every pair of sets, but H mixes ranks "
                             f"{sorted(set(ranks.tolist()))}: give the pairs of equal rank")
    elif isinstance(pairs, torch.Tensor) and pairs.is_cuda:
        if pairs.ndim != 2 or pairs.shape[1] != 2 or pairs.dtype.is_floating_point or pairs.dtype == torch.bool:
            raise ValueError(f"pairs must be a (P, 2) integer array of set indices, not {pairs.dtype} {tuple(pairs.shape)}")
        pairs_dev = pairs
        if pairs.numel():
            if int(pairs.min()) < 0 or int(pairs.max()) >= n_sets:
                raise ValueError(f"pairs names a set H does not have ({n_sets} sets)")
            if not stack:
                r = torch.from_numpy(ranks).to(pairs.device)[pairs.long()]
                differ = (r[:, 0] != r[:, 1]).nonzero()
                if differ.numel():
                    bad = int(differ[0, 0])
                    a, b = pairs[bad].tolist()
                    raise ValueError(f"pair {bad} compares H[{a}] (rank {ranks[a]}) with H[{b}] (rank {ranks[b]}): "
                                     "both sets of a pair must have the same rank")
    else:
        pairs = _match_pairs(pairs, ranks, n_sets)
    # the sets as one fp64 array (a CUDA one never leaves its device), checked for finiteness in one pass
    if stack:
        flat = sets.detach().to(torch.float64).contiguous().view(-1)
    elif on_device:
        dev = next(h.device for h in sets if isinstance(h, torch.Tensor))
        flat = torch.cat([torch.as_tensor(h, device=dev).detach().to(torch.float64).reshape(-1) for h in sets])
    else:
        flat = np.concatenate([np.asarray(h, dtype=np.float64).ravel() for h in sets])
    if not bool((torch.isfinite(flat) if on_device else np.isfinite(flat)).all()):
        if stack:
            raise ValueError("H contains a non-finite entry")
        finite = [bool((torch.isfinite(h) if isinstance(h, torch.Tensor) else np.isfinite(h)).all()) for h in sets]
        bad = finite.index(False)
        raise ValueError(f"H[{bad}] contains a non-finite entry")

    lib = nat.lib()
    if not torch.cuda.is_available():
        raise nat.NativeError("match_synergies_batched needs a CUDA device; there is no CPU fallback")
    dev = flat.device if on_device else torch.device(f"cuda:{torch.cuda.current_device()}")
    with torch.cuda.device(dev):
        table = torch.zeros((n_sets, 2), dtype=torch.int64, device=dev)  # ms_synergy_set: offset, then k | reserved << 32
        dH = flat if on_device else torch.from_numpy(flat).to(dev)
        if stack:
            table[:, 0] = torch.arange(n_sets, device=dev) * (kmax * m)
            table[:, 1] = kmax
        else:
            offsets = np.concatenate([[0], np.cumsum(ranks * m)[:-1]])
            table.copy_(torch.from_numpy(np.stack([offsets, ranks], axis=1)))
        if pairs_dev is not None:
            dP = pairs_dev.to(device=dev, dtype=torch.int32).contiguous()
        elif pairs is not None:
            dP = torch.from_numpy(pairs).to(dev)
        else:
            dP = None  # every pair a < b: the kernel decodes the pair index, no list is built
        P = int(dP.shape[0]) if dP is not None else n_sets * (n_sets - 1) // 2
        d_mean = torch.empty(P, dtype=torch.float64, device=dev)
        d_sim = torch.empty((P, kmax), dtype=torch.float64, device=dev) if similarities else None
        d_perm = torch.empty((P, kmax), dtype=torch.int8, device=dev) if permutations else None
        work = torch.empty(int(lib.ms_synergy_match_workspace_bytes(n_sets)), dtype=torch.uint8, device=dev)
        stream = torch.cuda.current_stream(dev)
        nat.check(lib.ms_synergy_match(
            dH.data_ptr(), m, table.data_ptr(), n_sets, kmax, dP.data_ptr() if dP is not None else None, P,
            d_perm.data_ptr() if d_perm is not None else None, d_sim.data_ptr() if d_sim is not None else None,
            d_mean.data_ptr(), work.data_ptr(), work.numel(), ctypes.c_void_p(stream.cuda_stream)), "ms_synergy_match")
    if on_device:
        return SynergyMatch(d_mean, d_sim, d_perm)
    return SynergyMatch(d_mean.cpu().numpy(), d_sim.cpu().numpy() if similarities else None,
                        d_perm.cpu().numpy() if permutations else None)


# ---- reference API ------------------------------------------------------------------------------------
def vaf(original_df: pandas.DataFrame, transformed_signal=None, components=None, reconstructed_signal=None) -> pandas.DataFrame:
    """Variance accounted for, overall and per muscle (analysis.py:597-667)."""
    if reconstructed_signal is None:
        reconstructed_signal = transformed_signal @ components
    error = original_df - reconstructed_signal

    def ss(arr, axis):
        return np.sum(arr.to_numpy() ** 2, axis=axis)

    overall = 1 - ss(error, (0, 1)) / ss(original_df, (0, 1))
    per_column = 1 - ss(error, 0) / ss(original_df, 0)
    labels = ["All signals"] + original_df.columns.tolist()
    values = [overall] + list(per_column.reshape(-1))
    return pandas.DataFrame({lbl: [val] for (lbl, val) in zip(labels, values)})


@dataclass
class NMFModel:
    """What the reference keeps of a fitted `sklearn.decomposition.NMF`."""

    n_components: int
    components_: np.ndarray
    n_iter_: int
    reconstruction_err_: float
    n_features_in_: int
    random_state: Optional[int]  # None: a deterministic init (nndsvd*)
    solver: str = "mu"
    beta_loss: str = "frobenius"
    init: str = "random"
    restarts: Optional[pandas.DataFrame] = None  # extension: one row per restart (seed, n_iter, err, VAF)
    max_iter: int = 100_000
    tol: float = 1e-6

    def transform(self, X):
        """sklearn's `NMF.transform`: the activations W >= 0 that fit X with these components fixed, by the model's
        solver, beta_loss, max_iter and tol, on the GPU in fp64 (`nmf_transform_batched`).  X: a DataFrame, an ndarray or a CUDA
        tensor (n, n_features_in_); returns an (n, n_components) ndarray, or a CUDA tensor for a CUDA input.  Raises
        sklearn's ValueErrors for non-finite or negative X and a wrong feature count, and emits its ConvergenceWarning
        when max_iter is reached with tol > 0."""
        import torch

        if isinstance(X, torch.Tensor) and X.is_cuda:
            if X.ndim != 2:
                raise ValueError(f"Expected 2D array, got {X.ndim}D array instead")
        else:
            X = np.asarray(X.to_numpy() if isinstance(X, pandas.DataFrame) else X, dtype=np.float64)
            if X.ndim != 2:
                raise ValueError(f"Expected 2D array, got {X.ndim}D array instead")
        _check_x(X, _TRANSFORM_CHECKS)
        if X.shape[1] != self.n_features_in_:
            raise ValueError(f"X has {X.shape[1]} features, but NMF is expecting {self.n_features_in_} features as input.")
        W, n_iter = _nmf_transform(X, [self.components_], None, self.solver, self.max_iter, self.tol, None, False,
                                   device_w=True, beta_loss=self.beta_loss)
        if self.tol > 0 and int(n_iter[0]) == self.max_iter:
            from sklearn.exceptions import ConvergenceWarning

            warnings.warn("Maximum number of iterations %d reached. Increase it to improve convergence." % self.max_iter,
                          ConvergenceWarning)
        W = W.reshape(X.shape[0], self.components_.shape[0])
        return W if isinstance(X, torch.Tensor) else W.cpu().numpy()

    def inverse_transform(self, W):
        """sklearn's `NMF.inverse_transform`: W @ components_ (a CUDA tensor for a CUDA W)."""
        import torch

        if isinstance(W, torch.Tensor):
            return W @ torch.as_tensor(self.components_, dtype=W.dtype, device=W.device)
        return np.asarray(W) @ self.components_


@dataclass
class SynergyRunResult:
    vaf_values: pandas.DataFrame
    components: Union[pandas.DataFrame, Mapping[int, pandas.DataFrame]]
    model: Union[NMFModel, Mapping[int, NMFModel]]
    transformed: Union[np.ndarray, Mapping[int, np.ndarray], None] = field(default=None, repr=False)


def _find_synergies_sklearn(processed_emg_df, n_components, max_components, **sklearn_kwargs) -> "SynergyRunResult":
    """find_synergies as the reference runs it (analysis.py:848-914): one sklearn.decomposition.NMF per rank."""
    from sklearn.decomposition import NMF

    def single(k):
        model = NMF(n_components=k, **sklearn_kwargs)
        transformed = model.fit_transform(processed_emg_df)
        values = vaf(processed_emg_df, components=model.components_, transformed_signal=transformed)
        comps = pandas.DataFrame(model.components_, columns=processed_emg_df.columns)
        return SynergyRunResult(values, comps, model, transformed)

    if max_components is None:
        return single(n_components)
    runs = OrderedDict((k, single(k)) for k in range(n_components, max_components + 1))
    vaf_values = pandas.concat([r.vaf_values for r in runs.values()])
    vaf_values.set_index(np.array(tuple(runs.keys())), inplace=True)
    return SynergyRunResult(vaf_values, {k: r.components for k, r in runs.items()}, {k: r.model for k, r in runs.items()},
                            {k: r.transformed for k, r in runs.items()})


# keywords of sklearn.decomposition.NMF that engine="gpu" accepts at scikit-learn's default value only
_SKLEARN_DEFAULTS = {"alpha_W": 0.0, "alpha_H": "same", "l1_ratio": 0.0, "shuffle": False, "verbose": 0}


def find_synergies(
    processed_emg_df: pandas.DataFrame,
    n_components: int,
    max_components: Optional[int] = None,
    *,
    max_iter: int = 100_000,
    tol: float = 1e-6,
    n_restarts: int = 1,
    engine: str = "auto",
    **sklearn_kwargs,
) -> SynergyRunResult:
    """Find muscle synergies with NMF (analysis.py:713-914) - all ranks and restarts in one launch.

    engine="auto": solver="mu", init="random", beta_loss="frobenius" (or 2), random_state=int run on the GPU, all ranks
    and restarts in one launch; `n_restarts` (extension) runs seeds random_state .. random_state+R-1 per rank and keeps,
    per rank, the restart with the smallest reconstruction error.  Any other scikit-learn configuration (the
    default solver="cd", nndsvd inits, regularisation ...) is forwarded to scikit-learn as the reference does.
    engine="sklearn" always forwards.  engine="gpu" runs on the GPU solver="cd" (the default; fp64, `nmf_cd_batched`)
    or "mu", with init None (resolved as scikit-learn does: "nndsvda" if k <= min(n_samples, n_features), else
    "random"), "nndsvd", "nndsvda" or "random", and raises NotImplementedError for any other keyword or value.  With
    solver="mu" it also runs beta_loss "kullback-leibler", "itakura-saito" or any float (fp64, `nmf_beta_batched`);
    solver="cd" with beta_loss != 2 raises scikit-learn's ValueError."""
    if engine not in ("auto", "sklearn", "gpu"):
        raise ValueError(f"engine must be 'auto', 'sklearn' or 'gpu', not {engine!r}")
    if processed_emg_df.empty:
        raise ValueError("empty EMG DataFrame")
    num_features = len(processed_emg_df.columns)
    if n_components < 1 or n_components > num_features:
        raise ValueError("invalid number of components")
    if max_components is not None and (max_components < n_components or max_components > num_features):
        raise ValueError("invalid number of components")
    if engine == "gpu":
        return _find_synergies_gpu(processed_emg_df, n_components, max_components, max_iter, tol, n_restarts,
                                   sklearn_kwargs)
    kw = dict(sklearn_kwargs)
    solver = kw.pop("solver", "cd")
    init = kw.pop("init", None)
    beta_loss = kw.pop("beta_loss", "frobenius")
    seed = kw.pop("random_state", None)
    if engine == "sklearn" or solver != "mu" or init != "random" or beta_loss not in ("frobenius", 2, 2.0) or kw:
        # Everything the batched kernels do not implement is what the reference itself does with it: the keywords go
        # to scikit-learn unchanged (analysis.py:848-864) - solver="cd" with an nndsvd* init is the tutorial's own call
        # (docs/source/tutorials/Finding muscle synergies.ipynb, cell 26).  This is the reference's code path, not a
        # fallback of the accelerated one: solver="mu", init="random" never comes here (unless engine="sklearn").
        if n_restarts != 1:
            raise ValueError("n_restarts is an extension of the batched mu solver; scikit-learn runs one initialisation")
        return _find_synergies_sklearn(processed_emg_df, n_components, max_components, max_iter=max_iter, tol=tol,
                                       **sklearn_kwargs)
    if seed is None:
        seed = int(np.random.randint(0, 2**31 - 1))
    ranks_sweep = [n_components] if max_components is None else list(range(n_components, max_components + 1))
    ranks = [k for k in ranks_sweep for _ in range(n_restarts)]
    seeds = [int(seed) + r for _ in ranks_sweep for r in range(n_restarts)]
    X = processed_emg_df.to_numpy(dtype=np.float64)
    res = nmf_mu_batched(X, ranks, seeds, max_iter=max_iter, tol=tol)
    return _synergy_result(processed_emg_df, max_components, ranks_sweep, n_restarts, {k: (res, i * n_restarts)
                           for i, k in enumerate(ranks_sweep)}, "mu", {k: "random" for k in ranks_sweep}, max_iter, tol)


def _synergy_result(processed_emg_df, max_components, ranks_sweep, n_restarts, batches, solver, inits, max_iter, tol,
                    beta_loss="frobenius"):
    """The SynergyRunResult of a sweep whose rank k has n_restarts consecutive problems in batch batches[k][0],
    starting at problem batches[k][1]: per rank, the restart with the smallest reconstruction error (the
    square-rooted β-divergence for beta_loss != "frobenius")."""
    num_features = len(processed_emg_df.columns)
    columns = processed_emg_df.columns
    labels = ["All signals"] + columns.tolist()
    per_rank = OrderedDict()
    for k in ranks_sweep:
        res, first = batches[k]
        sl = slice(first, first + n_restarts)
        best = first + int(np.argmin(res.err[sl]))
        table = pandas.DataFrame(res.vaf[sl].astype(np.float64), columns=labels)
        table.insert(0, "reconstruction_err", res.err[sl].astype(np.float64))
        table.insert(0, "n_iter", res.n_iter[sl])
        table.insert(0, "random_state", res.seeds[sl])
        seed = int(res.seeds[best])
        model = NMFModel(k, res.H[best].astype(np.float64), int(res.n_iter[best]), float(res.err[best]),
                         num_features, seed if seed >= 0 else None, solver=solver, beta_loss=beta_loss, init=inits[k],
                         restarts=table, max_iter=max_iter, tol=tol)
        transformed = res.W[best].astype(np.float64)
        comps = pandas.DataFrame(model.components_, columns=columns)
        vaf_values = vaf(processed_emg_df, components=model.components_, transformed_signal=transformed)
        per_rank[k] = SynergyRunResult(vaf_values, comps, model, transformed)
    if max_components is None:
        return per_rank[ranks_sweep[0]]
    vaf_values = pandas.concat([r.vaf_values for r in per_rank.values()])
    vaf_values.set_index(np.array(tuple(per_rank.keys())), inplace=True)
    return SynergyRunResult(
        vaf_values,
        {k: r.components for k, r in per_rank.items()},
        {k: r.model for k, r in per_rank.items()},
        {k: r.transformed for k, r in per_rank.items()},
    )


def _find_synergies_gpu(df, n_components, max_components, max_iter, tol, n_restarts, sklearn_kwargs):
    """find_synergies(engine="gpu"): the configurations the kernels implement, every other one refused by name."""
    kw = dict(sklearn_kwargs)
    solver = kw.pop("solver", "cd")
    init = kw.pop("init", None)
    beta_loss = kw.pop("beta_loss", "frobenius")
    seed = kw.pop("random_state", None)
    for name, default in _SKLEARN_DEFAULTS.items():
        if name in kw and kw[name] == default and type(kw[name]) is type(default):
            del kw[name]
    if kw:
        raise NotImplementedError(f"find_synergies(engine='gpu') does not implement {', '.join(f'{k}={v!r}' for k, v in kw.items())}")
    if solver not in ("cd", "mu"):
        raise NotImplementedError(f"find_synergies(engine='gpu') does not implement solver={solver!r}")
    if init not in (None, "nndsvd", "nndsvda", "random"):
        raise NotImplementedError(f"find_synergies(engine='gpu') does not implement init={init!r}")
    try:
        beta = _beta_to_float(beta_loss)
    except ValueError:
        raise NotImplementedError(f"find_synergies(engine='gpu') does not implement beta_loss={beta_loss!r}") from None
    if beta != 2.0:
        if solver != "mu":
            raise _beta_solver_error(solver, beta_loss)
        if init == "nndsvd":
            warnings.warn("The multiplicative update ('mu') solver cannot update zeros present in the initialization, "
                          "and so leads to poorer results when used jointly with init='nndsvd'. You may try "
                          "init='nndsvda' or init='nndsvdar' instead.", UserWarning)
    n, m = df.shape
    ranks_sweep = [n_components] if max_components is None else list(range(n_components, max_components + 1))
    inits = {k: init if init is not None else ("nndsvda" if k <= min(n, m) else "random") for k in ranks_sweep}
    if n_restarts < 1:
        raise ValueError("n_restarts must be positive")
    if n_restarts > 1 and any(v != "random" for v in inits.values()):
        raise ValueError("n_restarts > 1 needs init='random': an nndsvd init is deterministic")
    if any(v == "random" for v in inits.values()) and seed is None:
        seed = int(np.random.randint(0, 2**31 - 1))
    X = df.to_numpy(dtype=np.float64)
    batches = {}
    for how in sorted(set(inits.values())):  # one launch per init kind (a sweep mixes them only when n < k)
        group = [k for k in ranks_sweep if inits[k] == how]
        ranks = [k for k in group for _ in range(n_restarts)]
        seeds = [int(seed) + r for _ in group for r in range(n_restarts)] if how == "random" else None
        if beta != 2.0:
            res = nmf_beta_batched(X, ranks, beta_loss, init=how, seeds=seeds, max_iter=max_iter, tol=tol)
        elif solver == "cd":
            res = nmf_cd_batched(X, ranks, init=how, seeds=seeds, max_iter=max_iter, tol=tol)
        elif how == "random":
            res = nmf_mu_batched(X, ranks, seeds, max_iter=max_iter, tol=tol)
        else:  # mu from the device's NNDSVD init
            start = nmf_cd_batched(X, ranks, init=how, max_iter=0, tol=0.0)
            res = nmf_mu_batched(X, ranks, np.full(len(ranks), -1), max_iter=max_iter, tol=tol,
                                 init=[(start.W[p], start.H[p]) for p in range(len(ranks))])
        if tol > 0 and (res.n_iter == max_iter).any():
            from sklearn.exceptions import ConvergenceWarning

            warnings.warn("Maximum number of iterations %d reached. Increase it to improve convergence." % max_iter,
                          ConvergenceWarning)
        batches.update({k: (res, i * n_restarts) for i, k in enumerate(group)})
    return _synergy_result(df, max_components, ranks_sweep, n_restarts, batches, solver, inits, max_iter, tol,
                           beta_loss if beta != 2.0 else "frobenius")
