"""Trial -> gait cycles -> envelopes -> synergies, without leaving the GPU (BASELINE configs[4]).

The flow of the reference's tutorial "Finding muscle synergies" (docs/source/tutorials, cells
4-30) applied per gait cycle, as SURVEY.md section 8d configs[4] spells it out:

    data = load_vicon_file(f)                       load_csv.py:96-135          (ms_scan + ms_parse)
    seg = Segmenter(data)                           project/segment.py:124-298  (ms_find_transitions)
    for each trecho, cycle:
        emg = data.emg[seg.get_times_of(trecho, cycle)]                          (window bounds only)
        env = normalize(time_normalize(rms(zero_center(emg), 0.5 s), 200))       analysis.py:230-594
        find_synergies(env, 1, 8, solver="mu", init="random", random_state=s)    analysis.py:713-914

Here the envelope is computed once per trial (zero-centred moving RMS over the whole recording,
then every cycle is resampled and amplitude-normalised - `emg.envelope_windows`) and all
cycles x ranks x restarts run as ONE launch of the batched NMF kernel on the device-resident
envelopes.  This module is an extension: the reference has no batch entry point.
"""
from collections.abc import Mapping
from dataclasses import dataclass, field
from typing import Dict, Iterable, List, Optional, Sequence, Tuple, Union

import numpy as np
import pandas

from .analysis import NMFBatchResult, match_synergies_batched, nmf_cd_batched, nmf_mu_batched, nmf_transform_batched
from .emg import envelope_windows
from .segment import Cycle, Segmenter, Trecho
from .vicon_data import ViconLoader, ViconNexusData


class _Frames(Mapping):
    """rank -> DataFrame, built from the array on first access (a trial has 64 of these; building
    them eagerly costs more host time than the GPU spends on the whole trial)."""

    def __init__(self, arrays: Dict[int, np.ndarray], columns):
        self._arrays, self._columns, self._frames = arrays, columns, {}

    def __getitem__(self, k):
        if k not in self._frames:
            self._frames[k] = pandas.DataFrame(self._arrays[k].astype(np.float64), columns=self._columns)
        return self._frames[k]

    def __iter__(self):
        return iter(self._arrays)

    def __len__(self):
        return len(self._arrays)


@dataclass
class CycleSynergies:
    """Synergies of one gait cycle: per rank, the restart with the smallest reconstruction error."""

    trecho: Trecho
    cycle: Cycle
    window: slice  # (frame, subframe) slice, as Segmenter.get_times_of returns it
    components: Mapping  # rank -> (rank x muscles) DataFrame of synergy vectors
    transformed: Dict[int, np.ndarray]  # rank -> (reduce_to x rank) activations
    n_iter: Dict[int, int]
    reconstruction_err: Dict[int, float]
    random_state: Dict[int, int]
    _vaf: np.ndarray = field(repr=False, default=None)  # (ranks, 1 + muscles)
    _labels: list = field(repr=False, default=None)
    _vaf_frame: Optional[pandas.DataFrame] = field(repr=False, default=None)

    @property
    def vaf_values(self) -> pandas.DataFrame:
        """index: rank; columns: "All signals" + muscles (the table of analysis.py:884-894)."""
        if self._vaf_frame is None:
            self._vaf_frame = pandas.DataFrame(self._vaf, columns=self._labels, index=np.array(list(self.components)))
        return self._vaf_frame


@dataclass
class TrialSynergies:
    cycles: List[CycleSynergies]
    envelopes: object = field(repr=False, default=None)  # (n_cycles, reduce_to, muscles) float64 CUDA tensor
    batch: Optional[NMFBatchResult] = field(repr=False, default=None)
    _restart_columns: dict = field(repr=False, default=None)
    _restarts: Optional[pandas.DataFrame] = field(repr=False, default=None)

    @property
    def restarts(self) -> pandas.DataFrame:
        """One row per (trecho, cycle, rank, restart): seed, n_iter, reconstruction error, overall VAF."""
        if self._restarts is None:
            self._restarts = pandas.DataFrame(self._restart_columns)
        return self._restarts

    def __getitem__(self, key: Tuple[Trecho, Cycle]) -> CycleSynergies:
        trecho, cycle = Segmenter._parse_trecho(key[0]), Segmenter._parse_cycle(key[1])
        for c in self.cycles:
            if c.trecho is trecho and c.cycle is cycle:
                return c
        raise KeyError(key)


def cycle_windows(segmenter: Segmenter) -> List[Tuple[Trecho, Cycle, slice]]:
    """The 4 trechos x 2 cycles of a trial, each first.start .. fourth.stop (segment.py:221-232)."""
    return [(t, c, segmenter.get_times_of(t, c)) for t in Trecho for c in Cycle]


class PendingTrial:
    """A trial whose GPU work (segmentation, envelopes, the NMF launch, the copies of its results) is queued:
    `finish()` waits for it and builds the TrialSynergies on the host."""

    def __init__(self, finish):
        self._finish, self._done = finish, None

    def finish(self) -> "TrialSynergies":
        if self._done is None:
            self._done = self._finish()
            self._finish = None
        return self._done


def _deterministic(solver: str, init: Optional[str]) -> bool:
    """True when trial_synergies(solver, init) starts from the deterministic NNDSVD init (one run per problem)."""
    if solver == "mu":
        if init not in (None, "random"):
            raise ValueError(f"solver='mu' runs from init='random', not {init!r}")
        return False
    if solver != "cd":
        raise ValueError(f"solver must be 'mu' or 'cd', not {solver!r}")
    if init not in (None, "nndsvd", "nndsvda", "random"):
        raise ValueError(f"solver='cd' runs from init 'nndsvd', 'nndsvda' or 'random', not {init!r}")
    return init != "random"


def trial_synergies(data: ViconNexusData, min_components: int = 1, max_components: int = 8,
                    n_restarts: Optional[int] = None, random_state: int = 0, max_iter: int = 200, tol: float = 1e-4,
                    window_size: float = 0.5, reduce_to: int = 200, segmenter: Optional[Segmenter] = None,
                    keep_batch: bool = False, seeds: Optional[Sequence[int]] = None, defer: bool = False,
                    solver: str = "mu", init: Optional[str] = None) -> Union[TrialSynergies, PendingTrial]:
    """Segments a loaded trial and factorises the EMG envelope of each of its 8 gait cycles for
    every rank in [min_components, max_components] from `n_restarts` random initialisations
    (default 20; seeds random_state .. random_state + n_restarts - 1, sklearn `init="random"` draws; `seeds` names
    them explicitly instead - the share of one GPU when the restarts of a trial are split over several).
    solver="mu" (fp32 multiplicative updates, `nmf_mu_batched`) or "cd" (sklearn's default coordinate descent, fp64,
    `nmf_cd_batched`); under "cd", init defaults to "nndsvda", and a deterministic init ("nndsvd", "nndsvda") runs
    one problem per cycle and rank: it takes exactly one seed (n_restarts 1, the default there), which only labels it.
    defer=True queues the GPU work and returns a PendingTrial: the caller can queue the next trial before it
    asks this one to `finish()` (the host-side tables of one trial are then built while the GPU factorises the next)."""
    muscles = data.emg.columns
    if not 1 <= min_components <= max_components <= len(muscles):
        raise ValueError("invalid number of components")
    deterministic = _deterministic(solver, init)
    if n_restarts is None:
        n_restarts = 1 if deterministic else 20
    seed_list = np.arange(random_state, random_state + n_restarts, dtype=np.int64) if seeds is None else np.asarray(list(seeds), dtype=np.int64)
    n_restarts = int(seed_list.shape[0])
    if n_restarts < 1:
        raise ValueError("n_restarts must be positive")
    if deterministic and n_restarts != 1:
        raise ValueError("a deterministic init (nndsvd, nndsvda) takes exactly one seed")
    seg = segmenter if segmenter is not None else Segmenter(data)
    wins = cycle_windows(seg)
    env = envelope_windows(data.emg, [w for (_, _, w) in wins], window_size=window_size, reduce_to=reduce_to)
    sweep = list(range(min_components, max_components + 1))
    n_cyc, n_k = len(wins), len(sweep)
    # problem order: cycle-major, then rank, then restart
    ranks = np.tile(np.repeat(np.array(sweep, dtype=np.int32), n_restarts), n_cyc)
    seeds = np.tile(seed_list, n_cyc * n_k)
    x_index = np.repeat(np.arange(n_cyc, dtype=np.int32), n_k * n_restarts)
    if solver == "cd":
        pending = nmf_cd_batched(env, ranks, init=init or "nndsvda", seeds=seeds, max_iter=max_iter, tol=tol,
                                 x_index=x_index, defer=True)
    else:
        pending = nmf_mu_batched(env, ranks, seeds, max_iter=max_iter, tol=tol, x_index=x_index, defer=True)

    def finish() -> TrialSynergies:
        return _trial_tables(pending.result(), data, wins, sweep, n_restarts, ranks, seeds, muscles, env, keep_batch)

    return PendingTrial(finish) if defer else finish()


def _trial_tables(res, data, wins, sweep, n_restarts, ranks, seeds, muscles, env, keep_batch) -> TrialSynergies:
    n_cyc, n_k = len(wins), len(sweep)
    labels = ["All signals"] + muscles
    err = res.err.reshape(n_cyc, n_k, n_restarts)
    best = err.argmin(axis=2)
    cycles = []
    for ci, (trecho, cycle, window) in enumerate(wins):
        rows, comps, acts, iters, errs, rstate = [], {}, {}, {}, {}, {}
        for ki, k in enumerate(sweep):
            p = (ci * n_k + ki) * n_restarts + int(best[ci, ki])
            rows.append(res.vaf[p].astype(np.float64))
            comps[k] = res.H[p]
            acts[k] = res.W[p].astype(np.float64)
            iters[k], errs[k], rstate[k] = int(res.n_iter[p]), float(res.err[p]), int(res.seeds[p])
        cycles.append(CycleSynergies(trecho, cycle, window, _Frames(comps, muscles), acts, iters, errs, rstate,
                                     np.array(rows), labels))
    restart_columns = {
        "trecho": np.repeat([t.value for (t, _, _) in wins], n_k * n_restarts),
        "cycle": np.repeat([c.value for (_, c, _) in wins], n_k * n_restarts),
        "n_components": ranks,
        "random_state": seeds,
        "n_iter": res.n_iter,
        "reconstruction_err": res.err.astype(np.float64),
        "All signals": res.vaf[:, 0].astype(np.float64),
    }
    return TrialSynergies(cycles, env, res if keep_batch else None, restart_columns)


def cross_cycle_vaf(trial: TrialSynergies, ranks: Optional[Sequence[int]] = None, solver: str = "cd",
                    max_iter: int = 100_000, tol: float = 1e-6) -> pandas.DataFrame:
    """How well each cycle's synergies generalise to the other cycles of the trial: for every rank, every cycle's
    envelope (`trial.envelopes`, on the device) is fitted with every cycle's synergies held fixed (sklearn's
    `NMF.transform` with `solver`, `max_iter`, `tol`), all ranks x sources x targets in one launch.  Returns the overall
    VAF; index (n_components, source trecho, source cycle), columns (target trecho, target cycle)."""
    cycles = trial.cycles
    ranks = list(cycles[0].components) if ranks is None else [int(k) for k in ranks]
    n_cyc = len(cycles)
    H = [cycles[s].components[k].to_numpy(dtype=np.float64) for k in ranks for s in range(n_cyc) for _ in range(n_cyc)]
    x_index = np.tile(np.arange(n_cyc, dtype=np.int32), len(ranks) * n_cyc)
    res = nmf_transform_batched(trial.envelopes, H, x_index=x_index, solver=solver, max_iter=max_iter, tol=tol)
    index = pandas.MultiIndex.from_tuples([(k, c.trecho.value, c.cycle.value) for k in ranks for c in cycles],
                                          names=["n_components", "trecho", "cycle"])
    columns = pandas.MultiIndex.from_tuples([(c.trecho.value, c.cycle.value) for c in cycles], names=["trecho", "cycle"])
    return pandas.DataFrame(res.vaf[:, 0].reshape(len(ranks) * n_cyc, n_cyc), index=index, columns=columns)


def synergy_similarity(trial: TrialSynergies, ranks: Optional[Sequence[int]] = None) -> pandas.DataFrame:
    """How alike the synergies of the trial's cycles are: for every rank, every pair of cycles' synergy sets (the best
    restart's `components`) is compared by matched cosine similarity (`match_synergies_batched`: unit-length synergy
    vectors, optimal one-to-one pairing, mean of the matched similarities), all ranks x pairs in one launch.  The
    companion of `cross_cycle_vaf`, in its layout: index (n_components, source trecho, source cycle), columns (target
    trecho, target cycle).  Pairs a < b are computed and mirrored, so the table is exactly symmetric; the diagonal is
    computed too."""
    cycles = trial.cycles
    ranks = list(cycles[0].components) if ranks is None else [int(k) for k in ranks]
    n_cyc = len(cycles)
    H = [c.components[k].to_numpy(dtype=np.float64) for k in ranks for c in cycles]
    a, b = np.triu_indices(n_cyc)
    pairs = np.concatenate([np.stack([a, b], axis=1) + r * n_cyc for r in range(len(ranks))])
    mean = match_synergies_batched(H, pairs).mean.reshape(len(ranks), -1)
    table = np.empty((len(ranks), n_cyc, n_cyc))
    table[:, a, b] = mean
    table[:, b, a] = mean
    index = pandas.MultiIndex.from_tuples([(k, c.trecho.value, c.cycle.value) for k in ranks for c in cycles],
                                          names=["n_components", "trecho", "cycle"])
    columns = pandas.MultiIndex.from_tuples([(c.trecho.value, c.cycle.value) for c in cycles], names=["trecho", "cycle"])
    return pandas.DataFrame(table.reshape(len(ranks) * n_cyc, n_cyc), index=index, columns=columns)


def synergies_for_files(paths: Sequence[str], loader: Optional[ViconLoader] = None, **kwargs) -> Iterable[Tuple[str, TrialSynergies]]:
    """`trial_synergies` over a list of trial files; the next file is read and uploaded while the
    current one is analysed (ViconLoader.load_files).  Yields (path, TrialSynergies) in order; a
    file that fails to load or to segment yields (path, exception) instead."""
    loader = loader if loader is not None else ViconLoader()
    caught = (ValueError, IndexError, KeyError)  # e.g. fewer than 40 transitions in the trial

    def finished(item):
        path, pending = item
        if isinstance(pending, Exception):
            return path, pending
        try:
            return path, pending.finish()
        except caught as exc:
            return path, exc

    # one trial deep: the GPU work of trial i is queued before the host looks at the results of trial i - 1.  The loader
    # kernel of a trial runs on the loader's pipeline streams and its transition search on the loader's high-priority
    # work stream - beside the factorisation of the trial before it, which fills the compute stream for milliseconds -
    # so that the envelopes and the NMF launch of trial i are queued while trial i - 1 is still being factorised.
    import torch

    work = loader.work_stream
    prev = None
    for path, data in loader.load_files(paths, to_host=False):
        if isinstance(data, Exception):
            cur = (path, data)
        else:
            try:
                seg = kwargs.get("segmenter")
                if seg is None:
                    with torch.cuda.stream(work):
                        for blk in data.blocks or ():
                            if blk is not None and blk.tensor is not None:
                                blk.tensor.record_stream(work)
                        seg = Segmenter(data)
                cur = (path, trial_synergies(data, defer=True, **dict(kwargs, segmenter=seg)))
            except caught as exc:
                cur = (path, exc)
        if prev is not None:
            yield finished(prev)
        prev = cur
    if prev is not None:
        yield finished(prev)


# ---- several GPUs: one process per GPU, no collective on the data path (SURVEY.md section 8e) ---------------------
def best_restart_table(path: str, trial: TrialSynergies) -> List[dict]:
    """The small per-trial result that travels between ranks: for every (cycle, rank) the best restart's seed,
    iteration count, reconstruction error and VAF row ("All signals" + muscles; analysis.py:642-667)."""
    rows = []
    for c in trial.cycles:
        for i, k in enumerate(c.components):
            rows.append({"file": path, "trecho": c.trecho.value, "cycle": c.cycle.value, "n_components": int(k),
                         "random_state": c.random_state[k], "n_iter": c.n_iter[k],
                         "reconstruction_err": c.reconstruction_err[k], "vaf": np.asarray(c._vaf[i], dtype=np.float64)})
    return rows


def merge_tables(tables: Iterable[List[dict]]) -> List[dict]:
    """Union of the ranks' tables; where several ranks hold the same (file, cycle, rank) - a trial whose restarts
    were split over the GPUs - the restart with the smallest reconstruction error wins (ties: smallest seed)."""
    best = {}
    for table in tables:
        for row in table:
            if "error" in row:
                best.setdefault((row["file"], "error"), row)
                continue
            key = (row["file"], row["trecho"], row["cycle"], row["n_components"])
            cur = best.get(key)
            if cur is None or (row["reconstruction_err"], row["random_state"]) < (cur["reconstruction_err"], cur["random_state"]):
                best[key] = row
    return [best[k] for k in sorted(best, key=lambda k: tuple(str(x) for x in k))]


def synergies_for_files_sharded(paths: Sequence[str], rank: Optional[int] = None, world: Optional[int] = None,
                                loader: Optional[ViconLoader] = None, gather: bool = True, analyse=None,
                                n_restarts: int = 20, random_state: int = 0, **kwargs) -> List[dict]:
    """`synergies_for_files` over the GPUs of one box.  Work is split with no exchange on the data path:

      * at least as many files as GPUs: by file, balanced by size (`sharding.shard`); every rank loads, segments
        and factorises its own trials;
      * fewer files than GPUs: by (rank, restart) - every rank loads every file and runs the restarts
        r with r % world == rank (the envelopes are recomputed rather than moved: a trial loads in
        milliseconds, and nothing crosses NVLink).

    Then ONE host-side gather of the small result tables (`sharding.gather_results`, torch.distributed object
    gather) and the best-of-restarts merge.  Returns, on every rank, the merged table: one dict per (file, trecho,
    cycle, n_components), or {"file", "error"} for a file that failed.  rank / world default to the process group's;
    `analyse(paths, **kw)` is the per-file generator (default `synergies_for_files`; tests inject a CPU stand-in)."""
    import os

    from .sharding import gather_results, shard

    if rank is None or world is None:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
        else:
            rank, world = 0, 1
    paths = [str(p) for p in paths]
    analyse = analyse if analyse is not None else synergies_for_files
    if _deterministic(kwargs.get("solver", "mu"), kwargs.get("init")):
        # one run per (cycle, rank) and no restarts to split: by file, and with fewer files than GPUs the ranks that
        # get no seed below have nothing to do
        n_restarts = 1
    if len(paths) >= world:
        sizes = [os.path.getsize(p) if os.path.exists(p) else 0 for p in paths]
        mine = shard(paths, rank, world, sizes)
        seeds = list(range(random_state, random_state + n_restarts))
    else:
        mine = paths
        seeds = [random_state + r for r in range(n_restarts) if r % world == rank]
    table: List[dict] = []
    if mine and seeds:
        kw = dict(kwargs)
        if loader is not None:
            kw["loader"] = loader
        for path, result in analyse(mine, seeds=seeds, **kw):
            if isinstance(result, Exception):
                table.append({"file": path, "error": f"{type(result).__name__}: {result}"})
            else:
                table += best_restart_table(path, result)
    if not gather:
        return table
    return merge_tables(gather_results(table))
