"""Run a per-tensor task over the GPUs of one node: one spawned worker process per GPU, no collective.

The items (tensor names) are bin-packed over the workers by element count (``sharding.partition_tensors``: LPT,
deterministic).  Worker i pins itself to cuda:i before any CUDA work and runs the task over its items in name order; each
item's result (any picklable object) comes back to the parent over a queue, and the parent yields the results in the
original item order as soon as each prefix of that order is complete.  The parent itself does no CUDA work, so it holds no
memory on GPU 0.  `wq --gpus N` and `sweep_cli --gpus N` run on this.
"""
from __future__ import annotations

import multiprocessing as mp
import queue
import signal
import traceback

from .sharding import partition_tensors

POLL_S = 0.5


class ShardError(RuntimeError):
    """An item's task raised in a worker, or a worker exited before it returned all its results."""


def gpu_count_error(gpus: int) -> str | None:
    """Why ``--gpus gpus`` cannot run on this node, or None.  The visible devices are the ones CUDA_VISIBLE_DEVICES leaves;
    with none there is nothing to run on (no CPU fallback)."""
    import torch
    visible = torch.cuda.device_count()
    if 1 <= gpus <= visible:
        return None
    return f"--gpus {gpus}: N must be between 1 and the number of visible CUDA devices, which is {visible}"


def _worker(rank: int, task, ctx, names: list[str], q) -> None:
    signal.signal(signal.SIGINT, signal.SIG_IGN)            # Ctrl-C is the parent's: it terminates the workers
    import torch
    torch.cuda.set_device(rank)
    for name in names:
        try:
            result = task(ctx, name)
        except Exception as exc:
            traceback.print_exc()
            q.put((rank, name, f"{type(exc).__name__} on cuda:{rank}: {exc}", None))
            return
        q.put((rank, name, None, result))


def merge_in_order(names: list[str], messages):
    """(name, result) in `names` order from ``(name, error, result)`` messages that arrive in any order: each result as soon
    as the results of every earlier name have arrived.  A message with an error raises ShardError naming its item at once."""
    order = {n: i for i, n in enumerate(names)}
    pending = {}
    nxt = 0
    for name, error, result in messages:
        if error is not None:
            raise ShardError(f"{name}: {error}")
        pending[order[name]] = result
        while nxt in pending:
            yield names[nxt], pending.pop(nxt)
            nxt += 1


def _receive(procs: dict, q, expected: dict):
    """``(name, error, result)`` messages of the workers ({rank: process}) in arrival order, until every worker has sent the
    `expected` number of results."""
    got = dict.fromkeys(procs, 0)
    while got != expected:
        # read before waiting: a worker that had exited by then had already put everything it sent into the queue's pipe
        exited = {r: p.exitcode is not None for r, p in procs.items()}
        try:
            rank, name, error, result = q.get(timeout=POLL_S)
        except queue.Empty:
            for r, p in procs.items():
                if exited[r] and got[r] < expected[r]:
                    raise ShardError(f"the worker on cuda:{r} exited with code {p.exitcode} before returning {expected[r] - got[r]} "
                                     f"of its {expected[r]} results") from None
            continue
        got[rank] += 1
        yield name, error, result


def run_sharded(task, ctx, names: list[str], sizes: list[int], gpus: int):
    """Yield ``(name, task(ctx, name))`` for every name, in `names` order, computed on `gpus` GPUs.

    task: a module-level function (it is pickled by reference); ctx: a picklable object given to every call; sizes: the
    element count of each name, for the bin packing.  On a task exception or a worker death every worker is terminated and
    joined and ShardError is raised; on KeyboardInterrupt, or when the caller closes the generator early, every worker is
    terminated and joined too.  No worker outlives the generator: close it (``contextlib.closing``) when not exhausting it."""
    parts = [[names[i] for i in part] for part in partition_tensors(sizes, gpus)]
    spawn = mp.get_context("spawn")
    q = spawn.Queue()
    procs = {rank: spawn.Process(target=_worker, args=(rank, task, ctx, part, q), name=f"qa-cuda{rank}", daemon=True)
             for rank, part in enumerate(parts) if part}
    expected = {rank: len(parts[rank]) for rank in procs}
    started = []
    try:
        for p in procs.values():
            p.start()
            started.append(p)
        yield from merge_in_order(names, _receive(procs, q, expected))
    finally:
        for p in started:
            if p.is_alive():
                p.terminate()
        for p in started:
            p.join()
        q.close()
