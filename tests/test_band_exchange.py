"""The exchange interface of descriptools_b200/bands.py on CPU: LocalExchange (all bands in one process, 1 to 4 bands)
and DistExchange over torch.distributed (gloo, world sizes 2 and 3) pass the same checks of halo, handoff, all_sum,
broadcast, solve and local_bands."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

ROWS, COLS = 3, 7


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rows(i):
    """band i's rows, known to every process"""
    return torch.arange(ROWS * COLS, dtype=torch.int64).view(ROWS, COLS) + 1000 * (i + 1)


def _summaries(n, seed):
    """valid flow-accumulation and arbitrary HAND boundary summaries of n bands (the same in every process)"""
    g = torch.Generator().manual_seed(seed)
    shape = (n, 2, COLS)
    fa = torch.empty((n, 6, COLS), dtype=torch.int64)
    fa[:, 0:2] = torch.randint(0, 5, shape, generator=g)
    term = (torch.randint(0, 2, shape, generator=g) << 30) | torch.randint(0, COLS, shape, generator=g)
    fa[:, 2:4] = torch.where(torch.rand(shape, generator=g) < 0.2, torch.full_like(term, -2), term)
    fa[:, 4:6] = torch.tensor([1, 2, 4, 8, 16, 32, 64, 128])[torch.randint(0, 8, shape, generator=g)]
    hand = torch.randint(-(1 << 62), 1 << 62, (n, 8, COLS), generator=g, dtype=torch.int64)
    return fa, hand


def _check(x, n):
    """every check of the interface on exchange x of n bands, from this process's side"""
    from descriptools_b200 import bands

    mine = list(x.local_bands)
    assert x.nbands == n
    assert mine == (list(range(n)) if isinstance(x, bands.LocalExchange) else [x.rank])

    # halo: two rows on each side; the outer halos of the first and last band stay untouched
    data = {i: _rows(i) for i in mine}
    halos = {i: (torch.full((2, COLS), -1, dtype=torch.int64), torch.full((2, COLS), -1, dtype=torch.int64)) for i in mine}
    x.halo([(data[i][0:2], data[i][ROWS - 2:], *halos[i]) for i in mine])
    for i in mine:
        above, below = halos[i]
        assert torch.equal(above, _rows(i - 1)[ROWS - 2:] if i > 0 else torch.full((2, COLS), -1, dtype=torch.int64)), i
        assert torch.equal(below, _rows(i + 1)[0:2] if i + 1 < n else torch.full((2, COLS), -1, dtype=torch.int64)), i

    # handoff: every band sends its rows to every other band, adjacent or not
    pairs = [(s, d) for s in range(n) for d in range(n) if s != d]
    got = {(s, d): torch.zeros((ROWS, COLS), dtype=torch.int64) for s, d in pairs if d in mine}
    x.handoff([(s, d, data.get(s), got.get((s, d))) for s, d in pairs])
    for (s, d), t in got.items():
        assert torch.equal(t, _rows(s)), (s, d)

    # all_sum of a host tensor: the sum over the processes, back on the host
    t = x.all_sum(torch.tensor([sum(i + 1 for i in mine), len(mine)], dtype=torch.int64))
    assert t.device.type == "cpu"
    assert t.tolist() == [n * (n + 1) // 2, n]

    # broadcast: band i's rows from its holder to every process
    for i in range(n):
        t = _rows(i) if i in mine else torch.zeros((ROWS, COLS), dtype=torch.int64)
        x.broadcast(t, i)
        assert torch.equal(t, _rows(i)), i

    # solve: every process gets its own bands' rows of the solve over all bands, and the solve's flag
    fa, hand = _summaries(n, seed=n)
    for solver, summ in ((bands.solve_flowacc_boundary, fa), (bands.solve_hand_boundary, hand)):
        flags = len(x.flags)
        res = x.solve([summ[i].clone() for i in mine], solver)
        want, flag = solver(summ)
        assert len(res) == len(mine)
        for i, r in zip(mine, res):
            assert torch.equal(r, want[i]), (solver.__name__, i)
        assert len(x.flags) == flags + 1 and bool(x.flags[-1]) == bool(flag)


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_local_exchange(n):
    from descriptools_b200 import bands

    _check(bands.LocalExchange(n), n)


def _worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist

        dist.init_process_group("gloo", rank=rank, world_size=world)
        from descriptools_b200 import bands

        _check(bands.DistExchange(), world)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", None))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, "fail", traceback.format_exc()))


@pytest.mark.parametrize("world", [2, 3])
def test_dist_exchange_gloo(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in results:
        assert status == "ok", f"rank {rank}: {info}"
