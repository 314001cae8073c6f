"""CPU, world_size 2, gloo: the N > 1 path's host logic -- shard bounds, ragged all-gather, gathered
masks / first-failure / IK sets equal to the single-process result.  Per-rank compute is the CPU oracle
(injected), so what is tested is sharding + collectives, not arithmetic."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import ik_reference as ref
import oracle
from conftest import sample_edges, sample_states

from torque_constrained_motion_planning_b200 import distributed as D


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _oracle_tt(q, qd, qdd, pm, mode="rne", want_tau=False, **kw):
    t = lambda a: None if a is None else (a.numpy() if torch.is_tensor(a) else a)
    _, ok = oracle.torque_test_batch(mode, t(q), t(qd), t(qdd), t(pm) if np.ndim(pm) else pm)
    return None, torch.as_tensor(ok)


def _oracle_edge(qa, qb, W, mass, mode="rne", **kw):
    t = lambda a: a.numpy() if torch.is_tensor(a) else a
    return torch.as_tensor(oracle.edge_feasibility(mode, t(qa), t(qb), W, mass))


def _oracle_ik(r, t, f):
    n = lambda a: a.numpy() if torch.is_tensor(a) else a
    sols, counts, _ = ref.host_ik(n(r), n(t), n(f))
    return torch.as_tensor(sols), torch.as_tensor(counts)


def _worker(rank, world, port, n_states, n_edges, n_poses, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        s_q, s_qd, s_qdd, s_m = sample_states(n_states, seed=2)
        mask, (lo, hi) = D.sharded_torque_test(s_q, s_qd, s_qdd, s_m, mode="rne", compute=_oracle_tt)
        _, full = oracle.torque_test_batch("rne", s_q, s_qd, s_qdd, s_m)
        assert (lo, hi) == D.shard_bounds(n_states, rank, world)
        assert np.array_equal(mask.numpy(), full)
        qa, qb = sample_edges(n_edges, seed=4)
        ff, _ = D.sharded_edge_feasibility(qa, qb, 16, 5.0, compute=_oracle_edge)
        assert np.array_equal(ff.numpy(), oracle.edge_feasibility("rne", qa, qb, 16, 5.0))
        rng = np.random.default_rng(3)
        qq = rng.uniform(-2.5, 2.5, size=(7, n_poses)); qq[3] = -np.abs(qq[3]) - 0.1; qq[5] = np.abs(qq[5])
        trans, rot = ref.fk_batch(qq)
        free = np.stack([qq[6], rng.uniform(-2.8, 2.8, n_poses)])
        sols, counts, _ = D.sharded_ik(rot, trans, free, compute=_oracle_ik)
        s_full, c_full, _ = ref.host_ik(rot, trans, free)
        assert np.array_equal(counts.numpy(), c_full) and np.array_equal(sols.numpy(), s_full)
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        q.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def test_shard_bounds_cover_everything():
    for n in [0, 1, 7, 100, 1_000_003]:
        for world in [1, 2, 3, 8]:
            blocks = [D.shard_bounds(n, r, world) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in blocks]
            assert max(sizes) - min(sizes) <= 1


@pytest.mark.timeout(180)
def test_world_size_2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, 1001, 37, 51, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=150) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    assert sorted(results) == [(0, "ok"), (1, "ok")], results
