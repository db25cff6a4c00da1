"""CPU (gloo, world_size 2): the exchange of the sharded SIF sweep (sif_dist.exchange_sweep_).  The kernels
need a GPU; what is checked here is the host logic: the stacked K Grams summed in one exchange equal the per-k
sums, the stacked K x P start blocks of the N < d case equal X_k^T Omega_npc of the global matrices, and the
grouping of the peer path (whole Grams per exchange slot, start blocks in slot-sized pieces) gives the same
result as one all-reduce of each stack."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NPCS = (0, 1, 3)


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _data(K, n_global, d):
    rng = np.random.default_rng(3)
    return rng.standard_normal((K, n_global, d)).astype(np.float32)         # same on every rank


class _GlooComm(object):
    """Stands in for PeerComm: the same in-place allreduce_ (and its slot limit), over gloo."""

    def __init__(self, slot_bytes):
        self.slot_bytes, self.sizes = slot_bytes, []

    def allreduce_(self, t):
        assert t.is_contiguous() and t.numel() * t.element_size() <= self.slot_bytes
        self.sizes.append(t.numel())
        dist.all_reduce(t)
        return t


def _worker(rank, world, port, K, n_global, d, slots, q):
    sys.path.insert(0, os.path.join(ROOT, 'multimodal-baselines_b200'))
    sys.path.insert(0, ROOT)
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import sif_dist
    from oracle import sif_oracle as so
    X = _data(K, n_global, d)
    lo, hi = sif_dist.shard_bounds(n_global, world, rank)
    Xl = torch.as_tensor(X[:, lo:hi])

    def local():
        G = torch.stack([Xl[k].T @ Xl[k] for k in range(K)]).contiguous()
        S0 = [Xl[k].double().T @ torch.as_tensor(sif_dist.local_omega_rows(n_global, lo, hi - lo, p, so.start_block))
              for k in range(K) for p in NPCS if p] if n_global < d else []
        return G, S0

    per_k = []
    for k in range(K):                                    # today's sharded path: one all-reduce per k
        G = (Xl[k].T @ Xl[k]).contiguous()
        sif_dist.allreduce_sum_(G)
        per_k.append(G)
    G, S0 = local()
    sif_dist.exchange_sweep_(G, S0)                        # torch.distributed: one all-reduce per stack
    res = {'per_k': torch.stack(per_k).numpy(), 'G': G.numpy(), 'S0': [b.numpy() for b in S0], 'peer': []}
    for slot in slots:                                     # the peer path's grouping
        comm = _GlooComm(slot)
        Gp, S0p = local()
        sif_dist.exchange_sweep_(Gp, S0p, comm=comm, slot_bytes=slot)
        res['peer'].append((slot, comm.sizes, Gp.numpy(), [b.numpy() for b in S0p]))
    q.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


def _run(K, n_global, d, slots):
    world = 2
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, K, n_global, d, slots, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in range(world)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return [r[1] for r in res]


@pytest.mark.parametrize('K,n_global,d', [(3, 157, 300), (12, 157, 300), (12, 700, 300)])
def test_stacked_exchange_equals_per_k_sums(K, n_global, d):
    sys.path.insert(0, ROOT)
    from oracle import sif_oracle as so
    slot = 4 * 1024 * 1024                                  # mmb_comm_slot_bytes(); checked on the GPU
    res = _run(K, n_global, d, slots=(slot, 400_000))        # 400 KB: one Gram per exchange, S0 in pieces
    X = _data(K, n_global, d).astype(np.float64)
    for r in res:
        np.testing.assert_array_equal(r['G'], r['per_k'])      # one exchange of the stack == K exchanges
        for k in range(K):
            np.testing.assert_allclose(r['G'][k], X[k].T @ X[k], rtol=1e-4, atol=1e-3)
        want_S0 = [X[k].T @ so.start_block(n_global, p) for k in range(K) for p in NPCS if p] if n_global < d else []
        assert len(r['S0']) == len(want_S0)
        for got, want in zip(r['S0'], want_S0):
            np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-9)
        for slot_bytes, sizes, G, S0 in r['peer']:
            per = slot_bytes // (4 * d * d)                      # whole Grams per exchange: 11 at d = 300
            grams = [min(per, K - k) * d * d for k in range(0, K, per)]
            assert sizes[:len(grams)] == grams
            s0_elems = sum(b.size for b in want_S0)
            assert sum(sizes[len(grams):]) == s0_elems and all(s * 8 <= slot_bytes for s in sizes[len(grams):])
            np.testing.assert_array_equal(G, r['G'])
            for a, b in zip(S0, r['S0']):
                np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(res[0]['G'], res[1]['G'])     # every rank solves on the same bits
    if K == 12:
        assert res[0]['peer'][0][1][:2] == [11 * d * d, d * d]     # K > 11: two Gram exchanges
