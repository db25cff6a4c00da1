"""torchrun --nproc-per-node R tools/sif_sweep_dist_check.py : the utterance-sharded SIF sweep
(sif_dist.sharded_sif_embedding_sweep) against today's sharded single-vector path and the single-GPU sweep.

Per rank it prints one line per check and exits non-zero (on every rank) if any check fails:
  * bit identity, on the NVLink peer exchange, of out[k, j] with sharded_sif_embedding(W[k], npc=npcs[j]) for
    K in {1, 3, 12} (12 Grams need two exchange slots) and npcs = (0, 1, 3).  The shapes keep n_local L < 8 V and
    L < 256, so both embeds take the general warp kernel, and n_local >= 4096 puts the Gram on the tcgen05 path;
  * against the single-GPU sweep of all ids: npc = 0 slices bit-equal to rows [lo, hi), components cos > 1 - 1e-5,
    rows within 2e-5 relative (tools/dist_check.py's tolerances);
  * the components bit-identical on every rank;
  * peer exchange against NCCL (comm=None): cos > 1 - 1e-7, rows within 1e-6;
  * n_global < d (157 utterances), a rank with n_local = 0, and RaggedIds blocks against padded blocks;
  * a bad id in one rank's block: IndexError from its status word on that rank only, and every rank returns
    well inside the exchange's 4 s timeout.
"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'multimodal-baselines_b200'))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import _native as nv  # noqa: E402
import sif_dist  # noqa: E402
import sif_functions as sf  # noqa: E402

NPCS = (0, 1, 3)


def make_inputs(dev, n_global, L, V, K, d=300, seed=5):
    """The same table, weights and ids on every rank (seeded device generator)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    table = 0.4 * torch.randn((V, d), device=dev, generator=g) + 0.3 * torch.randn((1, d), device=dev, generator=g)
    table[0] = 0
    W = torch.rand((K, V), device=dev, generator=g) * 0.9 + 0.1
    ids = torch.randint(1, V, (n_global, L), device=dev, generator=g)
    lens = torch.randint(1, L + 1, (n_global, 1), device=dev, generator=g)
    ids[torch.arange(L, device=dev)[None, :] >= lens] = 0
    return table, W.contiguous(), ids


def same_bits(a, b):
    return a.shape == b.shape and bool(torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)))


def rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)) if b.numel() else 0.0


def cos(a, b):
    return float(torch.nn.functional.cosine_similarity(a.double(), b.double(), dim=1).min())


def gathered_equal(t):
    xs = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(xs, t.contiguous())
    return all(torch.equal(xs[0], x) for x in xs)


class Checker(object):
    def __init__(self, rank):
        self.rank, self.ok = rank, True

    def __call__(self, name, good, detail=''):
        self.ok = self.ok and bool(good)
        print('rank %d %s: %s -> %s' % (self.rank, name, detail, 'ok' if good else 'FAIL'), flush=True)


def against_single(chk, tag, out, pcs, table, W, ids_all, lo, hi, npcs):
    """The single-GPU sweep of all ids, rows [lo, hi): npc = 0 bit for bit, else dist_check.py's tolerances."""
    want = sf.sif_embedding_sweep(table, W, ids_all, npcs=npcs)
    K = W.shape[0]
    raw = all(same_bits(out[k, j], want[k, j, lo:hi]) for k in range(K) for j, p in enumerate(npcs) if p == 0)
    errs, coss = [0.0], [1.0]
    for k in range(K):
        want_pcs = None
        for j, p in enumerate(npcs):
            if p:
                errs.append(rel(out[k, j], want[k, j, lo:hi]))
                if want_pcs is None:
                    # the single-GPU sweep returns no components: solve them the same way from all rows
                    emb = sf.sweep_embed(table, W[k:k + 1].contiguous(), ids_all)[0]
                    G = sf.sweep_grams(emb)
                    want_pcs = {q: sf.pc_from_gram(G[0], q, ids_all.shape[0], X_t=emb[0]) for q in npcs if q}
                coss.append(cos(pcs[k][j], want_pcs[p]))
    chk(tag + ' vs single-GPU sweep', raw and max(errs) < 2e-5 and min(coss) > 1 - 1e-5,
        'npc=0 bit-equal %s, rows err %.2e, pc cos %.8f' % (raw, max(errs), min(coss)))


def check_case(chk, dev, world, rank, n_global, L, V, K, bounds=None, ragged=False, single=True, nccl=True):
    table, W, ids = make_inputs(dev, n_global, L, V, K)
    lo, hi = bounds if bounds is not None else sif_dist.shard_bounds(n_global, world, rank)
    ids_l = ids[lo:hi].contiguous()
    tag = 'N=%d K=%d n_local=%d' % (n_global, K, hi - lo)
    out, pcs, st = sif_dist.sharded_sif_embedding_sweep(table, W, ids_l, n_global, lo, npcs=NPCS)
    nv.raise_on_status(st, V)
    sif_dist.default_comm().check()
    # today's sharded path, one call per (k, npc), same peer exchange
    bits = True
    for k in range(K):
        for j, p in enumerate(NPCS):
            emb, pc, _ = sif_dist.sharded_sif_embedding(table, W[k].contiguous(), ids_l, n_global, lo, npc=p)
            bits = bits and same_bits(out[k, j], emb) and (p == 0 or same_bits(pcs[k][j], pc))
    chk(tag + ' vs sharded_sif_embedding', bits, 'bit-identical %s' % bits)
    reps = all(gathered_equal(pcs[k][j]) for k in range(K) for j, p in enumerate(NPCS) if p)
    chk(tag + ' replicas', reps, 'components identical on every rank %s' % reps)
    if single:
        against_single(chk, tag, out, pcs, table, W, ids, lo, hi, NPCS)
    if nccl:
        out_n, pcs_n, _ = sif_dist.sharded_sif_embedding_sweep(table, W, ids_l, n_global, lo, npcs=NPCS, comm=None)
        err = max(rel(out[k, j], out_n[k, j]) for k in range(K) for j in range(len(NPCS)))
        c = min(cos(pcs[k][j], pcs_n[k][j]) for k in range(K) for j, p in enumerate(NPCS) if p)
        chk(tag + ' peer vs NCCL', err < 1e-6 and c > 1 - 1e-7, 'rows err %.2e, pc cos %.9f' % (err, c))
    if ragged:
        out_r, pcs_r, st_r = sif_dist.sharded_sif_embedding_sweep(table, W, sf.to_ragged(ids_l), n_global, lo,
                                                                  npcs=NPCS)
        nv.raise_on_status(st_r, V)
        err = max(rel(out_r[k, j], out[k, j]) for k in range(K) for j in range(len(NPCS)))
        c = min(cos(pcs_r[k][j], pcs[k][j]) for k in range(K) for j, p in enumerate(NPCS) if p)
        chk(tag + ' RaggedIds vs padded', err < 1e-6 and c > 1 - 1e-7,
            'rows err %.2e, pc cos %.9f, bit-identical %s' % (err, c, same_bits(out_r, out)))


def check_bad_id(chk, dev, world, rank):
    """A bad id on the last rank only: that rank's status word raises IndexError, every rank returns at once."""
    n_global, L, V, K = 2000 * world, 32, 5000, 2
    table, W, ids = make_inputs(dev, n_global, L, V, K, seed=9)
    lo, hi = sif_dist.shard_bounds(n_global, world, rank)
    ids_l = ids[lo:hi].contiguous()
    if rank == world - 1:
        ids_l[3, 5] = V
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out, pcs, st = sif_dist.sharded_sif_embedding_sweep(table, W, ids_l, n_global, lo, npcs=(1, 2))
    try:
        nv.raise_on_status(st, V)
        raised = False
    except IndexError:
        raised = True
    dt = time.perf_counter() - t0
    comm = sif_dist.default_comm()
    timed_out = bool(int(comm.status.item()) & nv.STATUS_COMM_TIMEOUT)
    good = raised == (rank == world - 1) and not timed_out and dt < 2.0
    chk('bad id on rank %d' % (world - 1), good, 'IndexError here %s, returned after %.3f s, peer timeout %s'
        % (raised, dt, timed_out))


def main():
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    local = int(os.environ.get('LOCAL_RANK', rank))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    chk = Checker(rank)
    assert sif_dist.default_comm() is not None, 'PeerComm was not created'
    per_rank, L, V = 6000, 64, 50_000           # n_local L = 384 k < 8 V = 400 k; n_local >= 4096: tcgen05 Gram
    for K in (1, 3, 12):
        check_case(chk, dev, world, rank, per_rank * world, L, V, K, single=K == 3, nccl=K == 3, ragged=K == 3)
    check_case(chk, dev, world, rank, 157, 20, 3016, 3, ragged=True)              # n_global < d: start blocks
    n0 = 1000                                                                      # the last rank owns no rows
    lo, hi = sif_dist.shard_bounds(n0, world - 1, rank) if rank < world - 1 else (n0, n0)
    check_case(chk, dev, world, rank, n0, 24, 3016, 3, bounds=(lo, hi))
    check_bad_id(chk, dev, world, rank)
    flag = torch.tensor([0 if chk.ok else 1], device=dev)
    dist.all_reduce(flag)
    sif_dist.close_default_comms()
    dist.destroy_process_group()
    sys.exit(int(flag.item() != 0))


if __name__ == '__main__':
    main()
