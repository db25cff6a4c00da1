"""Sharded SIF sweep probe: sif_dist.sharded_sif_embedding_sweep against K x P sharded_sif_embedding calls.

    torchrun --nproc-per-node R tools/sif_sweep_dist_probe.py [--ks 2,4,8] [--reps 3]
        [--out profiles/r05_sif_sweep_dist.jsonl]

Workload: bench.py's (10 M utterances x 64 tokens, V = 400 k, d = 300, Zipf ids, right-padded; MMB_BENCH_N / _L /
_V honoured), split over the R ranks as bench.py splits it (rank r draws its block with seed 1000 + r).  K weight
vectors a / (a + p(w)), a log-spaced in [1e-4, 1e-2]; npcs = (1,) and (1, 2, 3).  For every (K, npcs):
  (a) one sharded_sif_embedding_sweep call, with CUDA events at its stage marks (embed, gram, allreduce, pc,
      project);
  (b) K x P sharded_sif_embedding calls (the production single-vector path: pre-scaled embed, fused Gram exchange).
After one warm-up of each arm (which also compares every out[k, j] of (a) with the matching call of (b): the embeds
differ by the pre-scaled table's one rounding per term, so the max relative row difference is recorded), the arms
alternate for --reps repeats behind a barrier; a time is the slowest rank's.  A configuration whose per-rank
memory, 4 K n_local d (1 + P) bytes (4 K n_local d at P = 1, which projects in place) plus one output of (b),
ids, table and 4 GB of slack, does not fit the card is skipped on every rank and logged as skipped.  At R = 1 the probe also times P
mmb_remove_pc calls against one mmb_remove_pc_multi on the first K vector's embeddings (npcs = (1, 2, 3)),
outputs compared bit for bit.  Each line carries the card's name, power limit and SM clock read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'multimodal-baselines_b200')
for _p in (ROOT, PKG, os.path.join(ROOT, 'tools')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import bench  # noqa: E402
from sif_sweep_probe import gpu_state, max_rel_diff, stats, timed  # noqa: E402


class Marks(object):
    """timers= callback: one CUDA event per stage mark."""

    def __init__(self):
        self.ev = [('start', torch.cuda.Event(enable_timing=True))]
        self.ev[0][1].record()

    def __call__(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev.append((name, e))

    def stages(self):
        self.ev[-1][1].synchronize()
        return {n: self.ev[i][1].elapsed_time(e) for i, (n, e) in enumerate(self.ev[1:])}


def slowest(ms):
    t = torch.tensor([ms], dtype=torch.float64, device='cuda')
    if dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier():
    if dist.is_initialized():
        dist.barrier()
    torch.cuda.synchronize()


def remove_pc_line(nv, sf, emb, reps):
    """P mmb_remove_pc calls against one mmb_remove_pc_multi (npcs = (1, 2, 3)) on one GPU."""
    npcs = (1, 2, 3)
    n, d = emb.shape
    G = sf.gram(emb)
    pcs = [sf.pc_from_gram(G, p, n) for p in npcs]
    outs = [torch.empty_like(emb) for _ in npcs]
    ref = [torch.empty_like(emb) for _ in npcs]
    P = len(npcs)
    pc_arr = (C.c_void_p * P)(*[p.data_ptr() for p in pcs])
    out_arr = (C.c_void_p * P)(*[o.data_ptr() for o in outs])
    npc_arr = (C.c_int * P)(*npcs)

    def multi():
        nv.check(nv.lib.mmb_remove_pc_multi(nv.ptr(emb), n, d, P, pc_arr, npc_arr, out_arr, nv.stream_ptr()))

    def singles():
        for pc, o in zip(pcs, ref):
            sf.project_out(emb, pc, out=o)

    multi(), singles()
    t_m, t_s = [], []
    for _ in range(reps):
        t_m.append(timed(multi))
        t_s.append(timed(singles))
    same = all(torch.equal(a, b) for a, b in zip(outs, ref))
    gb = 4.0 * n * d * (1 + P) / 1e9
    return {'probe': 'remove_pc_multi', 'n': n, 'd': d, 'npcs': list(npcs), 'multi_ms': stats(t_m),
            'p_single_calls_ms': stats(t_s), 'ratio_median': round(np.median(t_m) / np.median(t_s), 3),
            'multi_alg_GBps': round(gb / (np.median(t_m) * 1e-3), 1), 'bit_identical': same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ks', default='2,4,8')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r05_sif_sweep_dist.jsonl'))
    args = ap.parse_args()
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', rank))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    import _native as nv
    import sif_dist
    import sif_functions as sf
    N, L, V, d = bench.N_UTT, bench.L_TOK, bench.VOCAB, bench.DIM
    table, _w, p = bench.make_table_and_weights(dev, V=V, d=d)
    lo, hi = sif_dist.shard_bounds(N, world, rank)
    n_local = hi - lo
    ids = bench.make_ids(dev, n_local, L, p, seed=1000 + rank)
    comm = sif_dist.default_comm() if world > 1 else None
    card = gpu_state(local)
    lines = []
    free, total = torch.cuda.mem_get_info()
    for K in [int(k) for k in args.ks.split(',')]:
        W = torch.stack([torch.as_tensor(bench_weights(p, a), device=dev) for a in np.geomspace(1e-4, 1e-2, K)])
        for npcs in ((1,), (1, 2, 3)):
            P = len(npcs)
            need = (4 * K * n_local * d * (1 if P == 1 else 1 + P) + 4 * n_local * d     # + one output of arm (b)
                    + ids.numel() * 8 + table.numel() * 4 + 4 * 2 ** 30)
            fits = torch.tensor([1 if need < total else 0], device=dev)
            if world > 1:
                dist.all_reduce(fits, op=dist.ReduceOp.MIN)
            base = {'probe': 'sharded_sweep', 'world': world, 'n_global': N, 'n_local_max': sif_dist.shard_bounds(
                N, world, 0)[1], 'L': L, 'V': V, 'd': d, 'K': K, 'npcs': list(npcs), **card}
            if not int(fits.item()):
                lines.append(dict(base, skipped='needs %.1f GB per rank of %.1f GB' % (need / 1e9, total / 1e9)))
                continue

            def sweep(marks=None):
                return sif_dist.sharded_sif_embedding_sweep(table, W, ids, N, lo, npcs=npcs, timers=marks, comm=comm)

            def singles(check=None):
                worst = 0.0
                for k in range(K):
                    for j, q in enumerate(npcs):
                        emb, _pc, st = sif_dist.sharded_sif_embedding(table, W[k], ids, N, lo, npc=q, comm=comm)
                        if check is not None:
                            worst = max(worst, max_rel_diff(check[k, j], emb))
                        del emb
                return worst

            out, _pcs, st = sweep()
            nv.raise_on_status(st, V)
            diff = slowest(singles(check=out))
            del out, _pcs
            t_sw, t_si, stages = [], [], []
            for _ in range(args.reps):
                barrier()
                m = Marks()
                o = sweep(m)[0]
                st_ms = m.stages()
                t_sw.append(slowest(sum(st_ms.values())))
                stages.append(st_ms)
                del o
                barrier()
                t_si.append(slowest(timed(singles)))
            med = {s: round(float(np.median([x[s] for x in stages])), 3) for s in stages[0]}
            lines.append(dict(base, sweep_ms=stats(t_sw), kp_single_calls_ms=stats(t_si),
                              ratio_median=round(float(np.median(t_sw) / np.median(t_si)), 3),
                              sweep_stage_ms_median_rank=med, max_rel_row_diff_vs_single_calls=diff))
            if rank == 0:
                print(json.dumps(lines[-1]), flush=True)
            torch.cuda.empty_cache()
    if world == 1:
        emb = sf.sweep_embed(table, W[:1].contiguous(), ids)[0][0]
        lines.append(dict(remove_pc_line(nv, sf, emb, args.reps), **card))
        print(json.dumps(lines[-1]), flush=True)
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'a') as fh:
            for ln in lines:
                fh.write(json.dumps(ln) + '\n')
    if world > 1:
        sif_dist.close_default_comms()
        dist.destroy_process_group()


def bench_weights(p, a):
    """a / (a + p(w)) over ids 1..V-1 and 1.0 for the pad id 0, float32 (bench.make_table_and_weights's form)."""
    return np.concatenate([[1.0], a / (a + p)]).astype(np.float32)


if __name__ == '__main__':
    main()
