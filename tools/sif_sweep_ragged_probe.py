"""SIF sweep on ragged (CSR) ids: one K-vector embed over the unpadded tokens (mmb_sif_embed_multi_ragged) against K
single-vector ragged embeds and against the padded K-vector embed.

    python tools/sif_sweep_ragged_probe.py [--ks 1,2,4,8] [--reps 5] [--out profiles/r04_sif_sweep_ragged.jsonl]

Workload: bench.py's (10 M utterances x 64 tokens, V = 400 k, d = 300, Zipf ids, right-padded with id 0),
MMB_BENCH_N / _L / _V honoured, converted once with sif_functions.to_ragged (the conversion is not timed).  K weight
vectors a / (a + p(w)) with a log-spaced in [1e-4, 1e-2] (a = 1e-3 for K = 1), pad weight 1.0.  CUDA-event times
after one warm-up of each arm, min / median / max over the repeats, the arms alternating within each repeat:
  (a) one mmb_sif_embed_multi_ragged call,
  (b) K x mmb_sif_embed_ragged (the single-vector kernel (a) reproduces bit for bit),
  (c) one mmb_sif_embed_multi call on the padded ids (the padded sweep).
One more line compares the single-vector kernels: mmb_sif_embed_ragged against mmb_sif_embed and mmb_sif_embed_ws
on the padded ids.  The POM shapes (real ids of tests/golden/sif_pom_full.npz: 100 x 1089 and 203 x 1357, 73 %
padding, V = 7763, d = 300) get the same three arms per K as latencies, each timed over a loop of --pom-iters calls.
Each line carries the card's name, power limit and SM clock read in the same run, the kernel of (a) with its
registers (cuobjdump of the built library), and the output check: (a) bit-equal to (b), max relative difference to
the padded result.  One JSON line per measurement, appended to --out.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'multimodal-baselines_b200')
for _p in (ROOT, PKG, os.path.join(ROOT, 'tools'), os.path.join(ROOT, 'tests', 'golden')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from sif_sweep_probe import gpu_state, kernel_registers, max_rel_diff, stats, timed  # noqa: E402


def sif_vectors(p, K, dev):
    a = [1e-3] if K == 1 else list(np.geomspace(1e-4, 1e-2, K))
    W = np.empty((K, p.size + 1), dtype=np.float64)
    W[:, 0] = 1.0
    for k, ak in enumerate(a):
        W[k, 1:] = ak / (ak + p)
    return a, torch.as_tensor(W.astype(np.float32), device=dev)


class Arms:
    """The three embeds of one (table, K vectors, ids) case; every call checks its return code."""

    def __init__(self, nv, table, W_t, ids, rag, emb, one):
        self.nv, self.lib = nv, nv.lib
        self.table, self.W_t, self.ids, self.rag, self.emb, self.one = table, W_t, ids, rag, emb, one
        self.V, self.d = table.shape
        self.K = W_t.shape[0]
        self.n, self.L = ids.shape
        self.wk = [W_t[k].contiguous() for k in range(self.K)]
        self.st = torch.zeros(1, dtype=torch.int32, device=table.device)
        self.mbytes = self.lib.mmb_sif_embed_multi_workspace_bytes(self.V, self.K)
        self.mws = torch.empty(self.mbytes, dtype=torch.uint8, device=table.device)

    def a(self):
        nv, r = self.nv, self.rag
        nv.check(self.lib.mmb_sif_embed_multi_ragged(
            nv.ptr(self.table), self.V, self.d, nv.ptr(self.W_t), self.K, nv.ptr(r.tokens), nv.ptr(r.offsets), self.n,
            r.L_pad, r.pad_id, nv.ptr(self.emb), nv.ptr(self.st), nv.ptr(self.mws), self.mbytes, nv.stream_ptr()))

    def single_ragged(self, k):
        nv, r = self.nv, self.rag
        nv.check(self.lib.mmb_sif_embed_ragged(
            nv.ptr(self.table), self.V, self.d, nv.ptr(self.wk[k]), nv.ptr(r.tokens), nv.ptr(r.offsets), self.n,
            r.L_pad, r.pad_id, nv.ptr(self.one), nv.ptr(self.st), nv.stream_ptr()))

    def b(self):
        for k in range(self.K):
            self.single_ragged(k)

    def c(self):
        nv = self.nv
        nv.check(self.lib.mmb_sif_embed_multi(
            nv.ptr(self.table), self.V, self.d, nv.ptr(self.W_t), self.K, nv.ptr(self.ids), self.n, self.L,
            nv.ptr(self.emb), nv.ptr(self.st), nv.ptr(self.mws), self.mbytes, nv.stream_ptr()))

    def single_padded(self, k):
        nv = self.nv
        nv.check(self.lib.mmb_sif_embed(nv.ptr(self.table), self.V, self.d, nv.ptr(self.wk[k]), nv.ptr(self.ids),
                                        self.n, self.L, nv.ptr(self.one), nv.ptr(self.st), nv.stream_ptr()))

    def check(self):
        """(a) bit-equal to (b) for every k; max relative difference of (a) to the padded result (mmb_sif_embed with
        W[k], which is (c)[k] bit for bit)."""
        self.a()
        kname = self.lib.mmb_last_kernel(1).decode()
        bit_equal, rel = True, 0.0
        for k in range(self.K):
            self.single_ragged(k)
            bit_equal = bit_equal and bool(torch.equal(self.emb[k].view(torch.int32), self.one.view(torch.int32)))
            self.single_padded(k)
            rel = max(rel, max_rel_diff(self.emb[k], self.one))
        self.nv.raise_on_status(self.st, self.V)
        return kname, bit_equal, rel


def run_arms(arms, reps, iters=1):
    fns = (arms.a, arms.b, arms.c)
    for f in fns:
        f()
    torch.cuda.synchronize()
    times = ([], [], [])
    for _ in range(reps):
        for f, t in zip(fns, times):
            t.append(timed(lambda: [f() for _ in range(iters)]) / iters)
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ks', default='1,2,4,8')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--pom-iters', type=int, default=50)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r04_sif_sweep_ragged.jsonl'))
    args = ap.parse_args()
    import _native as nv
    import sif_functions as sf
    lib = nv.lib
    dev = nv.require_cuda()
    ks = [int(k) for k in args.ks.split(',')]
    out_lines = []

    def emit(line):
        print(json.dumps(line), flush=True)
        out_lines.append(line)

    # ---- the bench workload
    N, L, V, d = bench.N_UTT, bench.L_TOK, bench.VOCAB, bench.DIM
    table, w1, p = bench.make_table_and_weights(dev, V=V, d=d)
    ids_full = bench.make_ids(dev, N, L, p, seed=1)
    rag_full = sf.to_ragged(ids_full)
    n_tok = int(rag_full.offsets[-1].item())
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    for K in ks:
        a, W_t = sif_vectors(p, K, dev)
        # utterances: the whole workload unless the K outputs, one comparison buffer and the scratch do not fit
        torch.cuda.empty_cache()
        free = torch.cuda.mem_get_info()[0]
        n = N
        while n > 1 and (K + 1) * n * d * 4 + V * d * 4 * 2 + (1 << 30) > free:
            n //= 2
        ids = ids_full[:n]
        rag = rag_full if n == N else sf.to_ragged(ids)
        emb = torch.empty((K, n, d), dtype=torch.float32, device=dev)
        one = torch.empty((n, d), dtype=torch.float32, device=dev)
        arms = Arms(nv, table, W_t, ids, rag, emb, one)
        ta, tb, tc = run_arms(arms, args.reps)
        clocks = gpu_state(torch.cuda.current_device())
        kname, bit_equal, rel = arms.check()
        tokens = int(rag.offsets[-1].item())
        ma, mc = float(np.median(ta)), float(np.median(tc))
        emit({
            'probe': 'sif_sweep_ragged', 'K': K, 'a': [float('%.3g' % x) for x in a], 'n_utt': n, 'L_pad': L, 'V': V,
            'd': d, 'tokens': tokens, 'pad_fraction': round(1.0 - tokens / float(n * L), 4),
            'n_utt_note': 'full workload' if n == N else 'reduced from %d to fit K outputs + comparison buffer' % N,
            **clocks, 'kernel': kname, 'kernel_registers': kernel_registers(nv.LIB_PATH, kname), 'reps': args.reps,
            'a_multi_ragged_ms': stats(ta), 'b_K_x_embed_ragged_ms': stats(tb), 'c_multi_padded_ms': stats(tc),
            'a_over_b': round(ma / float(np.median(tb)), 3), 'a_over_c': round(ma / mc, 3),
            # algorithmic bytes: ids (+ offsets) once, every token's row once, K outputs
            'a_bytes_per_s': round((n * (d * 4 * K + 8) + tokens * (8 + d * 4)) / (ma * 1e-3), 1),
            'c_bytes_per_s': round(n * (L * 8 + L * d * 4 + K * d * 4) / (mc * 1e-3), 1),
            'check_a_bit_equal_b': bit_equal, 'check_a_max_rel_diff_padded': rel,
        })
        del arms, emb, one, W_t
        if rag is not rag_full:
            del rag
        torch.cuda.empty_cache()

    # ---- single-vector kernels: ragged against padded (never timed before)
    torch.cuda.empty_cache()
    one = torch.empty((N, d), dtype=torch.float32, device=dev)
    sbytes = lib.mmb_sif_embed_workspace_bytes(V, d, N, L)
    sws = torch.empty(max(sbytes, 256), dtype=torch.uint8, device=dev)
    P = lambda t: nv.ptr(t)                                    # noqa: E731

    def ragged():
        nv.check(lib.mmb_sif_embed_ragged(P(table), V, d, P(w1), P(rag_full.tokens), P(rag_full.offsets), N, L, 0,
                                          P(one), P(st), nv.stream_ptr()))

    def padded():
        nv.check(lib.mmb_sif_embed(P(table), V, d, P(w1), P(ids_full), N, L, P(one), P(st), nv.stream_ptr()))

    def padded_ws():
        nv.check(lib.mmb_sif_embed_ws(P(table), V, d, P(w1), P(ids_full), N, L, P(one), P(st), P(sws), sbytes,
                                      nv.stream_ptr()))

    fns = (ragged, padded, padded_ws)
    names = []
    for f in fns:
        f()
        torch.cuda.synchronize()
        names.append(lib.mmb_last_kernel(0).decode())
    times = ([], [], [])
    for _ in range(args.reps):
        for f, t in zip(fns, times):
            t.append(timed(f))
    clocks = gpu_state(torch.cuda.current_device())
    nv.raise_on_status(st, V)
    emit({'probe': 'sif_embed_ragged_vs_padded', 'K': 1, 'n_utt': N, 'L_pad': L, 'V': V, 'd': d, 'tokens': n_tok,
          'pad_fraction': round(1.0 - n_tok / float(N * L), 4), **clocks, 'kernels': names, 'reps': args.reps,
          'ragged_ms': stats(times[0]), 'padded_embed_ms': stats(times[1]), 'padded_embed_ws_ms': stats(times[2]),
          'ragged_over_padded_embed': round(float(np.median(times[0]) / np.median(times[1])), 3),
          'ragged_over_padded_embed_ws': round(float(np.median(times[0]) / np.median(times[2])), 3)})
    del one, sws, rag_full, ids_full, table
    torch.cuda.empty_cache()

    # ---- the POM shapes: latencies
    import cases
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'sif_pom_full.npz'))
    w_pom = np.asarray(g['weights'], dtype=np.float64).reshape(-1)
    table = torch.as_tensor(cases.table(w_pom.size, 300, seed=11), device=dev)
    for split in ('valid', 'test'):
        ids = torch.as_tensor(g[split + '_ids'].astype(np.int64), device=dev)
        rag = sf.to_ragged(ids)
        n, Lp = ids.shape
        tokens = int(rag.offsets[-1].item())
        for K in ks:
            W = np.stack([w_pom * s for s in np.linspace(1.0, 0.5, K)]).astype(np.float32)
            W_t = torch.as_tensor(W, device=dev)
            emb = torch.empty((K, n, 300), dtype=torch.float32, device=dev)
            one = torch.empty((n, 300), dtype=torch.float32, device=dev)
            arms = Arms(nv, table, W_t, ids, rag, emb, one)
            ta, tb, tc = run_arms(arms, args.reps, iters=args.pom_iters)
            clocks = gpu_state(torch.cuda.current_device())
            kname, bit_equal, rel = arms.check()
            emit({'probe': 'sif_sweep_ragged_pom', 'split': split, 'K': K, 'n_utt': n, 'L_pad': Lp, 'V': w_pom.size,
                  'd': 300, 'tokens': tokens, 'pad_fraction': round(1.0 - tokens / float(n * Lp), 4), **clocks,
                  'kernel': kname, 'kernel_registers': kernel_registers(nv.LIB_PATH, kname), 'reps': args.reps,
                  'iters_per_rep': args.pom_iters, 'a_multi_ragged_ms': stats(ta), 'b_K_x_embed_ragged_ms': stats(tb),
                  'c_multi_padded_ms': stats(tc), 'check_a_bit_equal_b': bit_equal,
                  'check_a_max_rel_diff_padded': rel})

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'a') as fh:
        for line in out_lines:
            fh.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
