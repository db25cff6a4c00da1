#!/usr/bin/env python
"""bench.py -- utterances/sec of the SIF hot path (embed + PC removal) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[3], SURVEY.md §8d "Config 4", the shape the roofline is
quoted on; it fits one GPU): N = 10,000,000 utterances x 64 tokens, 400,000-word vocabulary,
d = 300, Zipf(1.1) ids, lengths ~U[16,64] right-padded with id 0, synthetic GloVe-like
table with a planted common direction.  One step = one pass of the whole batch through
get_sentence_embeddings: gather + weighted average -> Gram -> principal component ->
projection subtraction.  With N > 1 ranks the 10 M utterances are sharded (strong scaling)
and the 300x300 Gram is summed with one NCCL all-reduce.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (inputs in HBM);
`e2e` = the same metric through the host-buffer API (pinned ids in, embeddings out, copies
inside the timed region); `roofline` = the dominant kernel (the gather/average) against the
measured HBM copy bandwidth; `cpu_baseline` = the oracle port of the reference's NumPy /
sklearn path timed on this box's host cores (bounded sample).

`--impl reference` times that CPU port instead (rank 0 only) and prints the same line shape.

`--dump-outputs DIR` writes what the last timed step returned, after the timed region, as float32 .npy
files (see dump_outputs).  The inputs depend only on the arguments and the MMB_BENCH_* variables, so two
builds run with the same ones can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'multimodal-baselines_b200')
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

OUT = sys.stdout
METRIC = 'utterances/sec (SIF embed + PC removal)'
UNIT = 'utterances/s'
N_UTT = int(os.environ.get('MMB_BENCH_N', 10_000_000))
L_TOK = int(os.environ.get('MMB_BENCH_L', 64))
VOCAB = int(os.environ.get('MMB_BENCH_V', 400_000))
DIM = 300
ZIPF_S = 1.1
# SURVEY.md §8(d): algorithmic bytes per utterance of the embed pass at L tokens, d floats:
# ids L*8 + gathered rows L*d*4 (every token counted, no cache credit) + output d*4.
EMBED_BYTES_PER_UTT = L_TOK * 8 + L_TOK * DIM * 4 + DIM * 4
WORKLOAD = 'sif_%dM_utt_x%d_tok_v%dk_d%d' % (N_UTT // 1_000_000, L_TOK, VOCAB // 1000, DIM) \
    if N_UTT >= 1_000_000 else 'sif_%d_utt_x%d_tok_v%d_d%d' % (N_UTT, L_TOK, VOCAB, DIM)


# ----------------------------------------------------------------------------- inputs
def zipf_pmf(V, s=ZIPF_S):
    p = 1.0 / np.arange(1, V, dtype=np.float64) ** s
    return p / p.sum()


def make_table_and_weights(device, V=VOCAB, d=DIM, seed=0):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    table = 0.4 * torch.randn((V, d), device=device, generator=g)
    table += 0.3 * torch.randn((1, d), device=device, generator=g)      # planted common direction
    table[0] = 0.0
    p = zipf_pmf(V)
    w = np.empty(V, dtype=np.float64)
    w[0] = 1.0
    w[1:] = 1e-3 / (1e-3 + p)                                            # sif.py:14-32 form
    return table.contiguous(), torch.as_tensor(w.astype(np.float32)).to(device), p


IDS_KIND = os.environ.get('MMB_BENCH_IDS', 'zipf')     # 'uniform': cache-hostile ids (secondary measurement)


def make_ids(device, n_rows, L, p, seed, out=None, block=1 << 20):
    """Zipf ids over 1..V-1 by inverse-CDF on the device, right-padded with 0."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    if IDS_KIND == 'uniform':
        p = np.full(p.size, 1.0 / p.size)
    cdf = torch.as_tensor(np.cumsum(p)).to(device=device, dtype=torch.float32)
    ids = out if out is not None else torch.empty((n_rows, L), dtype=torch.int64, device=device)
    ar = torch.arange(L, device=device)[None, :]
    for s in range(0, n_rows, block):
        e = min(n_rows, s + block)
        u = torch.rand((e - s, L), device=device, generator=g)
        tok = torch.searchsorted(cdf, u).clamp_(max=p.size - 1) + 1
        lens = torch.randint(16 if L >= 16 else 1, L + 1, (e - s, 1), device=device, generator=g)
        tok[ar >= lens] = 0
        ids[s:e] = tok
    return ids


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                 '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def window(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        rows = [l for t, l in self.lines if t0 - 0.15 <= t <= t1 + 0.15] or [l for _, l in self.lines[-3:]]
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            f = [x.strip() for x in r.split(',')]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for nm, val in zip(names, f[2:6]):
                if val.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


# ----------------------------------------------------------------------------- CPU arm
def reference_fn():
    """(get_sentence_embeddings, kind, description): the reference's OWN sif.get_sentence_embeddings from
    oracle/_ref (unmodified copies of its sif.py / sif_functions.py, made by oracle/make_ref.py where the reference
    tree exists), else the oracle port with the reference's Python loops."""
    from oracle import make_ref
    from oracle import sif_oracle as so
    mod = make_ref.load()
    if mod is not None:
        return mod.get_sentence_embeddings, 'reference', ("the reference's own sif.get_sentence_embeddings "
                                                          '(oracle/_ref/reference_sif.zip: its unmodified sif.py + sif_functions.py, Python loops '
                                                          '+ sklearn TruncatedSVD)')
    return so.get_sentence_embeddings_loop, 'port', ("oracle port of sif.py:84-94 with the reference's own Python loops "
                                                     '+ sklearn TruncatedSVD')


def cpu_port_rate(table_np, weights_np, ids_np, repeats=1):
    """The reference path (its own Python loops + sklearn) on host cores."""
    fn, kind, desc = reference_fn()
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn(table_np, weights_np, ids_np)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return ids_np.shape[0] / best, best, kind, desc


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    fn, kind, how = reference_fn()
    sample = int(os.environ.get('MMB_REF_SAMPLE', 20_000))     # ~1 s per step: 23 steps (driver default) ~ 25 s in all
    rng = np.random.default_rng(0)
    p = zipf_pmf(VOCAB)
    table = (0.4 * rng.standard_normal((VOCAB, DIM), dtype=np.float32)
             + 0.3 * rng.standard_normal((1, DIM), dtype=np.float32))
    table[0] = 0
    weights = np.concatenate([[1.0], 1e-3 / (1e-3 + p)])
    cdf = np.cumsum(p)
    ids = np.minimum(np.searchsorted(cdf, rng.random((sample, L_TOK))), p.size - 1) + 1
    lens = rng.integers(16, L_TOK + 1, size=(sample, 1))
    ids[np.arange(L_TOK)[None, :] >= lens] = 0
    ids = ids.astype(np.int64)
    for _ in range(args.warmup):
        fn(table, weights, ids)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn(table, weights, ids)
    dt = (time.perf_counter() - t0) / args.steps
    value = sample / dt
    cores = cpu_threads()
    desc = '%d-utterance sample of the %s workload per step; %s' % (sample, WORKLOAD, how)
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'sample_utterances_per_step': sample},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': kind, 'sample': desc},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }), file=OUT, flush=True)


# ----------------------------------------------------------------------------- GPU arm
def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as fh:
            return float(json.load(fh)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md: 6.65 TB/s)'


def load_tensor_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
            return float(json.load(fh)['bf16_tflops'])
    except Exception:
        return 1590.0


def measure_tf32_peak(dev, n=8192, reps=10):
    """Dense TF32 GEMM rate of this GPU, measured the way MEASURED_PEAKS.json measures bf16
    (torch.matmul n^3, 2 n^3 FLOP, best of `reps`, CUDA events): the driver records no TF32 figure,
    and the Gram kernel's pipe is kind::tf32.  Runs after the timed regions."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn((n, n), device=dev)
        b = torch.randn((n, n), device=dev)
        for _ in range(3):
            torch.matmul(a, b)
        best = None
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    except Exception:
        return None
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def norm_kernel_name(name):
    """'void mmb::sif_embed_warp_kernel<3, 0, 2, 4, 0>(const float4 *, ...)' (ncu) and
    'sif_embed_warp_kernel<3,false,2,4,false>' (mmb_last_kernel) -> the same key."""
    name = (name or '').strip()
    if name.startswith('void '):
        name = name[5:]
    depth, cut = 0, len(name)
    for k, ch in enumerate(name):                  # drop the argument list (the first '(' outside <...>)
        if ch == '<':
            depth += 1
        elif ch == '>':
            depth -= 1
        elif ch == '(' and depth == 0:
            cut = k
            break
    name = name[:cut].replace(' ', '').replace('true', '1').replace('false', '0')
    return name.split('::')[-1]


def load_ncu_record(kernel, ids_kind):
    """The committed `ncu --set full` record of the embed kernel for this id distribution
    (profiles/embed_traffic.json, written by tools/embed_traffic.py from the .ncu-rep summaries).  It is
    used only when it was captured on the SAME kernel instantiation the library reports it launched;
    otherwise (None, reason)."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'embed_traffic.json')) as fh:
            t = json.load(fh)
    except Exception as e:
        return None, 'profiles/embed_traffic.json unreadable (%s)' % e
    rec = t.get(ids_kind)
    if not isinstance(rec, dict):
        return None, 'no %s record in profiles/embed_traffic.json' % ids_kind
    if norm_kernel_name(rec.get('ncu_kernel_name')) != norm_kernel_name(kernel):
        return None, 'stale capture: ncu saw %s, this run launched %s' % (rec.get('ncu_kernel_name'), kernel)
    return rec, rec.get('source')


def time_embed_only(lib, nv, table, vocab_w, ids, reps=5, warm=3):
    """CUDA-event time of the embed kernel alone on `ids` (current stream)."""
    import sif_dist as mdist
    n, L = ids.shape
    V, d = table.shape
    emb = torch.empty((n, d), dtype=torch.float32, device=ids.device)
    st = torch.zeros(1, dtype=torch.int32, device=ids.device)
    ws_bytes = lib.mmb_sif_embed_workspace_bytes(V, d, n, L)         # the same entry point the timed step uses
    ws = mdist._embed_scratch(ws_bytes, ids.device) if ws_bytes else None
    ms = []
    for it in range(warm + reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nv.check(lib.mmb_sif_embed_ws(nv.ptr(table), V, d, nv.ptr(vocab_w), nv.ptr(ids), n, L, nv.ptr(emb), nv.ptr(st),
                                      nv.ptr(ws), ws_bytes, nv.stream_ptr()))
        e1.record()
        e1.synchronize()
        if it >= warm:
            ms.append(e0.elapsed_time(e1))
    return float(np.mean(ms)), emb


def rel_rows(got, want):
    """max over rows of max|got - want| / max|want| (the parity tests' metric)."""
    scale = want.abs().amax(dim=-1, keepdim=True).clamp_min(1e-30)
    return float(((got - want).abs() / scale).max())


def verify_run(ctx):
    """Parity of what was just timed (VERDICT r1 #1): every check lands in the JSON line's `verify` block and
    a failure makes bench.py exit non-zero.  Checkers: the NumPy oracle on a CPU-sized sample, float64 torch
    linear algebra on the device for the 10 M-row quantities, NCCL for the cross-rank sum."""
    import torch.distributed as dist
    import sif_dist as mdist
    import sif_functions as sf
    from oracle import sif_oracle as so
    nv, lib = ctx['nv'], ctx['lib']
    table, vocab_w, ids = ctx['table'], ctx['vocab_w'], ctx['ids']
    emb, pc, lo, world, rank, dev = ctx['emb'], ctx['pc'], ctx['lo'], ctx['world'], ctx['rank'], ctx['dev']
    n_local = ids.shape[0]
    checks = {}

    # (1) pre-projection averages of this rank's first rows against the NumPy oracle (float64 accumulate)
    n_o = min(int(os.environ.get('MMB_VERIFY_ORACLE_ROWS', 4096)), n_local)
    _, avg = time_embed_only(lib, nv, table, vocab_w, ids, reps=1, warm=0)          # the same kernel, untimed
    if n_o > 0:
        ids_np = ids[:n_o].cpu().numpy()
        w_np = so.seq2weight(ids_np, np.ones(ids_np.shape), vocab_w.double().cpu().numpy())
        want = so.get_weighted_average(table.cpu().numpy(), ids_np, w_np)
        checks['avg_vs_oracle'] = {'rows': n_o, 'err': rel_rows(avg[:n_o].double().cpu(), torch.as_tensor(want)),
                                   'tol': 1e-5}
    # (2) the component against the top eigenvector of the float64 Gram of ALL rows (summed over ranks)
    G64 = torch.zeros((DIM, DIM), dtype=torch.float64, device=dev)
    for s0 in range(0, n_local, 1 << 20):
        blk = avg[s0:s0 + (1 << 20)].double()
        G64 += blk.T @ blk
    if world > 1:
        dist.all_reduce(G64)
    evals, evecs = torch.linalg.eigh(G64)
    v = evecs[:, -1]
    checks['pc_vs_float64_eigvec'] = {'abs_cos': abs(float(pc[0].double() @ v)), 'min': 0.9999,
                                      'eig_gap_ratio': float(evals[-1] / evals[-2])}
    # (3) the timed output rows against avg - (avg pc^T) pc evaluated in float64
    pcd = pc.double()
    rows = torch.cat([torch.arange(0, min(50_000, n_local), device=dev),
                      torch.arange(max(0, n_local - 50_000), n_local, device=dev)]).unique()
    a = avg[rows].double()
    want = a - (a @ pcd.T) @ pcd
    checks['emb_vs_float64_projection'] = {'rows': int(rows.numel()), 'err': rel_rows(emb[rows].double(), want),
                                           'tol': 1e-5}
    del avg
    # (4) multi-GPU: peers arrived, identical component bits on every rank, NCCL all-reduce path agrees
    if world > 1:
        comm = mdist.default_comm()
        if comm is not None:
            comm.check()
        pcs = [torch.empty_like(pc) for _ in range(world)]
        dist.all_gather(pcs, pc.contiguous())
        checks['pc_identical_on_all_ranks'] = {'ok': bool(all(torch.equal(pcs[0], q) for q in pcs))}
        if comm is not None:
            emb_n, pc_n, _ = mdist.sharded_sif_embedding(table, vocab_w, ids, N_UTT, lo, npc=1, comm=None)
            # two FP32 summation orders of the ranks' Grams (rank order here, NCCL's ring / tree there): the
            # components agree to ~1e-8 in cosine, the projected rows (small after the common direction is gone)
            # to a few 1e-7 of their maxima at 2 ranks and ~1e-6 at 8 -- half the embedding tolerance is the bar
            checks['peer_exchange_vs_nccl'] = {'pc_cos': float(pc[0].double() @ pc_n[0].double()), 'min_cos': 1 - 1e-7,
                                               'emb_err': rel_rows(emb, emb_n), 'tol': 5e-6}
            del emb_n
    # (5) the host-buffer (e2e) result against the device-resident one (Gram summed per chunk: different
    #     FP32 order, same tolerance as the embeddings)
    if ctx.get('e2e_sample') is not None:
        r, h = ctx['e2e_sample']
        checks['e2e_vs_device'] = {'rows': int(r.numel()), 'err': rel_rows(h.double(), emb[r].double().cpu()),
                                   'tol': 1e-5}

    def passed(c):
        if 'ok' in c:
            return c['ok']
        good = True
        if 'err' in c:
            good = good and c['err'] < c['tol']
        if 'emb_err' in c:
            good = good and c['emb_err'] < c['tol']
        if 'abs_cos' in c:
            good = good and c['abs_cos'] >= c['min']
        if 'pc_cos' in c:
            good = good and c['pc_cos'] > c['min_cos']
        return bool(good)
    for c in checks.values():
        c['ok'] = passed(c)
    flag = torch.tensor([0 if all(c['ok'] for c in checks.values()) else 1], device=dev)
    failed = {}
    if world > 1:
        dist.all_reduce(flag)
        mine = {k: c for k, c in checks.items() if not c['ok']}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)           # which check failed on which rank, for the line
        failed = {'rank%d' % r: g for r, g in enumerate(gathered) if g}
    else:
        failed = {'rank0': {k: c for k, c in checks.items() if not c['ok']}} if int(flag.item()) else {}
    return {'ok': int(flag.item()) == 0, 'rank0': checks, 'ranks_failed': int(flag.item()), 'failed': failed}


DUMP_ROWS = 32768      # 32768 x 300 float32 = 39 MB: the whole N x d output would be 12 GB


def dump_rows(n):
    """The embedding rows --dump-outputs writes: a fixed, seeded sample of the n global rows, ascending."""
    rng = np.random.default_rng(0)
    return np.sort(rng.choice(n, size=min(DUMP_ROWS, n), replace=False))


def dump_outputs(out_dir, emb, pc, lo, world, rank):
    """Write the last timed step's outputs under out_dir: pc.npy, the (npc, d) principal component, and
    embeddings.npy, the projected embedding rows dump_rows(N_UTT) of the (N, d) result, both float32.  With
    several ranks each rank contributes the sampled rows of its shard and rank 0 writes."""
    import torch.distributed as dist
    rows = dump_rows(N_UTT)
    mine = rows[(rows >= lo) & (rows < lo + emb.shape[0])] - lo
    part = emb[torch.as_tensor(mine, device=emb.device)].cpu().numpy()
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, part)
        part = np.concatenate(parts)              # shards are contiguous in rank order: rows stay ascending
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, 'embeddings.npy'), part.astype(np.float32))
        np.save(os.path.join(out_dir, 'pc.npy'), pc.cpu().numpy().astype(np.float32))


def mmb_secondary(steps=50):
    """SURVEY.md 8(d) secondary metric, recorded by the driver's own bench run: one MMB2 latent-optimisation
    step (heads -> word + 6 Gaussian terms -> backward -> SGD) at the MOSI and the real-POM layouts, as this
    repo's captured graph (dense text and token ids) next to the reference's formulas in stock PyTorch on
    the same GPU (tools/bench_mmb.py)."""
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import bench_mmb
    out = {}
    for shape in ('mosi', 'pom_real'):
        try:
            r = bench_mmb.run(shape, steps, do_cpu=False)
            out[shape] = {'batch': bench_mmb.B, 'N_T_V_A_Vd': r['N_T_V_A_Vd'],
                          'ms_graph': r['b200_fused_cuda_graph']['ms_per_step'],
                          'ms_graph_token_ids': r.get('b200_fused_cuda_graph_token_ids', {}).get('ms_per_step'),
                          'ms_eager_api': r['b200_fused']['ms_per_step'],
                          'ms_stock_torch_same_gpu': r['b200_stock_torch']['ms_per_step'],
                          'unit': 'ms per step (fwd + bwd + SGD), CUDA events, %d steps' % steps}
        except Exception as e:                      # the secondary block must never cost the primary line
            out[shape] = {'error': '%s: %s' % (type(e).__name__, e)}
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-verify', action='store_true')
    ap.add_argument('--no-secondary', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the GPU path\'s outputs; --impl reference has none')
    args.warmup = max(args.warmup, 0)
    # stdout carries exactly ONE JSON line: keep the real stdout for it and point fd 1 at stderr, so that
    # whatever else writes to fd 1 (NCCL's version banner at NCCL_DEBUG >= VERSION, library prints, the
    # reference helpers' progress lines) cannot land in front of it
    global OUT
    sys.stdout.flush()
    OUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    if args.impl == 'reference':
        run_reference_arm(args)
        return

    if os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
        os.environ['NCCL_DEBUG'] = 'WARN'           # NCCL's version banner goes to stdout: keep it to the one JSON line
    import torch.distributed as dist
    import _native as nv
    import sif_functions as sf
    import sif_dist as mdist
    from _native import lib

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        mdist.bind_to_gpu_numa_node(local_rank)     # host threads + pinned buffers next to this rank's GPU
        dist.init_process_group('nccl', device_id=dev)
    warmup = max(args.warmup, 3)

    lo, hi = mdist.shard_bounds(N_UTT, world, rank)
    n_local = hi - lo
    table, vocab_w, p = make_table_and_weights(dev)
    ids = make_ids(dev, n_local, L_TOK, p, seed=1000 + rank)
    torch.cuda.synchronize()

    # ---- device-resident steps, per-stage CUDA events on the launching stream ------------
    stages = ('embed', 'gram', 'allreduce', 'pc', 'project')

    def run_step(record=None):
        marks = []

        def mark(name):
            if record is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((name, e))
        out = mdist.sharded_sif_embedding(table, vocab_w, ids, N_UTT, lo, npc=1, timers=mark)
        if record is not None:
            record.append(marks)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        emb, pc, st = run_step()
    barrier()
    nv.raise_on_status(st, VOCAB)
    embed_kernel = (lib.mmb_last_kernel(0) or b'').decode()
    sampler = ClockSampler(local_rank)
    time.sleep(0.25)
    records = []
    start = torch.cuda.Event(enable_timing=True)
    stop = torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    launches0 = int(lib.mmb_launch_count())
    start.record()
    step_starts = []
    for _ in range(args.steps):
        s = torch.cuda.Event(enable_timing=True)
        s.record()
        step_starts.append(s)
        emb, pc, st = run_step(records)
    stop.record()
    launches = int(lib.mmb_launch_count()) - launches0         # counted by the library's launch sites
    barrier()
    t_wall1 = time.time()
    ms_total = start.elapsed_time(stop)
    stage_ms = {k: 0.0 for k in stages}
    for s0, marks in zip(step_starts, records):
        prev = s0
        for name, e in marks:
            stage_ms[name] += prev.elapsed_time(e)
            prev = e
    stage_ms = {k: v / args.steps for k, v in stage_ms.items()}
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = N_UTT / (ms_per_step * 1e-3)
    clocks = sampler.window(t_wall0, t_wall1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, emb, pc, lo, world, rank)

    # ---- end to end: pinned host ids in, float32 embeddings out, copies inside the region --
    e2e = None
    e2e_sample = None
    if not args.no_e2e:
        h_ids = nv.PinnedArray((n_local, L_TOK), np.int64)
        h_out = nv.PinnedArray((n_local, DIM), np.float32)
        torch.as_tensor(h_ids.array).copy_(ids)          # D2H once, outside the timed region
        torch.cuda.synchronize()
        omega = np.ascontiguousarray(sf.start_block(DIM if N_UTT >= DIM else N_UTT, 1))

        def e2e_step():
            if world == 1:
                nv.check(lib.mmb_sif_embedding_host(nv.ptr(table), VOCAB, DIM, nv.ptr(vocab_w),
                                                    nv.np_ptr(h_ids.array), n_local, L_TOK, 1, nv.np_ptr(omega),
                                                    nv.np_ptr(h_out.array), 0, None, nv.GRAM_AUTO, 0))
            elif mdist.default_comm() is not None and N_UTT >= DIM:
                mdist.default_comm().sif_embedding_host(table, vocab_w, h_ids.array, h_out.array, N_UTT, npc=1)
            else:
                d_ids = torch.as_tensor(h_ids.array).to(dev, non_blocking=True)
                e, _pc, _st = mdist.sharded_sif_embedding(table, vocab_w, d_ids, N_UTT, lo, npc=1)
                torch.as_tensor(h_out.array).copy_(e, non_blocking=True)
                torch.cuda.synchronize()
        emb_keep = emb
        del emb
        torch.cuda.empty_cache()
        for _ in range(2):
            e2e_step()
        barrier()
        n_e2e = max(1, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / n_e2e], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        emb = emb_keep
        r = torch.cat([torch.arange(0, min(20_000, n_local)), torch.arange(max(0, n_local - 20_000), n_local)]).unique()
        e2e_sample = (r.to(dev), torch.as_tensor(h_out.array)[r].clone())
        e2e = {'value': N_UTT / float(dt.item()), 'unit': UNIT,
               'h2d_bytes_per_step': int(N_UTT) * L_TOK * 8, 'd2h_bytes_per_step': int(N_UTT) * DIM * 4,
               'ms_per_step': float(dt.item()) * 1e3, 'steps': n_e2e,
               # what the copies alone would take on this box's links, measured here on this rank's pinned
               # buffers (H2D of the ids, then D2H of the embeddings: the projection needs the global component,
               # so the two cannot overlap within one split) -- `e2e` as a fraction of that ceiling
               'api': 'mmb_sif_embedding_host (C ABI, pinned host buffers, float32 out)' if world == 1 else
                      ('mmb_sif_embedding_host_peer (C ABI, pinned host buffers per rank, Gram summed over NVLink)'
                       if mdist.default_comm() is not None else
                       'pinned ids -> dist.sharded_sif_embedding -> pinned float32 out, per rank')}
        # copy-only ceiling: the same buffers, the same bytes, no compute; all ranks at once
        d_tmp_i = torch.empty((n_local, L_TOK), dtype=torch.int64, device=dev)
        d_tmp_o = torch.empty((n_local, DIM), dtype=torch.float32, device=dev)
        hi_t, ho_t = torch.as_tensor(h_ids.array), torch.as_tensor(h_out.array)
        d_tmp_i.copy_(hi_t, non_blocking=True)
        ho_t.copy_(d_tmp_o, non_blocking=True)
        best = None
        for _rep in range(3):                     # max over ranks per repetition, best repetition
            rows_per = 1 << 18                    # the pipeline's chunk size: the same copy pattern, minus the compute
            barrier()
            t0 = time.perf_counter()
            for r0 in range(0, n_local, rows_per):
                d_tmp_i[r0:r0 + rows_per].copy_(hi_t[r0:r0 + rows_per], non_blocking=True)
            torch.cuda.synchronize()
            t_h2d = time.perf_counter() - t0
            barrier()
            t0 = time.perf_counter()
            for r0 in range(0, n_local, rows_per):
                ho_t[r0:r0 + rows_per].copy_(d_tmp_o[r0:r0 + rows_per], non_blocking=True)
            torch.cuda.synchronize()
            t_d2h = time.perf_counter() - t0
            cur = torch.tensor([t_h2d, t_d2h], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(cur, op=dist.ReduceOp.MAX)
            best = cur if best is None else torch.minimum(best, cur)
        tt = best
        ceil_s = float(tt.sum().item())
        e2e['copy_ceiling'] = {'h2d_ms': float(tt[0].item()) * 1e3, 'd2h_ms': float(tt[1].item()) * 1e3,
                               'h2d_gbs_aggregate': N_UTT * L_TOK * 8 / float(tt[0].item()) / 1e9,
                               'd2h_gbs_aggregate': N_UTT * DIM * 4 / float(tt[1].item()) / 1e9,
                               'value': N_UTT / ceil_s, 'frac': (N_UTT / float(dt.item())) / (N_UTT / ceil_s),
                               'how': 'H2D of the ids then D2H of the embeddings on the same pinned buffers, all ranks '
                                      'at once in the pipeline\'s 2^18-row chunks, max over ranks, best of 3, no compute; numa: %s' % mdist.numa_note()}
        del d_tmp_i, d_tmp_o
        h_ids.free()
        h_out.free()

    # ---- parity of what was timed ------------------------------------------------------------
    verify = None
    if not args.no_verify:
        verify = verify_run(dict(nv=nv, lib=lib, table=table, vocab_w=vocab_w, ids=ids, emb=emb, pc=pc, lo=lo,
                                 world=world, rank=rank, dev=dev, e2e_sample=e2e_sample))

    # ---- roofline of the dominant kernel + CPU baseline (rank 0) ---------------------------
    peak, peak_src = load_peaks()
    tf32_peak = measure_tf32_peak(dev) if rank == 0 else None
    tf32_src = 'measured here: torch.matmul TF32 8192^3, best of 10'
    if not tf32_peak:
        tf32_peak, tf32_src = load_tensor_peak() / 2.0, 'bf16_tflops / 2 (TF32, assumed)'
    embed_s = stage_ms['embed'] * 1e-3
    rec, rec_src = load_ncu_record(embed_kernel, IDS_KIND)
    traffic = rec['dram_bytes_per_utterance'] * n_local if rec else None
    achieved = n_local * EMBED_BYTES_PER_UTT / embed_s / 1e9
    # compulsory DRAM traffic of one launch: every id once, every table row that is referenced once (bounded by
    # the table), every output row once
    compulsory = n_local * L_TOK * 8 + min(VOCAB, n_local * L_TOK) * DIM * 4 + n_local * DIM * 4
    roofline = {'bound': 'hbm', 'kernel': embed_kernel, 'kernel_source': 'mmb_last_kernel(0): recorded by the dispatch',
                'achieved': achieved, 'peak': peak,
                'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
                'frac_note': 'algorithmic bytes (SURVEY 8d: every token a 1200-byte row, no cache credit) over the '
                             'measured HBM copy rate; above 1 because Zipf ids re-read hot rows from L1/L2 and the '
                             'kernel merges repeated rows of a 32-token chunk -- the HBM side is dram_frac, the '
                             'binding resources are l1_lsu_frac / l2_fabric_frac',
                # what HBM itself carried (ncu DRAM bytes per utterance of the committed capture of THIS kernel
                # on this id distribution x this run's launch time)
                'dram_gbs': (traffic / embed_s / 1e9) if traffic else None,
                'dram_frac': (traffic / embed_s / 1e9 / peak) if traffic else None,
                'traffic_source': rec_src,
                'l1_lsu_frac': rec.get('l1_lsu_wavefronts_pct') / 100.0 if rec and rec.get('l1_lsu_wavefronts_pct') else None,
                'l2_fabric_frac': rec.get('l2_to_l1_pct_of_lts_cap') / 100.0 if rec and rec.get('l2_to_l1_pct_of_lts_cap') else None,
                'compulsory_bytes': compulsory,
                'traffic_over_compulsory': (traffic / compulsory) if traffic else None,
                'compulsory_floor_ms': compulsory / (peak * 1e9) * 1e3,
                'frac_of_compulsory_roofline': compulsory / (peak * 1e9) / embed_s,
                'peak_source': peak_src, 'algorithmic_bytes_per_launch': n_local * EMBED_BYTES_PER_UTT,
                'launch_ms': stage_ms['embed'], 'stage_ms': stage_ms,
                # the other two streaming stages against their own bounds (SURVEY.md 8d): the Gram's
                # algorithmic 2 d^2 FLOP per utterance against the TF32 GEMM rate measured in this run (the 3xTF32
                # kernel executes 2.05x the algorithmic FLOPs), the projection's 2 d 4 bytes per utterance against
                # the measured copy bandwidth
                'other_stages': {
                    'gram': {'bound': 'tensor', 'unit': 'TFLOP/s',
                             'achieved': n_local * 2.0 * DIM * DIM / (stage_ms['gram'] * 1e-3) / 1e12,
                             'peak': tf32_peak, 'peak_source': tf32_src, 'executed_over_algorithmic': 2.05},
                    'project': {'bound': 'hbm', 'unit': 'GB/s',
                                'achieved': n_local * 2.0 * DIM * 4 / (stage_ms['project'] * 1e-3) / 1e9,
                                'peak': peak}}}
    for _st in roofline['other_stages'].values():
        _st['frac'] = _st['achieved'] / _st['peak']

    # ---- the same kernel where HBM IS the bound: ids uniform over the vocabulary (cache-hostile), reduced N ----
    hbm_leg = None
    if rank == 0 and IDS_KIND == 'zipf' and os.environ.get('MMB_BENCH_HBM_LEG', '1') != '0':
        n_u = min(int(os.environ.get('MMB_BENCH_HBM_LEG_N', 2_000_000)), n_local)
        global_kind = globals()['IDS_KIND']
        globals()['IDS_KIND'] = 'uniform'
        try:
            del emb
            torch.cuda.empty_cache()
            ids_u = make_ids(dev, n_u, L_TOK, p, seed=77)
        finally:
            globals()['IDS_KIND'] = global_kind
        ms_u, _e = time_embed_only(lib, nv, table, vocab_w, ids_u)
        k_u = (lib.mmb_last_kernel(0) or b'').decode()
        rec_u, src_u = load_ncu_record(k_u, 'uniform')
        alg = n_u * EMBED_BYTES_PER_UTT / (ms_u * 1e-3) / 1e9
        dram = rec_u['dram_bytes_per_utterance'] * n_u / (ms_u * 1e-3) / 1e9 if rec_u else None
        hbm_leg = {'ids': 'uniform over the %d rows (table %.2f GB > L2), lengths U[16,64], pad id 0' % (VOCAB, VOCAB * DIM * 4 / 1e9),
                   'utterances': n_u, 'kernel': k_u, 'launch_ms': ms_u, 'algorithmic_gbs': alg,
                   'algorithmic_frac': alg / peak,
                   'dram_bytes_per_utterance_ncu': rec_u['dram_bytes_per_utterance'] if rec_u else None,
                   'dram_gbs': dram, 'frac': (dram / peak) if dram else None, 'peak': peak, 'traffic_source': src_u,
                   'note': 'frac = ncu DRAM bytes of the committed capture of this kernel on these ids x this run\'s '
                           'CUDA-event time / measured copy peak; algorithmic_frac > frac because the merged pad run '
                           'and L2 hits are not DRAM traffic'}
        del ids_u, _e
        torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sample = int(os.environ.get('MMB_CPU_SAMPLE', 200_000))       # ~10 s of the reference's Python loops
        sample = min(sample, n_local)
        rate, secs, kind, how = cpu_port_rate(table.cpu().numpy(), vocab_w.double().cpu().numpy(),
                                              ids[:sample].cpu().numpy())
        cpu = {'value': rate, 'unit': UNIT, 'cores': cpu_threads(), 'kind': kind,
               'sample': 'first %d utterances of this workload, %.1f s; %s (BLAS threads = all cores)' % (sample, secs, how)}
    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary:
        del ids
        torch.cuda.empty_cache()
        secondary = {'mmb2_step': mmb_secondary()}
    if world > 1 and not args.no_secondary:
        # SURVEY.md 8e "MMB training" on this process group: the data-parallel latent optimisation must reproduce
        # the reference loop's goldens with the utterances sharded over the ranks (head gradients summed over NVLink
        # peer memory, global-batch mean, synchronised BatchNorm), then one B = 512 step is timed
        try:
            sys.path.insert(0, os.path.join(ROOT, 'tools'))
            sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
            import dp_check
            ok_dp, lines = dp_check.check_goldens(rank, world, dev)
            step = dp_check.time_step(rank, world, dev)
            fl = torch.tensor([0 if ok_dp else 1], device=dev)
            dist.all_reduce(fl)
            secondary = {'mmb2_step_data_parallel': dict(step, goldens_reproduced=int(fl.item()) == 0,
                                                         rank0_checks=lines)}
            if verify is not None:
                verify['dp_mmb_goldens'] = int(fl.item()) == 0
                verify['ok'] = verify['ok'] and verify['dp_mmb_goldens']
        except Exception as e:
            secondary = {'mmb2_step_data_parallel': {'error': '%s: %s' % (type(e).__name__, e)}}
    sampler.stop()

    if rank == 0:
        print(json.dumps({
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'utterances': N_UTT, 'tokens_per_utterance': L_TOK, 'vocab': VOCAB,
                       'dim': DIM, 'ids': ('uniform over the vocabulary (cache-hostile variant)' if IDS_KIND == 'uniform'
                                           else 'Zipf(1.1)') + ', lengths U[16,64], pad id 0', 'npc': 1,
                       'parallelism': 'utterance shards x%d + 1 all-reduce of the 300x300 Gram (%s)' % (
                           world, 'NVLink peer memory, fused into the Gram reduce kernel' if (world > 1 and mdist.default_comm() is not None) else 'NCCL' if world > 1 else 'none at 1 GPU'),
                       'l2': 'inputs larger than L2 (ids %.1f GB + embeddings %.1f GB per rank, table 0.48 GB)'
                             % (n_local * L_TOK * 8 / 1e9, n_local * DIM * 4 / 1e9)},
            'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches,
            'gpu_launches_source': 'mmb_launch_count() around the timed region (%d steps): every launch site of '
                                   'libmmb_b200.so counts itself' % args.steps,
            'verify': verify, 'roofline': roofline, 'roofline_hbm_bound': hbm_leg, 'cpu_baseline': cpu,
            'secondary': secondary,
        }), file=OUT, flush=True)
    if world > 1:
        mdist.close_default_comms()
        dist.destroy_process_group()
    if verify is not None and not verify['ok']:
        sys.stderr.write('bench.py: VERIFY FAILED: %s\n' % json.dumps(verify))
        sys.exit(3)


if __name__ == '__main__':
    main()
