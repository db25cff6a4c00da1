"""SIF sweep probe: one K-vector embed (mmb_sif_embed_multi) against K single-vector embeds on the bench workload.

    python tools/sif_sweep_probe.py [--ks 1,2,4,8] [--reps 5] [--out profiles/r03_sif_sweep.jsonl]

Workload: bench.py's (10 M utterances x 64 tokens, V = 400 k, d = 300, Zipf ids, right-padded), MMB_BENCH_N / _L /
_V honoured.  K weight vectors a / (a + p(w)) with a log-spaced in [1e-4, 1e-2] (a = 1e-3 for K = 1).  For every K,
CUDA-event times after one warm-up of each arm:
  (a) one mmb_sif_embed_multi call,
  (b) K x mmb_sif_embed_ws (the production single-vector path: weights folded into a scratch table),
  (c) K x mmb_sif_embed (the general kernel (a) reproduces bit for bit),
  (d) sif_embedding_sweep(npcs=(1,)) against K x sif_embedding_device(npc=1) (embed + Gram + component + projection).
(a) and (b) alternate in the same process, as do the two sides of (d); every arm reports min / median / max over
the repeats.  The table (480 MB) is read from L2 only in part: the ids stream 5 GB per pass and the outputs K x 12 GB.
Each line also carries the card's name, power limit and SM clock read in the same run, the kernel of (a)
(mmb_last_kernel(1)) with its registers (cuobjdump of the built library), the achieved algorithmic bytes/s
(L * 8 + L * d * 4 + K * d * 4 per utterance for (a)), and the output check: (a) bit-equal to (c), max relative
difference to (b).  One JSON line per K, appended to --out.
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'multimodal-baselines_b200')
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402


def gpu_state(index=0):
    """name, power limit and clocks of the card, read now (nvidia-smi, read-only query)."""
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        r = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                           capture_output=True, text=True, timeout=30)
        f = [x.strip() for x in r.stdout.strip().split(',')]
        return {'gpu': f[0], 'power_limit_w': float(f[1]), 'sm_mhz': float(f[2]), 'sm_max_mhz': float(f[3])}
    except Exception as e:                                      # noqa: BLE001
        return {'gpu': torch.cuda.get_device_name(index), 'nvidia_smi_error': repr(e)}


def mangled_args(kname):
    """'sif_embed_multi_warp_kernel<3,4,2,2,false>' -> ('sif_embed_multi_warp_kernel', 'ILi3ELi4ELi2ELi2ELb0EE')."""
    m = re.match(r'(\w+)<([^>]*)>', kname)
    if not m:
        return kname, ''
    parts = []
    for a in m.group(2).split(','):
        a = a.strip()
        parts.append('Lb1E' if a == 'true' else 'Lb0E' if a == 'false' else 'Li%dE' % int(a))
    return m.group(1), 'I' + ''.join(parts) + 'E'


def kernel_registers(lib_path, kname):
    exe = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    try:
        out = subprocess.run([exe, '-res-usage', lib_path], capture_output=True, text=True, timeout=120).stdout
    except Exception:                                           # noqa: BLE001
        return None
    name, args = mangled_args(kname)
    lines = out.splitlines()
    for i, line in enumerate(lines):
        if name in line and args in line and i + 1 < len(lines):
            m = re.search(r'REG:(\d+)', lines[i + 1])
            return int(m.group(1)) if m else None
    return None


def stats(xs):
    xs = sorted(xs)
    return {'min': round(xs[0], 3), 'median': round(float(np.median(xs)), 3), 'max': round(xs[-1], 3)}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def max_rel_diff(a, b, block=1 << 20):
    """max over rows of max|a - b| / max|b| (rows of b that are all zero: scale 1)."""
    worst = 0.0
    for s in range(0, a.shape[0], block):
        x, y = a[s:s + block], b[s:s + block]
        scale = y.abs().amax(1).clamp_min(0)
        scale[scale == 0] = 1.0
        worst = max(worst, float(((x - y).abs().amax(1) / scale).max()))
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ks', default='1,2,4,8')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r03_sif_sweep.jsonl'))
    args = ap.parse_args()
    import _native as nv
    import sif_functions as sf
    lib = nv.lib
    dev = nv.require_cuda()
    N, L, V, d = bench.N_UTT, bench.L_TOK, bench.VOCAB, bench.DIM
    table, _w, p = bench.make_table_and_weights(dev, V=V, d=d)
    ids_full = bench.make_ids(dev, N, L, p, seed=1)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    S = lambda: nv.stream_ptr()                                  # noqa: E731
    out_lines = []
    for K in [int(k) for k in args.ks.split(',')]:
        a = [1e-3] if K == 1 else list(np.geomspace(1e-4, 1e-2, K))
        W = np.empty((K, V), dtype=np.float64)
        W[:, 0] = 1.0
        for k, ak in enumerate(a):
            W[k, 1:] = ak / (ak + p)
        W_t = torch.as_tensor(W.astype(np.float32), device=dev)
        # utterances: the whole workload unless the K outputs, one comparison buffer and the scratch do not fit
        torch.cuda.empty_cache()
        free = torch.cuda.mem_get_info()[0]
        n = N
        while n > 1 and (K + 1) * n * d * 4 + V * d * 4 * 2 + (1 << 30) > free:
            n //= 2
        ids = ids_full[:n]
        emb = torch.empty((K, n, d), dtype=torch.float32, device=dev)
        one = torch.empty((n, d), dtype=torch.float32, device=dev)
        mbytes = lib.mmb_sif_embed_multi_workspace_bytes(V, K)
        mws = torch.empty(mbytes, dtype=torch.uint8, device=dev)
        sbytes = lib.mmb_sif_embed_workspace_bytes(V, d, n, L)
        sws = torch.empty(max(sbytes, 256), dtype=torch.uint8, device=dev)
        wk = [W_t[k].contiguous() for k in range(K)]

        def arm_a():
            nv.check(lib.mmb_sif_embed_multi(nv.ptr(table), V, d, nv.ptr(W_t), K, nv.ptr(ids), n, L, nv.ptr(emb),
                                             nv.ptr(st), nv.ptr(mws), mbytes, S()))

        def arm_b():
            for k in range(K):
                nv.check(lib.mmb_sif_embed_ws(nv.ptr(table), V, d, nv.ptr(wk[k]), nv.ptr(ids), n, L, nv.ptr(one),
                                              nv.ptr(st), nv.ptr(sws), sbytes, S()))

        def arm_c():
            for k in range(K):
                nv.check(lib.mmb_sif_embed(nv.ptr(table), V, d, nv.ptr(wk[k]), nv.ptr(ids), n, L, nv.ptr(one),
                                           nv.ptr(st), S()))

        for f in (arm_a, arm_b, arm_c):
            f()
        torch.cuda.synchronize()
        kname = lib.mmb_last_kernel(1).decode()
        ta, tb, tc = [], [], []
        for _ in range(args.reps):
            ta.append(timed(arm_a))
            tb.append(timed(arm_b))
        for _ in range(args.reps):
            tc.append(timed(arm_c))
        clocks = gpu_state(torch.cuda.current_device())
        nv.raise_on_status(st, V)
        # output check: (a)[k] vs (c) bit for bit, vs (b) relative
        bit_equal, rel_b = True, 0.0
        for k in range(K):
            nv.check(lib.mmb_sif_embed(nv.ptr(table), V, d, nv.ptr(wk[k]), nv.ptr(ids), n, L, nv.ptr(one),
                                       nv.ptr(st), S()))
            bit_equal = bit_equal and bool(torch.equal(emb[k].view(torch.int32), one.view(torch.int32)))
            nv.check(lib.mmb_sif_embed_ws(nv.ptr(table), V, d, nv.ptr(wk[k]), nv.ptr(ids), n, L, nv.ptr(one),
                                          nv.ptr(st), nv.ptr(sws), sbytes, S()))
            rel_b = max(rel_b, max_rel_diff(emb[k], one))
        del emb, one, mws, sws
        torch.cuda.empty_cache()
        # (d) the whole pipeline, npc = 1
        td_sweep, td_single = [], []
        r = sf.sif_embedding_sweep(table, W_t, ids, npcs=(1,))
        del r
        r = sf.sif_embedding_device(table, wk[0], ids, npc=1)
        del r
        def singles():
            for k in range(K):
                sf.sif_embedding_device(table, wk[k], ids, npc=1)

        for _ in range(max(2, args.reps // 2)):
            td_sweep.append(timed(lambda: sf.sif_embedding_sweep(table, W_t, ids, npcs=(1,))))
            torch.cuda.empty_cache()
            td_single.append(timed(singles))
            torch.cuda.empty_cache()
        bytes_a = n * (L * 8 + L * d * 4 + K * d * 4)
        bytes_b = K * n * (L * 8 + L * d * 4 + d * 4)
        ma, mb = float(np.median(ta)), float(np.median(tb))
        line = {
            'probe': 'sif_sweep', 'K': K, 'a': [float('%.3g' % x) for x in a], 'n_utt': n, 'L': L, 'V': V, 'd': d,
            'n_utt_note': 'full workload' if n == N else 'reduced from %d to fit K outputs + comparison buffer' % N,
            **clocks,
            'kernel': kname, 'kernel_registers': kernel_registers(nv.LIB_PATH, kname),
            'reps': args.reps,
            'a_multi_ms': stats(ta), 'b_K_x_embed_ws_ms': stats(tb), 'c_K_x_embed_ms': stats(tc),
            'd_sweep_npc1_ms': stats(td_sweep), 'd_K_x_sif_embedding_device_ms': stats(td_single),
            'a_over_b': round(ma / mb, 3),
            'a_bytes_per_s': round(bytes_a / (ma * 1e-3), 1), 'b_bytes_per_s': round(bytes_b / (mb * 1e-3), 1),
            'check_a_bit_equal_c': bit_equal, 'check_a_max_rel_diff_b': rel_b,
        }
        print(json.dumps(line), flush=True)
        out_lines.append(line)
        del ids, W_t, wk
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'a') as fh:
        for line in out_lines:
            fh.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
