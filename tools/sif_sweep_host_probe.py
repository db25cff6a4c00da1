"""Host-buffer SIF sweep probe: mmb_sif_embedding_sweep_host against the NumPy sweep it replaced and against K x P
single-vector host calls, on bench.py's workload, with the pinned D2H ceiling measured in the same run.

    python tools/sif_sweep_host_probe.py [--ns 1000000,2000000] [--big 10000000] [--reps 2]
        [--out profiles/r06_sif_sweep_host.jsonl]

Workload: bench.py's table (V = 400 k, d = 300) and Zipf ids (L = 64, right-padded), K weight vectors
a / (a + p(w)) with a log-spaced in [1e-4, 1e-2].  Lines:
  * 'd2h_ceiling': a pinned 1 GiB device-to-host copy, best of 3 (tools/pcie_probe.py's method);
  * 'sweep_host' for (K, P) in (1, 1), (4, 1), (4, 3) at each N of --ns, float64 out, each arm timed with a host
    clock around the synchronous call (the last ends in a device synchronise):
      new_pinned_ms   mmb_sif_embedding_sweep_host into a pinned (K, P, N, d) array (pinned ids),
      new_pageable_ms the same into a plain NumPy array,
      old_numpy_ms    the NumPy sweep this entry point replaced: ids uploaded at once, sif_embedding_sweep,
                      .double(), .cpu(),
      kp_single_ms    K x P mmb_sif_embedding_host calls, each into its out[k, j] slice of a pinned array;
    d2h_GB is K P N d 8 / 1e9 and predicted_d2h_ms that over the measured ceiling (a prediction: the D2H alone);
    d2h_fraction_of_ceiling is d2h_GB / new_pinned_ms over the ceiling (the whole call counted, embed included);
    the new path's output is compared with the old path's bit for bit on every 97th utterance;
  * 'sweep_host_big' at N = --big, K = 4, float32 out and P as large as half the host's RAM allows (at most 3),
    the new path only: the old path's device bytes for that size (byte model in the line) exceed the card.
A configuration whose host arrays do not fit half of the host's available RAM is logged as skipped.  Every line
carries the card's name, power limit and SM clock, read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'multimodal-baselines_b200')
for _p in (ROOT, PKG, os.path.join(ROOT, 'tools')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from sif_sweep_probe import gpu_state, stats  # noqa: E402


def host_available():
    with open('/proc/meminfo') as fh:
        for line in fh:
            if line.startswith('MemAvailable:'):
                return int(line.split()[1]) * 1024
    return os.sysconf('SC_AVPHYS_PAGES') * os.sysconf('SC_PAGE_SIZE')


def d2h_ceiling(nv, gb=1.0, reps=3):
    n = int(gb * (1 << 30))
    h = nv.PinnedArray((n,), np.uint8)
    ht = torch.from_numpy(h.array)
    dv = torch.empty(n, dtype=torch.uint8, device='cuda')
    ht.copy_(dv)
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(reps):
        t0 = time.perf_counter()
        ht.copy_(dv, non_blocking=True)
        torch.cuda.synchronize()
        best = max(best, n / (time.perf_counter() - t0))
    del ht
    h.free()
    return best


def old_device_bytes(N, L, K, P, d):
    """Device bytes of the NumPy sweep this entry point replaced: ids, emb (K, N, d), out (K, P, N, d) when
    P > 1 (P = 1 projects in place), and out.double()."""
    return N * (L * 8 + K * d * 4 + (K * P * d * 4 if P > 1 else 0) + K * P * d * 8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ns', default='1000000,2000000')
    ap.add_argument('--big', type=int, default=10_000_000)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r06_sif_sweep_host.jsonl'))
    args = ap.parse_args()
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    import _native as nv
    import sif_functions as sf
    L, V, d = bench.L_TOK, bench.VOCAB, bench.DIM
    table, _w, p = bench.make_table_and_weights(dev, V=V, d=d)
    card = gpu_state(0)
    total_dev = torch.cuda.mem_get_info()[1]

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def emit(line):
        line = dict(line, **card)
        print(json.dumps(line), flush=True)
        with open(args.out, 'a') as fh:
            fh.write(json.dumps(line) + '\n')

    ceiling = d2h_ceiling(nv)
    emit({'probe': 'd2h_ceiling', 'pinned_GBps': round(ceiling / 1e9, 2), 'bytes': 1 << 30})

    def weights(K):
        a = np.geomspace(1e-4, 1e-2, K) if K > 1 else np.array([1e-3])
        return torch.stack([torch.as_tensor(np.concatenate([[1.0], ak / (ak + p)]).astype(np.float32), device=dev)
                            for ak in a]).contiguous()

    def new_call(W, ids, npcs, out):
        K, P = W.shape[0], len(npcs)
        n = ids.shape[0]
        omegas = [np.ascontiguousarray(sf.start_block(d if n >= d else n, q)) if q else None for q in npcs]
        om = (C.c_void_p * P)(*[o.ctypes.data if o is not None else None for o in omegas])
        nv.check(nv.lib.mmb_sif_embedding_sweep_host(nv.ptr(table), V, d, nv.ptr(W), K, nv.np_ptr(ids), n, L, P,
                                                     (C.c_int * P)(*npcs), om, nv.np_ptr(out),
                                                     int(out.dtype == np.float64), nv.GRAM_AUTO, 0))

    def old_call(W, ids, npcs):
        out = sf.sif_embedding_sweep(table, W, torch.as_tensor(ids).to(dev), npcs=npcs)
        return out.double().cpu().numpy()

    def single_calls(W, ids, npcs, out):
        n = ids.shape[0]
        for k in range(W.shape[0]):
            for j, q in enumerate(npcs):
                om = np.ascontiguousarray(sf.start_block(d if n >= d else n, q)) if q else None
                nv.check(nv.lib.mmb_sif_embedding_host(nv.ptr(table), V, d, nv.ptr(W[k]), nv.np_ptr(ids), n, L, q,
                                                       nv.np_ptr(om), nv.np_ptr(out[k, j]), 1, None, nv.GRAM_AUTO, 0))

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    def host_ids(n, seed):
        h = nv.PinnedArray((n, L), np.int64)
        h.array[:] = bench.make_ids(dev, n, L, p, seed=seed).cpu().numpy()
        return h

    for n in [int(x) for x in args.ns.split(',')]:
        ids_h = host_ids(n, seed=1)
        ids = ids_h.array
        for K, npcs in ((1, (1,)), (4, (1,)), (4, (1, 2, 3))):
            P = len(npcs)
            out_bytes = K * P * n * d * 8
            base = {'probe': 'sweep_host', 'n': n, 'L': L, 'V': V, 'd': d, 'K': K, 'npcs': list(npcs),
                    'out_dtype': 'float64', 'd2h_GB': round(out_bytes / 1e9, 3),
                    'old_path_device_GB': round(old_device_bytes(n, L, K, P, d) / 1e9, 2),
                    'new_path_device_GB': round(K * n * d * 4 / 1e9, 2)}
            # pinned out + pageable out + the old path's own result (one at a time) + the single calls' pinned out
            if 3 * out_bytes > 0.5 * host_available():
                emit(dict(base, skipped='needs %.1f GB of host RAM, %.1f GB available'
                          % (3 * out_bytes / 1e9, host_available() / 1e9)))
                continue
            W = weights(K)
            pin = nv.PinnedArray((K, P, n, d), np.float64)
            page = np.empty((K, P, n, d), dtype=np.float64)
            page.fill(0.0)                                   # first touch outside the timed window
            t_pin, t_page, t_old, t_single = [], [], [], []
            new_call(W, ids, npcs, pin.array)                # warm-up (pool, modules)
            for _ in range(args.reps):
                t_pin.append(clock(lambda: new_call(W, ids, npcs, pin.array))[0])
                t_page.append(clock(lambda: new_call(W, ids, npcs, page))[0])
            del page
            nv.lib.mmb_host_pipeline_trim(0)
            same = None
            for r in range(args.reps):
                ms, old = clock(lambda: old_call(W, ids, npcs))
                t_old.append(ms)
                if r == 0:
                    same = bool(np.array_equal(old[:, :, ::97].view(np.int64), pin.array[:, :, ::97].view(np.int64)))
                del old
                torch.cuda.empty_cache()
            single_calls(W, ids, npcs, pin.array)            # warm-up
            for _ in range(args.reps):
                t_single.append(clock(lambda: single_calls(W, ids, npcs, pin.array))[0])
            pin.free()
            nv.lib.mmb_host_pipeline_trim(0)
            med = float(np.median(t_pin))
            emit(dict(base, new_pinned_ms=stats(t_pin), new_pageable_ms=stats(t_page), old_numpy_ms=stats(t_old),
                      kp_single_ms=stats(t_single), predicted_d2h_ms=round(out_bytes / ceiling * 1e3, 1),
                      d2h_fraction_of_ceiling=round(out_bytes / (med * 1e-3) / ceiling, 3),
                      new_over_old_median=round(med / float(np.median(t_old)), 3),
                      new_bits_equal_old_every_97th_row=same))
        ids_h.free()

    # the large batch: new path only
    n, K = args.big, 4
    per_p = K * n * d * 4
    P = int(min(3, (0.5 * host_available() - n * L * 8) // per_p))
    base = {'probe': 'sweep_host_big', 'n': n, 'L': L, 'V': V, 'd': d, 'K': K, 'out_dtype': 'float32',
            'host_available_GB': round(host_available() / 1e9, 1), 'card_GB': round(total_dev / 1e9, 1)}
    if P < 1:
        emit(dict(base, skipped='one (K, 1, N, d) float32 output does not fit half the host RAM'))
    else:
        npcs = tuple(range(1, P + 1))
        old_need = old_device_bytes(n, L, K, P, d)
        ids_h = host_ids(n, seed=2)
        W = weights(K)
        pin = nv.PinnedArray((K, P, n, d), np.float32)
        new_call(W, ids_h.array, npcs, pin.array)
        t = [clock(lambda: new_call(W, ids_h.array, npcs, pin.array))[0] for _ in range(args.reps)]
        out_bytes = K * P * n * d * 4
        med = float(np.median(t))
        emit(dict(base, npcs=list(npcs), new_pinned_ms=stats(t), d2h_GB=round(out_bytes / 1e9, 2),
                  predicted_d2h_ms=round(out_bytes / ceiling * 1e3, 1),
                  d2h_fraction_of_ceiling=round(out_bytes / (med * 1e-3) / ceiling, 3),
                  new_path_device_GB=round(per_p / 1e9, 1),
                  old_path_device_GB_byte_model=round(old_need / 1e9, 1),
                  old_path='not run: its byte model needs %.0f GB of device memory, the card has %.0f GB'
                  % (old_need / 1e9, total_dev / 1e9) if old_need > total_dev else 'fits, not run'))
        pin.free()
        ids_h.free()
    nv.lib.mmb_host_pipeline_trim(0)


if __name__ == '__main__':
    main()
