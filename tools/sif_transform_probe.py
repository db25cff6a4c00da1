"""SIF fit / transform probe: the fused transform (mmb_sif_transform, mmb_sif_transform_host) and the host fit
(mmb_sif_fit_host) against the two-pass and fit-and-apply paths they stand beside, on bench.py's workload.

    python tools/sif_transform_probe.py [--n 10000000] [--reps 3] [--out profiles/r07_sif_transform.jsonl]

Workload: bench.py's table (V = 400 k, d = 300), SIF weights and Zipf ids (L = 64, right-padded).  Lines:
  * 'copy_ceilings': a pinned 1 GiB H2D alone, D2H alone, and both at once on the one GPU (two streams), best of 3;
  * 'transform_device' for npc in (1, 3): CUDA-event medians of --reps rounds with the arms alternating:
      fused_ms     mmb_sif_transform,
      two_pass_ms  mmb_sif_embed_ws + mmb_remove_pc,
      embed_ms     mmb_sif_embed_ws alone,
    and whether the fused output equals the two-pass output bit for bit;
  * 'transform_host' for float32 and float64 pinned out (pinned ids), host clock around the synchronous calls:
      transform_ms   mmb_sif_transform_host (npc = 1, the components of the split),
      embedding_ms   mmb_sif_embedding_host (npc = 1: fit and apply),
    each set against the serial copy ceiling (H2D of the ids + D2H of the result, one after the other) and the
    concurrent one (both directions at the rates measured together);
  * 'fit_host': mmb_sif_fit_host against mmb_sif_embedding_host (float32 pinned out), with the device bytes of each
    (byte model below), and whether the two components are bit-identical.
Every line carries the card's name, power limit and SM clock, read in the same run.
"""
import argparse
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
from sif_sweep_host_probe import host_available  # noqa: E402


def copy_ceilings(gb=1.0, reps=3):
    """Best-of-reps bytes/s of pinned H2D alone, D2H alone, and of each while the other runs."""
    import _native as nv
    n = int(gb * (1 << 30))
    hin, hout = nv.PinnedArray((n,), np.uint8), nv.PinnedArray((n,), np.uint8)
    t_in, t_out = torch.from_numpy(hin.array), torch.from_numpy(hout.array)
    din, dout = torch.empty(n, dtype=torch.uint8, device='cuda'), torch.empty(n, dtype=torch.uint8, device='cuda')
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def run(h2d, d2h):
        torch.cuda.synchronize()
        ev = []
        for on, st, fn in ((h2d, s_in, lambda: din.copy_(t_in, non_blocking=True)),
                           (d2h, s_out, lambda: t_out.copy_(dout, non_blocking=True))):
            if on:
                with torch.cuda.stream(st):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    fn()
                    b.record()
                    ev.append((a, b))
        torch.cuda.synchronize()
        return [n / (a.elapsed_time(b) * 1e-3) for a, b in ev]

    run(True, True)
    best = {'h2d': 0.0, 'd2h': 0.0, 'both_h2d': 0.0, 'both_d2h': 0.0}
    for _ in range(reps):
        best['h2d'] = max(best['h2d'], run(True, False)[0])
        best['d2h'] = max(best['d2h'], run(False, True)[0])
        a, b = run(True, True)
        best['both_h2d'], best['both_d2h'] = max(best['both_h2d'], a), max(best['both_d2h'], b)
    del t_in, t_out
    hin.free()
    hout.free()
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10_000_000)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r07_sif_transform.jsonl'))
    args = ap.parse_args()
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    import _native as nv
    import sif_functions as sf
    lib = nv.lib
    n, L, V, d = args.n, bench.L_TOK, bench.VOCAB, bench.DIM
    table, w, p = bench.make_table_and_weights(dev, V=V, d=d)
    card = gpu_state(0)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def emit(line):
        line = dict(line, **card)
        print(json.dumps(line), flush=True)
        with open(args.out, 'a') as fh:
            fh.write(json.dumps(line) + '\n')

    c = copy_ceilings()
    emit({'probe': 'copy_ceilings', 'bytes': 1 << 30, 'pinned_h2d_GBps': round(c['h2d'] / 1e9, 2),
          'pinned_d2h_GBps': round(c['d2h'] / 1e9, 2), 'both_at_once_h2d_GBps': round(c['both_h2d'] / 1e9, 2),
          'both_at_once_d2h_GBps': round(c['both_d2h'] / 1e9, 2)})

    # ---- device-resident transform
    ids = bench.make_ids(dev, n, L, p, seed=1)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = lib.mmb_sif_embed_workspace_bytes(V, d, n, L)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
    fused = torch.empty((n, d), dtype=torch.float32, device=dev)
    emb = torch.empty((n, d), dtype=torch.float32, device=dev)
    _, pc3 = sf.sif_embedding_device(table, w, ids[:1_000_000], npc=3, return_pc=True)

    def arm_fused(pc):
        nv.check(lib.mmb_sif_transform(nv.ptr(table), V, d, nv.ptr(w), nv.ptr(ids), n, L, nv.ptr(pc), pc.shape[0],
                                       nv.ptr(fused), nv.ptr(st), nv.ptr(ws), ws_bytes, nv.stream_ptr()))

    def arm_embed(pc=None):
        nv.check(lib.mmb_sif_embed_ws(nv.ptr(table), V, d, nv.ptr(w), nv.ptr(ids), n, L, nv.ptr(emb), nv.ptr(st),
                                      nv.ptr(ws), ws_bytes, nv.stream_ptr()))

    def arm_two_pass(pc):
        arm_embed()
        nv.check(lib.mmb_remove_pc(nv.ptr(emb), n, d, nv.ptr(pc), pc.shape[0], nv.ptr(emb), nv.stream_ptr()))

    def event_ms(fn, pc):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(pc)
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    for npc in (1, 3):
        pc = pc3[:npc].contiguous()
        arms = {'fused_ms': arm_fused, 'two_pass_ms': arm_two_pass, 'embed_ms': arm_embed}
        for fn in arms.values():
            fn(pc)
        t = {k: [] for k in arms}
        for _ in range(max(5, args.reps)):
            for k, fn in arms.items():
                t[k].append(event_ms(fn, pc))
        arm_fused(pc)
        arm_two_pass(pc)
        torch.cuda.synchronize()
        same = bool(torch.equal(fused.view(torch.int32), emb.view(torch.int32)))
        emit(dict({'probe': 'transform_device', 'n': n, 'L': L, 'V': V, 'd': d, 'npc': npc,
                   'kernel': lib.mmb_last_kernel(0).decode(), 'fused_bits_equal_two_pass': same},
                  **{k: stats(v) for k, v in t.items()},
                  fused_over_two_pass_median=round(float(np.median(t['fused_ms']) / np.median(t['two_pass_ms'])), 3),
                  fused_minus_embed_median_ms=round(float(np.median(t['fused_ms']) - np.median(t['embed_ms'])), 2)))
    del fused, emb, ws
    torch.cuda.empty_cache()

    # ---- host buffers
    need = n * L * 8 + n * d * 8 + n * d * 4
    if need > 0.6 * host_available():
        emit({'probe': 'transform_host', 'n': n, 'skipped': 'needs %.1f GB of pinned host memory, %.1f GB available'
              % (need / 1e9, host_available() / 1e9)})
        return
    ids_h = nv.PinnedArray((n, L), np.int64)
    ids_h.array[:] = ids.cpu().numpy()
    del ids
    torch.cuda.empty_cache()
    omega = np.ascontiguousarray(sf.start_block(d, 1))
    pc1 = np.ascontiguousarray(pc3[:1].cpu().numpy())
    ids_bytes = n * L * 8

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    def transform_host(out):
        nv.check(lib.mmb_sif_transform_host(nv.ptr(table), V, d, nv.ptr(w), nv.np_ptr(ids_h.array), n, L,
                                            nv.np_ptr(pc1), 1, nv.np_ptr(out), int(out.dtype == np.float64), 0))

    def embedding_host(out, pc_out=None):
        nv.check(lib.mmb_sif_embedding_host(nv.ptr(table), V, d, nv.ptr(w), nv.np_ptr(ids_h.array), n, L, 1,
                                            nv.np_ptr(omega), nv.np_ptr(out), int(out.dtype == np.float64),
                                            nv.np_ptr(pc_out), nv.GRAM_AUTO, 0))

    for dt in (np.float32, np.float64):
        out = nv.PinnedArray((n, d), dt)
        out_bytes = n * d * np.dtype(dt).itemsize
        transform_host(out.array)
        embedding_host(out.array)
        tt, te = [], []
        for _ in range(args.reps):
            tt.append(clock(lambda: transform_host(out.array)))
            te.append(clock(lambda: embedding_host(out.array)))
        serial = (ids_bytes / c['h2d'] + out_bytes / c['d2h']) * 1e3
        concurrent = max(ids_bytes / c['both_h2d'], out_bytes / c['both_d2h']) * 1e3
        emit({'probe': 'transform_host', 'n': n, 'L': L, 'V': V, 'd': d, 'npc': 1, 'out_dtype': np.dtype(dt).name,
              'out_pinned': True, 'ids_pinned': True, 'h2d_GB': round(ids_bytes / 1e9, 2),
              'd2h_GB': round(out_bytes / 1e9, 2), 'transform_ms': stats(tt), 'embedding_ms': stats(te),
              'serial_copy_ceiling_ms': round(serial, 1), 'concurrent_copy_ceiling_ms': round(concurrent, 1),
              'transform_over_embedding_median': round(float(np.median(tt) / np.median(te)), 3)})
        out.free()
        lib.mmb_host_pipeline_trim(0)

    # ---- fit
    out = nv.PinnedArray((n, d), np.float32)
    pc_fit, pc_emb = np.empty((1, d), np.float32), np.empty((1, d), np.float32)

    def fit_host():
        nv.check(lib.mmb_sif_fit_host(nv.ptr(table), V, d, nv.ptr(w), nv.np_ptr(ids_h.array), n, L, 1,
                                      nv.np_ptr(omega), nv.np_ptr(pc_fit), nv.GRAM_AUTO, 0))

    fit_host()
    embedding_host(out.array, pc_emb)
    tf, te = [], []
    for _ in range(args.reps):
        tf.append(clock(fit_host))
        te.append(clock(lambda: embedding_host(out.array, pc_emb)))
    chunk = min(n, 1 << 18)
    ws = lib.mmb_sif_workspace_bytes(n, d, 1)
    scaled = lib.mmb_sif_embed_workspace_bytes(V, d, n, L)
    fixed = 2 * chunk * L * 8 + ws + scaled + d * 11 * 8 + d * 4 + d * d * 4
    emit({'probe': 'fit_host', 'n': n, 'L': L, 'V': V, 'd': d, 'npc': 1, 'fit_ms': stats(tf), 'embedding_ms': stats(te),
          'h2d_GB': round(ids_bytes / 1e9, 2), 'h2d_ceiling_ms': round(ids_bytes / c['h2d'] * 1e3, 1),
          'fit_pc_bits_equal_embedding_host': bool(np.array_equal(pc_fit.view(np.int32), pc_emb.view(np.int32))),
          'fit_device_bytes_model': '2 chunk L 8 + chunk d 4 + Gram/solve ws + pre-scaled table',
          'fit_device_GB': round((fixed + chunk * d * 4) / 1e9, 3),
          'embedding_device_bytes_model': 'N d 4 + 2 chunk L 8 + Gram/solve ws + pre-scaled table',
          'embedding_device_GB': round((fixed + n * d * 4) / 1e9, 3)})
    out.free()
    ids_h.free()
    lib.mmb_host_pipeline_trim(0)


if __name__ == '__main__':
    main()
