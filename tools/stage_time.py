"""Per-stage device times of the SIF path (embed, tcgen05 Gram, component solve, projection) on a
slice of the bench workload, plus correctness of the Gram and the component solve against float64
torch.  PROFILE_N sets the number of utterances (default 4 M); IDS=uniform draws the ids uniformly
instead of from the bench's Zipf law.  Every output line is tagged with IDS and any MMB_* variable
set, such as MMB_BENCH_V:   PROFILE_N=4000000 python tools/stage_time.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'multimodal-baselines_b200'))
import numpy as np
import torch
import bench
import _native as nv
import sif_functions as sf
from _native import lib

n = int(os.environ.get('PROFILE_N', 4_000_000))
ids_kind = os.environ.get('IDS', 'zipf')
dev = torch.device('cuda')
table, vw, p = bench.make_table_and_weights(dev)
if ids_kind == 'uniform':
    p = np.full(bench.VOCAB - 1, 1.0 / (bench.VOCAB - 1))
ids = bench.make_ids(dev, n, bench.L_TOK, p, seed=1000)
emb = torch.empty((n, 300), device=dev)
st = torch.zeros(1, dtype=torch.int32, device=dev)
torch.cuda.synchronize()


def timed(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def embed():
    nv.check(lib.mmb_sif_embed(nv.ptr(table), table.shape[0], 300, nv.ptr(vw), nv.ptr(ids), n, bench.L_TOK,
                               nv.ptr(emb), nv.ptr(st), nv.stream_ptr()))


tag = ' '.join('%s=%s' % (k, v) for k, v in sorted(os.environ.items()) if k.startswith('MMB_') or k == 'IDS')
ms = timed(embed)
print('[%s] embed   %8.3f ms  n=%d  %.1f M utt/s  %.0f GB/s algorithmic' % (
    tag, ms, n, n / ms / 1e3, n * bench.EMBED_BYTES_PER_UTT / ms / 1e6))
ref = emb.clone()

G = sf.gram(emb, nv.GRAM_TF32X3)
ms = timed(lambda: sf.gram(emb, nv.GRAM_TF32X3))
m = min(n, 400_000)
G64 = emb[:m].double().T @ emb[:m].double()
Gm = sf.gram(emb[:m].contiguous(), nv.GRAM_TF32X3)
G32 = sf.gram(emb[:m].contiguous(), nv.GRAM_FP32)
scale = G64.abs().max().item()
print('[%s] gram    %8.3f ms  %.1f TFLOP/s algorithmic; err vs f64 on %d rows: tc %.2e fp32 %.2e sym %.1e' % (
    tag, ms, n * 180000 / ms / 1e9, m, (Gm.double() - G64).abs().max().item() / scale,
    (G32.double() - G64).abs().max().item() / scale, (Gm - Gm.T).abs().max().item()))

for npc in (1, 3):
    pc = sf.pc_from_gram(G, npc, n)
    ms = timed(lambda: sf.pc_from_gram(G, npc, n), reps=10)
    w, v = torch.linalg.eigh(G.double())
    top = v[:, -npc:].flip(1).T
    cos = (pc.double() * top).sum(1).abs()
    print('[%s] solve   %8.3f ms  npc=%d  |cos| vs eigh(G): %s  norm %s' % (
        tag, ms, npc, ['%.8f' % c for c in cos.tolist()], ['%.6f' % x for x in pc.norm(dim=1).tolist()]))
pc = sf.pc_from_gram(G, 1, n)
ms = timed(lambda: sf.project_out(emb, pc, out=emb))
print('[%s] project %8.3f ms  %.0f GB/s' % (tag, ms, n * 2400 / ms / 1e6))
if os.environ.get('DUMP'):
    torch.save({'emb0': ref[:1000].cpu(), 'G': G.cpu(), 'pc1': sf.pc_from_gram(G, 1, n).cpu(),
                'pc3': sf.pc_from_gram(G, 3, n).cpu()}, os.path.join(ROOT, 'gpurun_out', os.environ['DUMP']))
