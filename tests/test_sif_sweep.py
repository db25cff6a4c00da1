"""The SIF sweep: K word-weight vectors over one gather (mmb_sif_embed_multi) and several numbers of removed
principal components (sif_functions.sif_embedding_sweep, sif.get_sentence_embeddings_sweep).

The primary evidence is bit identity: every emb[k] of the multi-vector kernel equals mmb_sif_embed with that
k's weights alone, on every kernel variant (warp- and CTA-per-utterance), every group size and partial last
group, negative ids, duplicate and pad runs, per-vector divisors and all-zero rows."""
import os

import numpy as np
import pytest

import cases
from oracle import sif_oracle as so

EMB_RTOL = 1e-5     # embeddings within 1e-5 relative of the float64 oracle
PC_COS = 0.9999     # components: |cos| >= 0.9999 up to sign


def group_size(d):
    """Weight vectors per gather pass (mmb_sif_embed_multi: by row chunks per lane)."""
    return 8 if d <= 256 else (4 if d <= 512 else 2)


@pytest.fixture(scope='module')
def mods():
    import torch
    import _native
    import sif_functions
    import sif
    assert torch.cuda.is_available()
    return _native, sif_functions, sif


def rel_err(got, want):
    scale = np.abs(want).max(axis=-1, keepdims=True)
    scale[scale == 0] = 1.0
    return float(np.max(np.abs(got - want) / scale))


def same_bits(a, b):
    import torch
    return a.shape == b.shape and bool(torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)))


def single_embed(nv, table_t, w_t, ids_t):
    """mmb_sif_embed: the general single-vector kernel the sweep must reproduce bit for bit."""
    import torch
    n, L = ids_t.shape
    V, d = table_t.shape
    emb = torch.empty((n, d), dtype=torch.float32, device=table_t.device)
    st = torch.zeros(1, dtype=torch.int32, device=table_t.device)
    nv.check(nv.lib.mmb_sif_embed(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.ptr(ids_t), n, L, nv.ptr(emb), nv.ptr(st),
                                  nv.stream_ptr()))
    nv.raise_on_status(st, V)
    return emb


def multi_embed(nv, table_t, W_t, ids_t):
    """mmb_sif_embed_multi -> (K, N, d)."""
    import torch
    n, L = ids_t.shape
    V, d = table_t.shape
    K = W_t.shape[0]
    dev = table_t.device
    emb = torch.empty((K, n, d), dtype=torch.float32, device=dev)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    nbytes = nv.lib.mmb_sif_embed_multi_workspace_bytes(V, K)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    nv.check(nv.lib.mmb_sif_embed_multi(nv.ptr(table_t), V, d, nv.ptr(W_t), K, nv.ptr(ids_t), n, L, nv.ptr(emb),
                                        nv.ptr(st), nv.ptr(ws), nbytes, nv.stream_ptr()))
    nv.raise_on_status(st, V)
    return emb


def sweep_inputs(n, L, V, d, K, seed):
    """Zipf ids (pad runs of id 0) with negative ids and a duplicate run planted; K SIF weight vectors for
    different `a`, vector 1 (or 0) with zero entries, and one vector whose weights are all zero on row 0."""
    rng = np.random.default_rng(seed)
    We = cases.table(V, d, seed=seed + 7)
    ids, p = cases.zipf_ids(rng, n, L, V)
    flat = ids.reshape(-1)
    if flat.size >= 4:
        pos = rng.choice(flat.size, size=max(2, flat.size // 50), replace=False)
        flat[pos] = -rng.integers(1, V + 1, size=pos.size)            # negative ids: wrap, weight 0
    if n > 1 and L > 1:
        ids[1, :min(L, 40)] = V // 2                                    # a run of one row inside a chunk
    a = np.geomspace(1e-4, 3e-2, K)
    W = np.stack([cases.sif_weights(p, ak) for ak in a]).astype(np.float32)
    kz = 1 if K > 1 else 0
    W[kz, np.arange(0, V, 3)] = 0.0                                     # its own divisor
    W[K - 1, ids[0][ids[0] >= 0]] = 0.0                                 # row 0 all zero for vector K-1 -> NaN
    return We, ids, W


SHAPES = [(1, 1, 5, 300), (7, 33, 50, 300), (300, 64, 1000, 300), (203, 1357, 7763, 300),
          (65, 5, 30, 64), (3, 300, 20, 128), (33, 9, 30, 512), (9, 260, 12, 516), (200, 64, 500, 1024),
          (5, 300, 20, 1024)]


def k_values(d):
    kg = group_size(d)
    return sorted({1, 2, 3, kg, kg + 3})


@pytest.mark.gpu
@pytest.mark.parametrize('n,L,V,d', SHAPES)
def test_multi_embed_bit_identical_to_single_calls(mods, n, L, V, d):
    """Every K in {1, 2, 3, Kg, Kg + 3}: each group size and a partial last group, both kernel variants."""
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    for K in k_values(d):
        We, ids, W = sweep_inputs(n, L, V, d, K, seed=n * 31 + L + d + K)
        table_t = torch.as_tensor(We, device=dev)
        ids_t = torch.as_tensor(ids, device=dev)
        W_t = torch.as_tensor(W, device=dev)
        got = multi_embed(nv, table_t, W_t, ids_t)
        assert nv.lib.mmb_last_kernel(1).decode().startswith('sif_embed_multi_')
        for k in range(K):
            want = single_embed(nv, table_t, W_t[k].contiguous(), ids_t)
            assert same_bits(got[k], want), (n, L, V, d, K, k)
        # the planted all-zero row is the single kernel's NaN row, and the zeroed vector has its own divisor
        assert bool(torch.isnan(got[K - 1, 0]).all())


@pytest.mark.gpu
@pytest.mark.parametrize('n,L,V,d', [(300, 64, 1000, 300), (203, 1357, 7763, 300), (200, 64, 500, 1024),
                                     (65, 5, 30, 64)])
def test_multi_embed_vs_float64_oracle(mods, n, L, V, d):
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    K = group_size(d) + 1
    We, ids, W = sweep_inputs(n, L, V, d, K, seed=n + 5 * L)
    got = multi_embed(nv, torch.as_tensor(We, device=dev), torch.as_tensor(W, device=dev),
                      torch.as_tensor(ids, device=dev)).double().cpu().numpy()
    for k in range(K):
        w = so.seq2weight(ids, np.ones(ids.shape), W[k])
        want = so.get_weighted_average(We, ids, w)
        ok = np.isfinite(want).all(1)
        assert rel_err(got[k][ok], want[ok]) < EMB_RTOL, k
        assert np.isnan(got[k][~ok]).all()


@pytest.mark.gpu
@pytest.mark.parametrize('n', [400, 229])
def test_sweep_pipeline_equals_single_vector_steps(mods, n):
    """(k, npc) slice == project_out(E_k, pc_from_gram(gram(E_k), npc, N, X_t=E_k)) bit for bit, N >= d and N < d
    (transposed start block from that k's own embedding); npc = 0 is the raw average; components agree with
    sklearn's TruncatedSVD."""
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    L, V, d, K = 24, 900, 300, 3
    rng = np.random.default_rng(n)
    We = cases.table(V, d, seed=n)
    ids, p = cases.zipf_ids(rng, n, L, V)
    W = np.stack([cases.sif_weights(p, a) for a in (3e-4, 1e-3, 1e-2)]).astype(np.float32)
    table_t, ids_t, W_t = (torch.as_tensor(x, device=dev) for x in (We, ids, W))
    npcs = (0, 1, 2, 3)
    out = sf.sif_embedding_sweep(table_t, W_t, ids_t, npcs=npcs)
    assert out.shape == (K, len(npcs), n, d) and out.dtype == torch.float32
    for k in range(K):
        E = single_embed(nv, table_t, W_t[k].contiguous(), ids_t)
        G = sf.gram(E)
        E64 = E.double().cpu().numpy()
        assert same_bits(out[k, 0], E)
        for j, npc in enumerate(npcs[1:], start=1):
            pc = sf.pc_from_gram(G, npc, n, X_t=E)
            assert same_bits(out[k, j], sf.project_out(E, pc)), (k, npc)
            want = so.compute_pc(E64, npc)
            got = pc.double().cpu().numpy()
            for i in range(npc):
                c = abs(float(np.dot(got[i], want[i])))
                assert c > PC_COS, (k, npc, i, c)
    # one npc: projected in place, the same bits
    one = sf.sif_embedding_sweep(table_t, W_t, ids_t, npcs=(2,))
    assert one.shape == (K, 1, n, d)
    assert same_bits(one[:, 0], out[:, 2])


@pytest.mark.gpu
@pytest.mark.parametrize('split', ['valid', 'test'])
def test_sweep_real_pom_fixtures(mods, golden_dir, split):
    """The real POM ids and weights as one of three vectors: the npc = 1 slice meets the golden tolerance."""
    nv, sf, sif = mods
    g = np.load(os.path.join(golden_dir, 'sif_pom_full.npz'))
    ids = g[split + '_ids'].astype(np.int64)
    We = cases.table(7763, 300, seed=11)
    w = np.asarray(g['weights'], dtype=np.float64).reshape(-1)
    others = [np.where(np.arange(w.size) % 5 == 0, 0.0, w), 0.5 * w]
    out = sif.get_sentence_embeddings_sweep(We, [others[0], w, others[1]], ids, npcs=(1,))
    assert out.dtype == np.float64 and out.shape == (3, 1) + ids.shape[:1] + (300,)
    assert rel_err(out[1, 0], g[split + '_emb'].astype(np.float64)) < EMB_RTOL


@pytest.mark.gpu
def test_sweep_errors_and_edges(mods):
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    We, ids, W = sweep_inputs(50, 12, 40, 128, 3, seed=3)
    table_t, W_t = torch.as_tensor(We, device=dev), torch.as_tensor(W, device=dev)
    bad = ids.copy()
    bad[4, 2] = 40                                      # id == V
    with pytest.raises(IndexError):
        sf.sif_embedding_sweep(table_t, W_t, torch.as_tensor(bad, device=dev))
    with pytest.raises(IndexError):
        sif.get_sentence_embeddings_sweep(We, W, bad)
    with pytest.raises(IndexError):                    # a vector shorter than the ids reach
        sif.get_sentence_embeddings_sweep(We, [W[0], W[1][:5]], ids)
    # N = 0
    empty = sf.sif_embedding_sweep(table_t, W_t, torch.zeros((0, 12), dtype=torch.int64, device=dev), npcs=(0, 1))
    assert empty.shape == (3, 2, 0, 128)
    # K = 1
    ids_t = torch.as_tensor(ids, device=dev)
    one = sf.sif_embedding_sweep(table_t, W_t[:1].contiguous(), ids_t, npcs=(0,))
    assert same_bits(one[0, 0], single_embed(nv, table_t, W_t[0].contiguous(), ids_t))
    # deterministic
    a = sf.sif_embedding_sweep(table_t, W_t, ids_t, npcs=(0, 1))
    b = sf.sif_embedding_sweep(table_t, W_t, ids_t, npcs=(0, 1))
    assert same_bits(a, b)
    with pytest.raises(ValueError):
        sf.sif_embedding_sweep(table_t, W_t, ids_t, npcs=(23,))
    # too small a workspace is refused
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    emb = torch.empty((3, 50, 128), device=dev)
    ws = torch.empty(64, dtype=torch.uint8, device=dev)
    rc = nv.lib.mmb_sif_embed_multi(nv.ptr(table_t), 40, 128, nv.ptr(W_t), 3, nv.ptr(ids_t), 50, 12, nv.ptr(emb),
                                    nv.ptr(st), nv.ptr(ws), 64, nv.stream_ptr())
    assert rc == nv.MMB_E_INVALID


@pytest.mark.gpu
def test_sweep_bench_shape_bit_identical(mods):
    """The bench workload's table and Zipf ids at 2 M utterances, K = 4 values of `a`: the prefetching warp
    kernel over a multi-wave grid, bit-equal to four mmb_sif_embed calls."""
    import importlib
    import torch
    nv, sf, sif = mods
    bench = importlib.import_module('bench')
    dev = torch.device('cuda')
    table, _w, p = bench.make_table_and_weights(dev, V=400_000, d=300)
    ids = bench.make_ids(dev, 2_000_000, 64, p, seed=1)
    W = np.empty((4, 400_000), dtype=np.float64)
    W[:, 0] = 1.0
    for k, a in enumerate((1e-4, 3e-4, 1e-3, 3e-3)):
        W[k, 1:] = a / (a + p)
    W_t = torch.as_tensor(W.astype(np.float32), device=dev)
    got = multi_embed(nv, table, W_t, ids)
    assert nv.lib.mmb_last_kernel(1).decode().startswith('sif_embed_multi_warp_kernel<3,4,')
    for k in range(4):
        assert same_bits(got[k], single_embed(nv, table, W_t[k].contiguous(), ids)), k


@pytest.mark.gpu
def test_numpy_entry_equals_device_result(mods):
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    We, ids, W = sweep_inputs(120, 20, 300, 300, 5, seed=9)
    host = sif.get_sentence_embeddings_sweep(We, W, ids, npcs=(0, 1))
    assert host.dtype == np.float64 and host.shape == (5, 2, 120, 300)
    devout = sf.sif_embedding_sweep(torch.as_tensor(We, device=dev), torch.as_tensor(W, device=dev),
                                    torch.as_tensor(ids, device=dev), npcs=(0, 1))
    np.testing.assert_array_equal(host, devout.double().cpu().numpy())
    # a sequence of vectors, and CUDA ids in -> float32 CUDA tensor out
    seq = sif.get_sentence_embeddings_sweep(We, list(W.astype(np.float64)), torch.as_tensor(ids, device=dev),
                                            npcs=(0, 1))
    assert seq.is_cuda and seq.dtype == torch.float32
    assert same_bits(seq, devout)


def test_sweep_has_no_cpu_fallback(monkeypatch):
    """Without a CUDA device the sweep raises; it never computes on the CPU."""
    import torch
    import _native
    import sif
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: False)
    with pytest.raises(_native.MMBError):
        sif.get_sentence_embeddings_sweep(np.zeros((4, 8), np.float32), np.ones((2, 4)), np.zeros((2, 3), np.int64))
