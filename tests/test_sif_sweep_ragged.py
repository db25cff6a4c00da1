"""The SIF sweep on ragged (CSR) ids: K word-weight vectors over one gather of the unpadded tokens
(mmb_sif_embed_multi_ragged), and sif_functions.sif_embedding_sweep / sif.get_sentence_embeddings_sweep on
RaggedIds.

The primary evidence is bit identity: every emb[k] equals mmb_sif_embed_ragged with that k's weights alone, on both
kernel variants (warp- and CTA-per-utterance), every group size and partial last group, with the pad run added in
closed form per vector (pad weight 1, 0 or fractional), interior pad ids, negative ids, duplicate runs, empty
utterances, per-vector divisors and NaN rows."""
import os

import numpy as np
import pytest

import cases
from oracle import sif_oracle as so

EMB_RTOL = 1e-5     # embeddings within 1e-5 relative of the float64 oracle
PAD_W = (1.0, 0.0, 0.37)    # pad weight of vector k: PAD_W[k % 3]


def group_size(d):
    """Weight vectors per gather pass (by row chunks per lane)."""
    return 8 if d <= 256 else (4 if d <= 512 else 2)


def k_values(d):
    kg = group_size(d)
    return sorted({1, 2, 3, kg, kg + 3})


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


def rel_err_t(got, want, block=1 << 18):
    """rel_err on the device, in row blocks (bench-sized outputs)."""
    worst = 0.0
    for s in range(0, want.shape[0], block):
        x, y = got[s:s + block], want[s:s + block]
        scale = y.abs().amax(-1, keepdim=True)
        scale[scale == 0] = 1.0
        worst = max(worst, float(((x - y).abs() / scale).max()))
    return worst


def same_bits(a, b):
    import torch
    return a.shape == b.shape and bool(torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)))


def single_ragged(nv, table_t, w_t, rag):
    """mmb_sif_embed_ragged: the single-vector kernel the ragged sweep must reproduce bit for bit."""
    import torch
    n, L = rag.shape
    V, d = table_t.shape
    emb = torch.empty((n, d), dtype=torch.float32, device=table_t.device)
    st = torch.zeros(1, dtype=torch.int32, device=table_t.device)
    nv.check(nv.lib.mmb_sif_embed_ragged(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.ptr(rag.tokens), nv.ptr(rag.offsets),
                                         n, L, rag.pad_id, nv.ptr(emb), nv.ptr(st), nv.stream_ptr()))
    nv.raise_on_status(st, V)
    return emb


def multi_ragged(nv, table_t, W_t, rag, ws_bytes=None):
    """mmb_sif_embed_multi_ragged -> (K, N, d); returns (rc, emb, status word)."""
    import torch
    n, L = rag.shape
    V, d = table_t.shape
    K = W_t.shape[0]
    dev = table_t.device
    emb = torch.empty((K, n, d), dtype=torch.float32, device=dev)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    nbytes = nv.lib.mmb_sif_embed_multi_workspace_bytes(V, K) if ws_bytes is None else ws_bytes
    ws = torch.empty(max(nbytes, 32), dtype=torch.uint8, device=dev)
    rc = nv.lib.mmb_sif_embed_multi_ragged(nv.ptr(table_t), V, d, nv.ptr(W_t), K, nv.ptr(rag.tokens),
                                           nv.ptr(rag.offsets), n, L, rag.pad_id, nv.ptr(emb), nv.ptr(st), nv.ptr(ws),
                                           nbytes, nv.stream_ptr())
    return rc, emb, int(st.item())


def multi_embed_ok(nv, table_t, W_t, rag):
    rc, emb, st = multi_ragged(nv, table_t, W_t, rag)
    assert rc == nv.MMB_OK and st == 0, (rc, st)
    return emb


def ragged_inputs(n, L, V, d, K, seed):
    """Right-padded Zipf ids (pad id 0) with interior pad ids, negative ids, a duplicate run inside one chunk, an
    utterance that is all padding and a planted NaN table row; K SIF weight vectors for different `a`, pad weight
    PAD_W[k % 3], vector 1 (or 0) with zero entries (its own divisor) and vector K-1 zero on utterance 0's
    tokens (a NaN row where utterance 0 has no weighted padding)."""
    rng = np.random.default_rng(seed)
    We = cases.table(V, d, seed=seed + 7)
    ids, p = cases.zipf_ids(rng, n, L, V)
    ids[(rng.random(ids.shape) < 0.05) & (np.arange(L)[None, :] < L // 2)] = 0     # interior pad ids
    flat = ids.reshape(-1)
    if flat.size >= 4:
        pos = rng.choice(flat.size, size=max(2, flat.size // 50), replace=False)
        flat[pos] = -rng.integers(1, V + 1, size=pos.size)                          # negative ids: wrap, weight 0
    if n > 1 and L > 1:
        ids[1, :min(L, 40)] = V // 2                                                # a run of one row inside a chunk
    if n > 3:
        ids[2] = 0                                                                  # all padding: length 0
    if n > 4 and V > 2:
        ids[4, 0] = V - 1
        We[V - 1] = np.nan                                                          # NaN row through utterance 4
    a = np.geomspace(1e-4, 3e-2, K)
    W = np.stack([cases.sif_weights(p, ak) for ak in a]).astype(np.float32)
    kz = 1 if K > 1 else 0
    W[kz, np.arange(3, V, 3)] = 0.0
    for k in range(K):
        W[k, 0] = PAD_W[k % 3]
    W[K - 1, ids[0][ids[0] > 0]] = 0.0
    return We, ids, W


SHAPES = [(1, 1, 5, 300), (7, 33, 50, 200), (300, 64, 1000, 300), (203, 1357, 7763, 300), (65, 5, 30, 64),
          (5, 300, 20, 128), (33, 9, 30, 512), (9, 260, 12, 512), (3, 300, 20, 200), (40, 200, 30, 512)]


def few_long(n, L):
    import torch
    return L >= 256 and n < 16 * torch.cuda.get_device_properties(0).multi_processor_count


def check_bit_identity(nv, sf, n, L, V, d, seed):
    import torch
    dev = torch.device('cuda')
    for K in k_values(d):
        We, ids, W = ragged_inputs(n, L, V, d, K, seed=seed + K)
        table_t = torch.as_tensor(We, device=dev)
        W_t = torch.as_tensor(W, device=dev)
        rag = sf.to_ragged(ids)
        got = multi_embed_ok(nv, table_t, W_t, rag)
        kname = nv.lib.mmb_last_kernel(1).decode()
        assert 'ragged' in kname, kname
        assert ('cta' in kname) == few_long(n, L), kname
        for k in range(K):
            want = single_ragged(nv, table_t, W_t[k].contiguous(), rag)
            assert same_bits(got[k], want), (n, L, V, d, K, k)
        if n > 4:
            assert bool(torch.isnan(got[:, 4]).all())                 # the NaN table row, every vector


@pytest.mark.gpu
@pytest.mark.parametrize('n,L,V,d', SHAPES)
def test_multi_ragged_bit_identical_to_single_ragged_calls(mods, n, L, V, d):
    """Every K in {1, 2, 3, Kg, Kg + 3}: each group size and a partial last group, both kernel variants."""
    nv, sf, sif = mods
    check_bit_identity(nv, sf, n, L, V, d, seed=n * 31 + L + d)


@pytest.mark.gpu
def test_multi_ragged_long_rows_on_the_warp_kernel(mods):
    """L_pad >= 256 with N >= 16 SMs: long rows, but enough of them for the warp-per-utterance kernel."""
    import torch
    nv, sf, sif = mods
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    check_bit_identity(nv, sf, 16 * sms + 5, 300, 500, 128, seed=17)


@pytest.mark.gpu
def test_multi_ragged_pad_row_edge_values(mods):
    """The pad term's FMA runs even at pad weight 0: a negative pad_id (wraps, weighs 0) whose row is inf gives the
    single kernel's NaN rows, and a -0 row stays bit-equal; a pad_id outside [-V, V) is fine where no utterance
    is padded."""
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    n, L, V, d = 50, 40, 60, 300
    We, ids, W = ragged_inputs(n, L, V, d, 3, seed=5)
    rag = sf.to_ragged(ids)
    W_t = torch.as_tensor(W, device=dev)
    for row in (np.inf, -0.0):
        We2 = We.copy()
        We2[V - 2] = row
        We2[2] = -0.0
        table_t = torch.as_tensor(We2, device=dev)
        for pad_id in (-2, 2):
            r = sf.RaggedIds(rag.tokens, rag.offsets, L, pad_id=pad_id)
            got = multi_embed_ok(nv, table_t, W_t, r)
            for k in range(3):
                assert same_bits(got[k], single_ragged(nv, table_t, W_t[k].contiguous(), r)), (row, pad_id, k)
    full = sf.to_ragged(np.arange(1, 25, dtype=np.int64).reshape(4, 6))
    table_t = torch.as_tensor(We, device=dev)
    r = sf.RaggedIds(full.tokens, full.offsets, 6, pad_id=V + 7)
    got = multi_embed_ok(nv, table_t, W_t, r)
    for k in range(3):
        assert same_bits(got[k], single_ragged(nv, table_t, W_t[k].contiguous(), r))


@pytest.mark.gpu
@pytest.mark.parametrize('n,L,V,d', [(300, 64, 1000, 300), (203, 1357, 7763, 300), (40, 200, 30, 512),
                                     (65, 5, 30, 64)])
def test_multi_ragged_vs_float64_oracle(mods, n, L, V, d):
    """Against the NumPy oracle on the padded matrix the ragged ids stand for; NaN rows match."""
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    K = group_size(d) + 1
    We, ids, W = ragged_inputs(n, L, V, d, K, seed=n + 5 * L)
    rag = sf.to_ragged(ids)
    padded = rag.to_padded().cpu().numpy()
    np.testing.assert_array_equal(padded, ids)
    got = multi_embed_ok(nv, torch.as_tensor(We, device=dev), torch.as_tensor(W, device=dev), rag)
    got = got.double().cpu().numpy()
    for k in range(K):
        w = so.seq2weight(padded, np.ones(padded.shape), W[k])
        with np.errstate(invalid='ignore', divide='ignore'):
            want = so.get_weighted_average(We, padded, w)
        dead = ~np.isfinite(want).all(axis=1)
        assert np.array_equal(dead, ~np.isfinite(got[k]).all(axis=1)), k
        assert rel_err(got[k][~dead], want[~dead]) < EMB_RTOL, k


@pytest.mark.gpu
@pytest.mark.parametrize('n', [400, 229])
def test_ragged_sweep_pipeline_equals_sif_embedding_ragged(mods, n):
    """(k, npc) slice == sif_embedding_ragged(table, W[k], ids, npc) bit for bit, N >= d and N < d; npc = 0 is the
    raw average; a single npc projects in place to the same bits."""
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    L, V, d, K = 24, 900, 300, 3
    rng = np.random.default_rng(n)
    We = cases.table(V, d, seed=n)
    ids, p = cases.zipf_ids(rng, n, L, V)
    W = np.stack([cases.sif_weights(p, a) for a in (3e-4, 1e-3, 1e-2)]).astype(np.float32)
    W[1, 0] = 0.5
    table_t, W_t = torch.as_tensor(We, device=dev), torch.as_tensor(W, device=dev)
    rag = sf.to_ragged(ids)
    npcs = (0, 1, 2, 3)
    out = sf.sif_embedding_sweep(table_t, W_t, rag, npcs=npcs)
    assert out.shape == (K, len(npcs), n, d) and out.dtype == torch.float32
    assert 'ragged' in nv.lib.mmb_last_kernel(1).decode()
    for k in range(K):
        for j, npc in enumerate(npcs):
            want = sf.sif_embedding_ragged(table_t, W_t[k].contiguous(), rag, npc=npc)
            assert same_bits(out[k, j], want), (k, npc)
    one = sf.sif_embedding_sweep(table_t, W_t, rag, npcs=(2,))
    assert one.shape == (K, 1, n, d)
    assert same_bits(one[:, 0], out[:, 2])


@pytest.mark.gpu
@pytest.mark.parametrize('split', ['valid', 'test'])
def test_ragged_sweep_real_pom_fixtures(mods, golden_dir, split):
    """The real POM ids (73 % padding) as CSR ids and the real weights as one of three vectors: the npc = 1 slice
    meets the golden tolerance and agrees with the padded sweep."""
    import torch
    nv, sf, sif = mods
    g = np.load(os.path.join(golden_dir, 'sif_pom_full.npz'))
    ids = g[split + '_ids'].astype(np.int64)
    We = cases.table(7763, 300, seed=11)
    w = np.asarray(g['weights'], dtype=np.float64).reshape(-1)
    vecs = [np.where(np.arange(w.size) % 5 == 0, 0.0, w), w, 0.5 * w]
    rag = sf.to_ragged(ids)
    out = sif.get_sentence_embeddings_sweep(We, vecs, rag, npcs=(1,))
    assert out.is_cuda and out.dtype == torch.float32 and out.shape == (3, 1) + ids.shape[:1] + (300,)
    got = out.double().cpu().numpy()
    assert rel_err(got[1, 0], g[split + '_emb'].astype(np.float64)) < EMB_RTOL
    padded = sif.get_sentence_embeddings_sweep(We, vecs, ids, npcs=(1,))
    for k in range(3):
        ok = np.isfinite(padded[k, 0]).all(axis=1)
        assert np.array_equal(ok, np.isfinite(got[k, 0]).all(axis=1)), k
        assert rel_err(got[k, 0][ok], padded[k, 0][ok]) < EMB_RTOL, k


@pytest.mark.gpu
def test_ragged_sweep_bench_shape(mods):
    """The bench workload's table and Zipf ids at 2 M utterances, converted with to_ragged, K = 4 values of `a`:
    bit-equal to four mmb_sif_embed_ragged calls, and within 2e-6 of the padded mmb_sif_embed_multi."""
    import importlib
    import torch
    nv, sf, sif = mods
    bench = importlib.import_module('bench')
    dev = torch.device('cuda')
    V = 400_000
    table, _w, p = bench.make_table_and_weights(dev, V=V, d=300)
    ids = bench.make_ids(dev, 2_000_000, 64, p, seed=1)
    W = np.empty((4, V), dtype=np.float64)
    W[:, 0] = 1.0
    for k, a in enumerate((1e-4, 3e-4, 1e-3, 3e-3)):
        W[k, 1:] = a / (a + p)
    W_t = torch.as_tensor(W.astype(np.float32), device=dev)
    rag = sf.to_ragged(ids)
    got = multi_embed_ok(nv, table, W_t, rag)
    assert nv.lib.mmb_last_kernel(1).decode().startswith('sif_embed_multi_ragged_warp_kernel<3,4,')
    for k in range(4):
        assert same_bits(got[k], single_ragged(nv, table, W_t[k].contiguous(), rag)), k
    padded = torch.empty_like(got)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    nbytes = nv.lib.mmb_sif_embed_multi_workspace_bytes(V, 4)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    nv.check(nv.lib.mmb_sif_embed_multi(nv.ptr(table), V, 300, nv.ptr(W_t), 4, nv.ptr(ids), ids.shape[0], 64,
                                        nv.ptr(padded), nv.ptr(st), nv.ptr(ws), nbytes, nv.stream_ptr()))
    nv.raise_on_status(st, V)
    for k in range(4):
        assert rel_err_t(got[k], padded[k]) < 2e-6, k


@pytest.mark.gpu
def test_ragged_sweep_errors_and_edges(mods):
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    n, L, V, d, K = 50, 12, 40, 128, 3
    We, ids, W = ragged_inputs(n, L, V, d, K, seed=3)
    table_t, W_t = torch.as_tensor(We, device=dev), torch.as_tensor(W, device=dev)
    rag = sf.to_ragged(ids)
    # a token equal to V
    bad = sf.RaggedIds(rag.tokens.clone(), rag.offsets, L, rag.pad_id)
    bad.tokens[5] = V
    with pytest.raises(IndexError):
        sf.sif_embedding_sweep(table_t, W_t, bad)
    # offsets that claim more tokens than L_pad
    longest = int(rag.lengths().max().item())
    with pytest.raises(IndexError):
        sf.sif_embedding_sweep(table_t, W_t, sf.RaggedIds(rag.tokens, rag.offsets, longest - 1, rag.pad_id))
    # a pad_id outside [-V, V) where utterances are padded
    for pad_id in (V, -V - 1):
        with pytest.raises(IndexError):
            sf.sif_embedding_sweep(table_t, W_t, sf.RaggedIds(rag.tokens, rag.offsets, L, pad_id))
    # too small a workspace; d beyond 512
    rc, _, _ = multi_ragged(nv, table_t, W_t, rag, ws_bytes=64)
    assert rc == nv.MMB_E_INVALID
    wide = torch.zeros((V, 516), dtype=torch.float32, device=dev)
    rc, _, _ = multi_ragged(nv, wide, W_t, rag)
    assert rc == nv.MMB_E_INVALID
    # N = 0
    empty = sf.to_ragged(torch.zeros((0, L), dtype=torch.int64, device=dev))
    out = sf.sif_embedding_sweep(table_t, W_t, empty, npcs=(0, 1))
    assert out.shape == (K, 2, 0, d)
    # a weight vector shorter than the ids reach: through the tokens, or through the pad id alone
    with pytest.raises(IndexError):
        sif.get_sentence_embeddings_sweep(We, [W[0], W[1][:5]], rag)
    small = sf.to_ragged(np.array([[1, 2, 0, 0], [3, 1, 2, 4]], dtype=np.int64), pad_id=0)
    shifted = sf.RaggedIds(small.tokens, small.offsets, 4, pad_id=30)
    with pytest.raises(IndexError):
        sif.get_sentence_embeddings_sweep(We, [W[0], W[1][:20]], shifted, npcs=(0,))
    unpadded = sf.RaggedIds(small.tokens, small.offsets, 2, pad_id=30)
    with pytest.raises(IndexError):     # utterance 1 is longer than L_pad = 2
        sif.get_sentence_embeddings_sweep(We, [W[0], W[1][:20]], unpadded, npcs=(0,))
    exact = sf.to_ragged(np.array([[1, 2], [3, 4]], dtype=np.int64))
    ok = sif.get_sentence_embeddings_sweep(We, [W[0], W[1][:20]], sf.RaggedIds(exact.tokens, exact.offsets, 2, 30),
                                           npcs=(0,))
    assert ok.shape == (2, 1, 2, d) and bool(torch.isfinite(ok).all())
    # deterministic
    a = sf.sif_embedding_sweep(table_t, W_t, rag, npcs=(0, 1))
    b = sf.sif_embedding_sweep(table_t, W_t, rag, npcs=(0, 1))
    assert same_bits(a, b)


def test_ragged_sweep_has_no_cpu_fallback(monkeypatch):
    """Without a CUDA device the sweep on RaggedIds raises; it never computes on the CPU."""
    import torch
    import _native
    import sif
    import sif_functions
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: False)
    rag = sif_functions.RaggedIds(torch.zeros(3, dtype=torch.int64), torch.tensor([0, 1, 3], dtype=torch.int64), 4)
    with pytest.raises(_native.MMBError):
        sif.get_sentence_embeddings_sweep(np.zeros((4, 8), np.float32), np.ones((2, 4)), rag)
