"""GPU parity of the SIF path (rows A1-A5) through the C ABI vs the CPU oracle and the
reference-generated golden fixtures."""
import os

import numpy as np
import pytest

import cases
from oracle import sif_oracle as so

pytestmark = pytest.mark.gpu

EMB_RTOL = 1e-5     # north_star: embeddings within 1e-5 relative
PC_COS = 0.9999     # north_star: |cos| >= 0.9999 up to sign
PC_SOLVE_TOL = 1e-12   # 1 - signed cos of mmb_pc_from_gram vs the oracle on the same Gram (~10x the B200 worst case)


@pytest.fixture(scope='module')
def mods():
    import torch
    import _native
    import sif_functions
    import sif
    assert torch.cuda.is_available()
    assert os.path.exists(_native.LIB_PATH)
    return _native, sif_functions, sif


def rel_err(got, want):
    scale = np.abs(want).max(axis=-1, keepdims=True)
    scale[scale == 0] = 1.0
    return float(np.max(np.abs(got - want) / scale))


def abs_cos(a, b):
    return abs(float(np.dot(a, b) / (np.linalg.norm(a) * np.linalg.norm(b))))


@pytest.mark.parametrize('name', ['sif_mosi_like.npz', 'sif_tall.npz'])
def test_golden_pipeline(mods, golden_dir, name):
    nv, sf, sif = mods
    g = np.load(os.path.join(golden_dir, name))
    We, weights, ids = g['We'], g['weights'], g['ids']
    w = sf.seq2weight(ids, np.ones(ids.shape), weights)
    assert w.dtype == np.float32
    np.testing.assert_array_equal(w, g['w'])                         # lookup: bit-exact
    avg = sf.get_weighted_average(We, ids, w)
    assert avg.dtype == np.float64 and avg.shape == (ids.shape[0], 300)
    assert rel_err(avg[:64], g['avg']) < EMB_RTOL
    pc = sf.compute_pc(avg, 1)
    assert pc.shape == (1, 300) and pc.dtype == np.float64
    assert float(np.dot(pc[0], g['pc'][0])) > PC_COS                 # sign convention too
    emb = sif.get_sentence_embeddings(We, weights, ids)
    assert emb.dtype == np.float64
    assert rel_err(emb[:64], g['emb']) < EMB_RTOL
    p = sf.Params()
    p.rmpc = 1
    emb2 = sf.SIF_embedding(We, ids, w, p)
    assert rel_err(emb2[:64], g['emb']) < EMB_RTOL
    p.rmpc = 0
    assert rel_err(sf.SIF_embedding(We, ids, w, p)[:64], g['avg']) < EMB_RTOL


def test_golden_pom_real_ids(mods, golden_dir):
    """Real POM ids (8 x 1357, right-padded with id 0 whose weight is 1.0) + real weights."""
    nv, sf, sif = mods
    g = np.load(os.path.join(golden_dir, 'sif_pom_real.npz'))
    ids = g['ids'].astype(np.int64)
    We = cases.table(7763, 300, seed=11)
    np.testing.assert_allclose(cases.checksum(We), g['table_sum'], rtol=1e-12)
    w = sf.seq2weight(ids, np.ones(ids.shape), g['weights'])
    np.testing.assert_array_equal(np.count_nonzero(w, axis=1), g['w_nonzero'])
    np.testing.assert_allclose(w.sum(1), g['w_rowsum'], rtol=1e-6)
    avg = sf.get_weighted_average(We, ids, w)                        # CTA-per-utterance kernel
    assert rel_err(avg, g['avg']) < EMB_RTOL
    emb = sif.get_sentence_embeddings(We, g['weights'], ids)
    assert rel_err(emb, g['emb']) < EMB_RTOL


@pytest.mark.parametrize('tag', list(cases.PC_CASES))
@pytest.mark.parametrize('npc', [1, 2, 3])
def test_compute_pc_matches_sklearn(mods, golden_dir, tag, npc):
    nv, sf, sif = mods
    g = np.load(os.path.join(golden_dir, 'pc_cases.npz'))
    n, gap, seed = cases.PC_CASES[tag]
    X = cases.pc_matrix(n, gap, seed)
    pc = sf.compute_pc(X, npc)
    want = g['%s_pc%d' % (tag, npc)]
    assert pc.shape == want.shape
    np.testing.assert_allclose(np.linalg.norm(pc, axis=1), 1.0, atol=1e-5)
    for i in range(npc):
        c = float(np.dot(pc[i], want[i]))
        assert c > PC_COS, (tag, npc, i, c)
    rm = sf.remove_pc(X, npc)
    assert rm.dtype == np.float64
    assert np.max(np.abs(rm[:16] - g['%s_rm%d' % (tag, npc)])) < 2e-4 * np.abs(X).max()


@pytest.mark.parametrize('d,n,npc', [(512, 2048, 22),   # k = 32 at the largest d
                                     (512, 384, 22),    # k = 32, N < d: Rayleigh-Ritz on span(X^T Omega)
                                     (8, 256, 2),       # tiny d: k = 12 > d, dependent columns dropped
                                     (129, 1000, 3),    # odd d
                                     (129, 1000, 1),    # npc = 1: the power-iteration fast path
                                     (129, 64, 1)])     # npc = 1, N < d
def test_pc_from_gram_matches_oracle(mods, d, n, npc):
    """The component solve alone, across its (d, k) range, against the float64 oracle on the same
    float32 Gram and start block.  X has singular values 0.9^i (floored at 0.9^40), so the leading
    eigenvalues of G are well separated and each component is defined to the last bit of float32."""
    import torch
    nv, sf, sif = mods
    rng = np.random.default_rng(d * 1000 + n + npc)
    m = min(n, d)
    P, _ = np.linalg.qr(rng.standard_normal((n, m)))
    U, _ = np.linalg.qr(rng.standard_normal((d, m)))
    X = (P * 0.9 ** np.minimum(np.arange(m), 40)) @ U.T
    G = (X.T @ X).astype(np.float32)
    S0 = X.T @ sf.start_block(n, npc) if n < d else sf.start_block(d, npc)
    dev = torch.device('cuda')
    pc = sf.pc_from_gram(torch.as_tensor(G, device=dev), npc, n, S0_t=torch.as_tensor(S0, device=dev))
    got = pc.double().cpu().numpy()
    want = so.compute_pc_from_gram(G.astype(np.float64), S0, npc, transposed=n < d)
    assert got.shape == want.shape == (npc, d)
    cos = np.sum(got * want, axis=1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(want, axis=1))
    assert np.all(1.0 - cos < PC_SOLVE_TOL), (d, n, npc, 1.0 - cos)


@pytest.mark.parametrize('n,L,V,d', [(1, 1, 5, 300), (7, 33, 50, 300), (300, 64, 1000, 300),
                                     (513, 20, 3016, 300), (40, 700, 400, 300), (65, 5, 30, 64),
                                     (33, 9, 30, 512), (3, 300, 20, 128),
                                     (33, 9, 30, 640), (5, 300, 20, 768), (200, 64, 500, 1024), (9, 260, 12, 516)])
def test_embed_shapes_vs_oracle(mods, n, L, V, d):
    """Ragged/edge shapes, both kernel variants (warp- and CTA-per-utterance), d != 300."""
    nv, sf, sif = mods
    rng = np.random.default_rng(n * 1000 + L)
    We = cases.table(V, d, seed=n + L)
    ids, p = cases.zipf_ids(rng, n, L, V)
    weights = cases.sif_weights(p)
    w = sf.seq2weight(ids, np.ones(ids.shape), weights)
    np.testing.assert_array_equal(w, so.seq2weight(ids, np.ones(ids.shape), weights))
    avg = sf.get_weighted_average(We, ids, w)
    want = so.get_weighted_average(We, ids, w)
    assert rel_err(avg, want) < EMB_RTOL
    # the fused lookup + gather (mmb_sif_embed: the prefetching warp kernel for d <= 512, the one-row-in-flight
    # configuration above) on the same ids, including the table's last rows
    import torch
    dev = torch.device('cuda')
    fused = sf.sif_embedding_device(torch.as_tensor(We, dtype=torch.float32, device=dev),
                                    torch.as_tensor(weights.astype(np.float32), device=dev),
                                    torch.as_tensor(ids, device=dev), npc=0)
    assert rel_err(fused.double().cpu().numpy(), want) < EMB_RTOL


def test_quirks(mods):
    """Pad id counted in the divisor, negative ids, zero weights, all-zero rows, masks."""
    nv, sf, sif = mods
    rng = np.random.default_rng(5)
    V, d = 40, 300
    We = cases.table(V, d, seed=9)
    weights = rng.uniform(0.1, 1.0, V)
    weights[0] = 1.0
    weights[7] = 0.0
    ids = rng.integers(1, V, size=(6, 10)).astype(np.int64)
    ids[0, 5:] = 0                     # padding counts: weight[0] = 1
    ids[1, 2] = -1                     # negative id: weight 0, NumPy wraps the row read
    ids[2, :] = 7                      # all weights zero -> 0/0 -> NaN row
    ids[3, 0] = 7                      # zero-weight token does not count in the divisor
    mask = np.ones(ids.shape)
    mask[4, 3:] = 0                    # masked tokens get weight 0
    w = sf.seq2weight(ids, mask, weights)
    want_w = so.seq2weight(ids, mask, weights)
    np.testing.assert_array_equal(w, want_w)
    with np.errstate(all='ignore'):
        want = so.get_weighted_average(We, ids, want_w)
    got = sf.get_weighted_average(We, ids, w)
    assert np.isnan(got[2]).all() and np.isnan(want[2]).all()
    ok = [0, 1, 3, 4, 5]
    assert rel_err(got[ok], want[ok]) < EMB_RTOL
    # explicit non-zero weight on a negative id: NumPy indexes from the end of the table
    w2 = w.copy()
    w2[1, 2] = 0.5
    assert rel_err(sf.get_weighted_average(We, ids, w2)[1:2], so.get_weighted_average(We, ids, w2)[1:2]) < EMB_RTOL


def test_index_errors(mods):
    nv, sf, sif = mods
    We = cases.table(20, 300, seed=1)
    weights = np.ones(20)
    ids = np.array([[1, 2, 25]], dtype=np.int64)
    with pytest.raises(IndexError):
        sf.seq2weight(ids, np.ones(ids.shape), weights)
    with pytest.raises(IndexError):
        sf.get_weighted_average(We, ids, np.ones(ids.shape, np.float32))
    with pytest.raises(IndexError):
        sif.get_sentence_embeddings(We, weights, ids)
    with pytest.raises(IndexError):
        sf.get_weighted_average(We, np.array([[-21]], dtype=np.int64), np.ones((1, 1), np.float32))


def test_empty_inputs(mods):
    nv, sf, sif = mods
    We = cases.table(20, 300, seed=1)
    assert sf.seq2weight(np.zeros((0, 5), np.int64), np.ones((0, 5)), np.ones(20)).shape == (0, 5)
    assert sf.get_weighted_average(We, np.zeros((0, 5), np.int64), np.zeros((0, 5), np.float32)).shape == (0, 300)


def test_gram_fp32_matches_numpy(mods):
    import torch
    nv, sf, sif = mods
    rng = np.random.default_rng(3)
    for n in (1, 31, 300, 2199, 20000):
        X = rng.standard_normal((n, 300)).astype(np.float32)
        G = sf.gram(torch.as_tensor(X).cuda(), nv.GRAM_FP32).cpu().numpy()
        want = X.astype(np.float64).T @ X.astype(np.float64)
        assert np.max(np.abs(G - want)) < 2e-6 * np.abs(want).max() * max(1, np.sqrt(n) / 30)
        np.testing.assert_array_equal(G, G.T)


def test_large_properties_full_size_slice(mods):
    """Size-independent properties at the bench shape (64 tokens, 400k vocab): after PC
    removal every row is orthogonal to the component, removal is idempotent, and the device
    path is bitwise deterministic."""
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    V, d, n, L = 400_000, 300, 200_000, 64
    table = 0.4 * torch.randn((V, d), device=dev, generator=g) + 0.3 * torch.randn((1, d), device=dev, generator=g)
    table[0] = 0
    u = torch.rand((n, L), device=dev, generator=g)
    ids = (u.pow(6.0) * (V - 1)).long() + 1
    lens = torch.randint(16, L + 1, (n, 1), device=dev, generator=g)
    ids[torch.arange(L, device=dev)[None, :] >= lens] = 0
    vw = torch.rand(V, device=dev, generator=g) * 0.9 + 0.1
    vw[0] = 1.0
    emb, pc = sf.sif_embedding_device(table, vw, ids, npc=1, return_pc=True)
    emb_b, pc_b = sf.sif_embedding_device(table, vw, ids, npc=1, return_pc=True)
    assert torch.equal(emb, emb_b) and torch.equal(pc, pc_b)
    proj = (emb.double() @ pc.double().T).abs().max().item()
    assert proj < 1e-4 * emb.abs().max().item()
    again = sf.project_out(emb, pc)
    assert (again - emb).abs().max().item() < 1e-5 * emb.abs().max().item()
    # spot-check rows against the oracle
    rows = torch.tensor([0, 1, 77777, n - 1], device=dev)
    w_rows = vw[ids[rows]].cpu().numpy()
    avg = so.get_weighted_average(table.cpu().numpy(), ids[rows].cpu().numpy(), w_rows)
    want = so.remove_pc_with(avg, pc.double().cpu().numpy())
    assert rel_err(emb[rows].double().cpu().numpy(), want) < EMB_RTOL


def test_gram_tcgen05_matches_float64(mods):
    """3xTF32 tcgen05 Gram vs float64 and vs the FP32 CUDA-core kernel; ragged K tails."""
    import torch
    nv, sf, sif = mods
    torch.manual_seed(1)
    for n in (1, 15, 16, 17, 300, 4097, 150_001):
        X = (0.4 * torch.randn(n, 300, device='cuda') + 0.3 * torch.randn(1, 300, device='cuda')).contiguous()
        want = X.double().T @ X.double()
        G = sf.gram(X, nv.GRAM_TF32X3)
        scale = want.abs().max().item()
        assert (G.double() - want).abs().max().item() < 2e-5 * scale, n
        assert torch.equal(G, G.T)
        assert torch.equal(G, sf.gram(X, nv.GRAM_TF32X3))            # deterministic
        G32 = sf.gram(X, nv.GRAM_FP32)
        assert (G - G32).abs().max().item() < 2e-5 * scale


def test_peer_exchange_single_rank(mods):
    """The NVLink exchange entry points with world = 1 (the multi-rank case is tools/dist_check.py
    under torchrun, tests/test_dist_gpu.py): the stand-alone all-reduce is the identity, and the
    fused Gram + exchange equals mmb_gram, on both Gram paths, over several epochs (slot parity)."""
    import ctypes as C
    import torch
    nv, sf = mods[0], mods[1]
    lib = nv.lib
    dev = torch.device('cuda')
    buf = C.c_void_p()
    nv.check(lib.mmb_comm_alloc(C.byref(buf)))
    try:
        assert lib.mmb_comm_bytes() >= 2 * 300 * 300 * 4
        handle = (C.c_char * 64)()
        nv.check(lib.mmb_comm_export(buf, handle))
        bufs = (C.c_void_p * 1)(buf.value)
        st = torch.zeros(1, dtype=torch.int32, device=dev)
        g = torch.Generator(device=dev).manual_seed(3)
        epoch = 0
        for n, dtype in ((90000, torch.float32), (3300, torch.float64), (7, torch.float32)):
            x = torch.randn(n, device=dev, generator=g, dtype=dtype)
            want = x.clone()
            epoch += 1
            nv.check(lib.mmb_allreduce_peer(nv.ptr(x), n, int(dtype == torch.float64), 0, 1, bufs,
                                            C.c_uint64(epoch), nv.ptr(st), nv.stream_ptr()))
            assert torch.equal(x, want)
        for n in (157, 5000, 20000):
            X = (0.4 * torch.randn(n, 300, device=dev, generator=g) + 0.3).contiguous()
            want = sf.gram(X)
            G = torch.empty((300, 300), device=dev)
            nbytes = lib.mmb_gram_workspace_bytes(n, 300, 0)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            epoch += 1
            nv.check(lib.mmb_gram_allreduce_peer(nv.ptr(X), n, 300, nv.ptr(G), nv.ptr(ws), nbytes, 0, 0, 1, bufs,
                                                 C.c_uint64(epoch), nv.ptr(st), nv.stream_ptr()))
            assert torch.equal(G, want), n
        assert int(st.item()) == 0
        with pytest.raises(ValueError):
            nv.check(lib.mmb_allreduce_peer(nv.ptr(G), 90000, 0, 0, 1, bufs, C.c_uint64(0), nv.ptr(st),
                                            nv.stream_ptr()))          # epoch must be > 0
    finally:
        torch.cuda.synchronize()
        nv.check(lib.mmb_comm_free(buf))


@pytest.mark.parametrize('chunk_rows', [0, 700, 4096])
def test_host_buffer_api_chunked(mods, chunk_rows):
    """mmb_sif_embedding_host (pinned ids in, embeddings out) with several chunk sizes: the chunked
    pipeline (per-chunk Gram summed in chunk order, projection overlapped with the D2H) gives the
    device-resident result up to the FP32 order of the Gram sum, in float32 and float64 output."""
    import torch
    nv, sf = mods[0], mods[1]
    lib = nv.lib
    dev = torch.device('cuda')
    rng = np.random.default_rng(17)
    V, d, n, L = 5000, 300, 9001, 24
    We = cases.table(V, d, 5)
    ids, p = cases.zipf_ids(rng, n, L, V)
    vw = np.concatenate([[1.0], 1e-3 / (1e-3 + p)]).astype(np.float32)
    t_We, t_vw, t_ids = torch.tensor(We, device=dev), torch.tensor(vw, device=dev), torch.tensor(ids, device=dev)
    want, pc_want = sf.sif_embedding_device(t_We, t_vw, t_ids, npc=1, return_pc=True)
    omega = np.ascontiguousarray(sf.start_block(d, 1))
    ids_c = np.ascontiguousarray(ids, dtype=np.int64)
    for f64 in (0, 1):
        out = np.empty((n, d), dtype=np.float64 if f64 else np.float32)
        pc = np.empty((1, d), dtype=np.float32)
        nv.check(lib.mmb_sif_embedding_host(nv.ptr(t_We), V, d, nv.ptr(t_vw), nv.np_ptr(ids_c), n, L, 1,
                                            nv.np_ptr(omega), nv.np_ptr(out), f64, nv.np_ptr(pc), nv.GRAM_AUTO,
                                            chunk_rows))
        assert abs_cos(pc[0], pc_want[0].cpu().numpy()) > 1 - 1e-9
        assert rel_err(out, want.cpu().numpy().astype(out.dtype)) < 2e-6


@pytest.mark.parametrize('split', ['valid', 'test'])
def test_golden_pom_full_splits(mods, golden_dir, split):
    """BASELINE config 3 at full size: the real POM valid (100 x 1089) and test (203 x 1357) ids and the
    real word weights, reference outputs from tests/golden/make_golden.py::golden_pom_full."""
    nv, sf, sif = mods
    g = np.load(os.path.join(golden_dir, 'sif_pom_full.npz'))
    ids = g[split + '_ids'].astype(np.int64)
    We = cases.table(7763, 300, seed=11)
    w = sf.seq2weight(ids, np.ones(ids.shape), g['weights'])
    np.testing.assert_array_equal(np.count_nonzero(w, axis=1), g[split + '_w_nonzero'])
    avg = sf.get_weighted_average(We, ids, w)
    assert rel_err(avg, g[split + '_avg'].astype(np.float64)) < EMB_RTOL
    pc = sf.compute_pc(avg, 1)
    assert float(np.dot(pc[0], g[split + '_pc'][0])) > PC_COS
    emb = sif.get_sentence_embeddings(We, g['weights'], ids)
    assert rel_err(emb, g[split + '_emb'].astype(np.float64)) < EMB_RTOL


def test_mosi_shape_three_splits(mods):
    """BASELINE configs 0/1, text side: MOSI-shaped splits (1284 / 229 / 686 utterances x 20 tokens,
    3016-row table), the principal component removed per split as simplesif.py:297-299 does -- the
    229-row split takes sklearn's transposed route (N < d), the others the plain one."""
    nv, sf, sif = mods
    rng = np.random.default_rng(2199)
    We = cases.table(3016, 300, seed=3)
    weights = None
    for n in (1284, 229, 686):
        ids, p = cases.zipf_ids(rng, n, 20, 3016)
        if weights is None:
            weights = cases.sif_weights(p)
        got = sif.get_sentence_embeddings(We, weights, ids)
        want = so.get_sentence_embeddings(We, weights, ids)
        assert got.shape == (n, 300) and got.dtype == np.float64
        assert rel_err(got, want) < EMB_RTOL, n


def test_embed_property_random_shapes(mods):
    """Property test (hypothesis): for random shapes, ragged lengths, duplicated / negative / padded ids
    and weights with exact zeros, seq2weight is bit-exact and the weighted average is within tolerance
    of the oracle; rows whose weights are all zero are NaN on both sides."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    nv, sf, sif = mods

    @settings(max_examples=40, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(n=st.integers(1, 70), L=st.integers(1, 130), V=st.integers(2, 300),
           d=st.sampled_from([4, 64, 300, 512, 1024]), seed=st.integers(0, 10 ** 6),
           p_neg=st.sampled_from([0.0, 0.05]), p_zero_w=st.sampled_from([0.0, 0.2]))
    def check(n, L, V, d, seed, p_neg, p_zero_w):
        rng = np.random.default_rng(seed)
        We = rng.standard_normal((V, d)).astype(np.float32)
        weights = rng.uniform(0.01, 1.0, V)
        weights[rng.random(V) < p_zero_w] = 0.0
        ids = rng.integers(0, V, size=(n, L)).astype(np.int64)
        lens = rng.integers(0, L + 1, size=n)
        ids[np.arange(L)[None, :] >= lens[:, None]] = 0
        neg = rng.random(ids.shape) < p_neg
        ids[neg] = -rng.integers(1, V + 1, size=int(neg.sum()))
        mask = (rng.random(ids.shape) < 0.9).astype(np.float64)
        w = sf.seq2weight(ids, mask, weights)
        want_w = so.seq2weight(ids, mask, weights)
        np.testing.assert_array_equal(w, want_w)
        with np.errstate(all='ignore'):
            want = so.get_weighted_average(We, ids, want_w)
        got = sf.get_weighted_average(We, ids, w)
        dead = ~np.isfinite(want).all(axis=1)
        assert (np.isnan(got[dead]).all() if dead.any() else True)
        if (~dead).any():
            assert rel_err(got[~dead], want[~dead]) < EMB_RTOL
    check()


@pytest.mark.parametrize('V,d,L', [(3000, 300, 40), (700, 64, 33), (129, 512, 7)])
def test_fused_lookup_equals_explicit_weights_large(mods, V, d, L):
    """The fused kernel (weights looked up per token, mmb_sif_embed) and the explicit-weight kernel
    (mmb_weighted_average fed with seq2weight's matrix) share one accumulation order, so at a batch large
    enough for the persistent grid-stride loop (several utterances per warp) they must agree bit for bit
    -- including negative ids, zero weights and an out-of-range id being reported."""
    import torch
    nv, sf = mods[0], mods[1]
    lib = nv.lib
    dev = torch.device('cuda')
    n = 70_000
    rng = np.random.default_rng(V + d)
    We = cases.table(V, d, seed=V)
    ids, p = cases.zipf_ids(rng, n, L, V)
    weights = cases.sif_weights(p)
    weights[rng.integers(1, V, 5)] = 0.0
    weights[rng.integers(1, V, 5)] = rng.uniform(0, 1, 5)          # out-of-order weights
    neg = rng.random(ids.shape) < 0.01
    ids[neg] = -rng.integers(1, V + 1, size=int(neg.sum()))
    t_We = torch.tensor(We, device=dev)
    t_vw = torch.tensor(weights.astype(np.float32), device=dev)
    t_ids = torch.tensor(ids, device=dev)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    hot = torch.empty((n, d), device=dev)
    nv.check(lib.mmb_sif_embed(nv.ptr(t_We), V, d, nv.ptr(t_vw), nv.ptr(t_ids), n, L, nv.ptr(hot), nv.ptr(st),
                               nv.stream_ptr()))
    w = torch.empty((n, L), device=dev)
    nv.check(lib.mmb_seq2weight(nv.ptr(t_ids), None, nv.ptr(t_vw), V, n, L, nv.ptr(w), nv.ptr(st), nv.stream_ptr()))
    plain = torch.empty((n, d), device=dev)
    nv.check(lib.mmb_weighted_average(nv.ptr(t_We), V, d, nv.ptr(t_ids), nv.ptr(w), n, L, nv.ptr(plain), nv.ptr(st),
                                      nv.stream_ptr()))
    assert int(st.item()) == 0
    assert torch.equal(torch.nan_to_num(hot, nan=12345.0), torch.nan_to_num(plain, nan=12345.0))
    rows = np.array([0, 1, 4242, n - 1])
    with np.errstate(all='ignore'):
        want = so.get_weighted_average(We, ids[rows], so.seq2weight(ids[rows], np.ones((4, L)), weights))
    ok = np.isfinite(want).all(axis=1)
    assert rel_err(hot[rows].double().cpu().numpy()[ok], want[ok]) < EMB_RTOL
    # an id outside [-V, V) is still reported
    t_ids[5, 0] = V + 3
    nv.check(lib.mmb_sif_embed(nv.ptr(t_We), V, d, nv.ptr(t_vw), nv.ptr(t_ids), n, L, nv.ptr(hot), nv.ptr(st),
                               nv.stream_ptr()))
    assert int(st.item()) & nv.STATUS_BAD_INDEX


# --------------------------------------------------------------------------------------------------
# SURVEY.md 8f N3: ragged (CSR) ids, device-side masks

@pytest.mark.parametrize('split', ['valid', 'test'])
def test_ragged_ids_equal_padded_reference_pom(mods, golden_dir, split):
    """The real POM splits (73 % padding, pad id 0 with weight 1.0) as CSR ids: same embeddings as the
    reference computed on the padded matrix -- the pad run is added in closed form, the divisor still counts it."""
    import torch
    nv, sf, sif = mods
    g = np.load(os.path.join(golden_dir, 'sif_pom_full.npz'))
    ids = g[split + '_ids'].astype(np.int64)
    We = cases.table(7763, 300, seed=11)
    rag = sf.to_ragged(ids)
    lens = rag.lengths().cpu().numpy()
    want_lens = np.array([np.max(np.nonzero(r)[0]) + 1 if r.any() else 0 for r in ids])
    np.testing.assert_array_equal(lens, want_lens)                              # offsets: bit-exact
    np.testing.assert_array_equal(rag.to_padded().cpu().numpy(), ids)           # lossless round trip
    assert int(rag.tokens.numel()) == int(want_lens.sum()) < ids.size // 2
    dev = torch.device('cuda')
    t_We = torch.tensor(We, device=dev)
    t_w = torch.tensor(g['weights'].astype(np.float32), device=dev)
    avg = sf.sif_embedding_ragged(t_We, t_w, rag, npc=0)
    assert rel_err(avg.double().cpu().numpy(), g[split + '_avg'].astype(np.float64)) < EMB_RTOL
    emb = sif.get_sentence_embeddings(We, g['weights'], rag)                    # the drop-in call takes RaggedIds
    assert rel_err(emb.double().cpu().numpy(), g[split + '_emb'].astype(np.float64)) < EMB_RTOL


@pytest.mark.parametrize('n,L,V,d,w0', [(300, 64, 900, 300, 1.0), (77, 33, 50, 128, 0.0), (5000, 64, 4000, 300, 0.25),
                                        (9, 1, 7, 64, 1.0), (40, 200, 30, 512, 1.0)])
def test_ragged_ids_vs_oracle(mods, n, L, V, d, w0):
    """Ragged ids against the NumPy oracle on the padded matrix: pad weight 1 / 0 / fractional, interior pad
    ids (the shared OOV row), empty utterances (all pad -> the divisor is L or 0 -> NaN as in NumPy)."""
    import torch
    nv, sf, sif = mods
    rng = np.random.default_rng(n + L)
    We = cases.table(V, d, seed=n)
    ids, p = cases.zipf_ids(rng, n, L, V)
    ids[rng.random(ids.shape) < 0.05] = 0            # interior zeros
    if n > 3:
        ids[2] = 0                                   # an utterance that is all padding
    weights = cases.sif_weights(p)
    weights[0] = w0
    w = so.seq2weight(ids, np.ones(ids.shape), weights)
    with np.errstate(invalid='ignore', divide='ignore'):
        want = so.get_weighted_average(We, ids, w)
    dev = torch.device('cuda')
    rag = sf.to_ragged(ids)
    np.testing.assert_array_equal(rag.to_padded().cpu().numpy(), ids)
    got = sf.sif_embedding_ragged(torch.tensor(We, device=dev), torch.tensor(weights.astype(np.float32), device=dev),
                                  rag, npc=0).double().cpu().numpy()
    dead = ~np.isfinite(want).all(axis=1)
    assert np.array_equal(dead, ~np.isfinite(got).all(axis=1))
    assert rel_err(got[~dead], want[~dead]) < EMB_RTOL
    # and the full pipeline equals the padded device call
    if n >= 300:
        a = sf.sif_embedding_ragged(torch.tensor(We, device=dev), torch.tensor(weights.astype(np.float32), device=dev),
                                    rag, npc=1)
        b = sf.sif_embedding_device(torch.tensor(We, device=dev), torch.tensor(weights.astype(np.float32), device=dev),
                                    torch.tensor(ids, device=dev), npc=1)
        ok = torch.isfinite(b).all(dim=1)
        assert rel_err(a[ok].double().cpu().numpy(), b[ok].double().cpu().numpy()) < EMB_RTOL


def test_device_masks_equal_reference_masks(mods, capsys):
    """update_masks / update_masks_vect (reference simplesif.py:36-47) on the device."""
    import torch
    import simplesif
    rng = np.random.default_rng(4)
    ids = rng.integers(0, 5, size=(37, 21)).astype(np.int64)
    m_ref, m_dev = {}, {}
    simplesif.update_masks(m_ref, ids, 12)
    simplesif.update_masks_device(m_dev, ids, 12)
    assert tuple(m_dev['text'].shape) == m_ref['text'].shape and m_dev['text'].stride(-1) == 0
    np.testing.assert_array_equal(m_dev['text'].cpu().numpy(), m_ref['text'].astype(np.float32))
    x = rng.standard_normal((19, 23, 45)).astype(np.float32)
    x[rng.random(x.shape) < 0.01] = 0.0
    x[:, 20:, :] = 0.0
    simplesif.update_masks_vect(m_ref, x, 'text_align')
    simplesif.update_masks_vect_device(m_dev, x, 'text_align')
    np.testing.assert_array_equal(m_dev['text_align'].cpu().numpy(), m_ref['text_align'].astype(np.float32))
    capsys.readouterr()


def test_prescaled_table_path_equals_general_kernel(mods):
    """Large batches fold the vocabulary weights into a scratch copy of the table (mmb_sif_embed_ws): same
    averages as the general kernel and the oracle (one extra rounding per term); a zero vocabulary weight
    hands the batch to the general kernel (the divisor must not count that token); negative ids wrap like
    NumPy and do not count; an out-of-range id still raises."""
    import torch
    nv, sf, sif = mods
    lib = nv.lib
    dev = torch.device('cuda')
    rng = np.random.default_rng(12)
    V, d, n, L = 2000, 300, 4000, 64                      # N * L = 256,000 >= 8 V
    We = cases.table(V, d, seed=3)
    ids, p = cases.zipf_ids(rng, n, L, V)
    ids[5, 3] = -7                                         # NumPy: row V - 7, weight 0
    weights = cases.sif_weights(p).astype(np.float32)
    t_We, t_ids = torch.tensor(We, device=dev), torch.tensor(ids, device=dev)

    def run(w_np, ids_t, use_ws):
        t_w = torch.tensor(w_np, device=dev)
        emb = torch.empty((ids_t.shape[0], d), dtype=torch.float32, device=dev)
        st = torch.zeros(1, dtype=torch.int32, device=dev)
        nbytes = lib.mmb_sif_embed_workspace_bytes(V, d, ids_t.shape[0], L) if use_ws else 0
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
        nv.check(lib.mmb_sif_embed_ws(nv.ptr(t_We), V, d, nv.ptr(t_w), nv.ptr(ids_t), ids_t.shape[0], L, nv.ptr(emb),
                                      nv.ptr(st), nv.ptr(ws) if use_ws else None, nbytes, nv.stream_ptr()))
        return emb, int(st.item()), nbytes, (lib.mmb_last_kernel(0) or b'').decode()

    fast, st, nbytes, kname = run(weights, t_ids, True)
    assert nbytes >= V * d * 4 and st == 0 and 'prescaled' in kname
    plain, st2, _, kname2 = run(weights, t_ids, False)
    assert st2 == 0 and 'prescaled' not in kname2
    w = so.seq2weight(ids, np.ones(ids.shape), weights.astype(np.float64))
    want = so.get_weighted_average(We, ids, w)
    assert rel_err(fast.double().cpu().numpy(), want) < EMB_RTOL
    assert rel_err(plain.double().cpu().numpy(), want) < EMB_RTOL
    assert rel_err(fast.double().cpu().numpy(), plain.double().cpu().numpy()) < 2e-6
    again, _, _, _ = run(weights, t_ids, True)
    assert torch.equal(fast, again)                        # deterministic
    # a zero weight somewhere in the vocabulary: the stand-by general kernel does the work, exactly
    wz = weights.copy()
    wz[ids[0, 0]] = 0.0
    fz, stz, _, _ = run(wz, t_ids, True)
    pz, _, _, _ = run(wz, t_ids, False)
    assert stz == 0 and torch.equal(fz, pz)
    wq = so.seq2weight(ids, np.ones(ids.shape), wz.astype(np.float64))
    assert rel_err(fz.double().cpu().numpy(), so.get_weighted_average(We, ids, wq)) < EMB_RTOL
    # an id outside [-V, V)
    bad = t_ids.clone()
    bad[17, 2] = V + 3
    _, stb, _, _ = run(weights, bad, True)
    assert stb & nv.STATUS_BAD_INDEX
    # too small a batch: no scratch requested, plain kernel
    assert lib.mmb_sif_embed_workspace_bytes(V, d, 10, L) == 0


def test_ragged_equals_padded_at_bench_shape(mods):
    """Size-independent property at the bench shape (64 tokens, 400 k vocabulary, 200 k utterances): the CSR path
    (padded -> lengths -> offsets -> compacted tokens -> mmb_sif_embed_ragged) gives the padded path's averages, the
    conversion is lossless, the offsets are the exclusive scan of the lengths, and an empty batch is a no-op."""
    import torch
    nv, sf, sif = mods
    dev = torch.device('cuda')
    g = torch.Generator(device=dev)
    g.manual_seed(3)
    V, d, n, L = 400_000, 300, 200_000, 64
    table = 0.4 * torch.randn((V, d), device=dev, generator=g) + 0.3 * torch.randn((1, d), device=dev, generator=g)
    ids = (torch.rand((n, L), device=dev, generator=g).pow(6.0) * (V - 1)).long() + 1
    lens = torch.randint(0, L + 1, (n, 1), device=dev, generator=g)          # includes empty utterances
    ids[torch.arange(L, device=dev)[None, :] >= lens] = 0
    vw = torch.rand(V, device=dev, generator=g) * 0.9 + 0.1
    vw[0] = 1.0
    rag = sf.to_ragged(ids)
    assert torch.equal(rag.lengths(), lens[:, 0])
    assert torch.equal(rag.offsets, torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), lens[:, 0].cumsum(0)]))
    assert torch.equal(rag.to_padded(), ids)
    a = sf.sif_embedding_ragged(table, vw, rag, npc=0)
    b = sf.sif_embedding_device(table, vw, ids, npc=0)
    assert rel_err(a.double().cpu().numpy(), b.double().cpu().numpy()) < 2e-6
    a2 = sf.sif_embedding_ragged(table, vw, rag, npc=0)
    assert torch.equal(a, a2)                                                  # deterministic
    empty = sf.to_ragged(torch.zeros((0, L), dtype=torch.int64, device=dev))
    assert empty.shape == (0, L) and int(empty.tokens.numel()) == 0
    assert sf.sif_embedding_ragged(table, vw, empty, npc=0).shape == (0, d)


def test_full_size_properties_10M(mods):
    """BASELINE configs[3] at FULL size (10 M utterances x 64 tokens, 400 k vocabulary, d = 300) through the composed
    device call: bitwise determinism, every output row orthogonal to the removed component, the component a unit
    vector with sklearn's sign rule, and sampled rows (first, last, and 62 in between) equal to the NumPy oracle's
    weighted average projected with that component.  (bench.py's `verify` block repeats this at every GPU count.)"""
    import torch
    import bench
    nv, sf, sif = mods
    dev = torch.device('cuda')
    torch.cuda.empty_cache()
    free, _total = torch.cuda.mem_get_info()
    if free < 60 * (1 << 30):
        pytest.skip('needs ~45 GB of device memory')
    n, L, V, d = 10_000_000, 64, 400_000, 300
    table, vw, p = bench.make_table_and_weights(dev, V=V, d=d)
    ids = bench.make_ids(dev, n, L, p, seed=2024)
    emb, pc = sf.sif_embedding_device(table, vw, ids, npc=1, return_pc=True)
    emb2, pc2 = sf.sif_embedding_device(table, vw, ids, npc=1, return_pc=True)
    assert torch.equal(pc, pc2) and torch.equal(emb, emb2)
    del emb2
    assert abs(float(pc.double().norm()) - 1.0) < 1e-6
    assert float(pc[0, pc[0].abs().argmax()]) > 0                                  # svd_flip(u_based_decision=False)
    worst = 0.0
    for s0 in range(0, n, 1 << 21):
        blk = emb[s0:s0 + (1 << 21)]
        worst = max(worst, float((blk @ pc[0]).abs().max()) / float(blk.abs().max()))
    assert worst < 1e-4
    rows = torch.cat([torch.tensor([0, n - 1]), torch.randint(1, n - 1, (62,), generator=torch.Generator().manual_seed(1))]).to(dev)
    ids_s = ids[rows]
    uniq, inv = torch.unique(ids_s, return_inverse=True)                            # a small table of the rows they touch
    We_s = table[uniq].cpu().numpy()
    w_s = vw[uniq].double().cpu().numpy()
    ids_np = inv.cpu().numpy()
    w = so.seq2weight(ids_np, np.ones(ids_np.shape), w_s)
    avg = so.get_weighted_average(We_s, ids_np, w)
    want = so.remove_pc_with(avg, pc.double().cpu().numpy())
    got = emb[rows].double().cpu().numpy()
    del emb, ids, table
    torch.cuda.empty_cache()
    assert rel_err(got, want) < EMB_RTOL
