"""SIF fit / transform: components fitted once (mmb_sif_fit_host, sif.fit_sentence_components), then removed from
any utterances' embeddings in one fused pass (mmb_sif_transform, mmb_sif_transform_host,
sif.transform_sentence_embeddings).

The contract is bit identity: the fused pass equals mmb_sif_embed_ws followed by mmb_remove_pc, the host transform
equals the device transform at every chunk size, the host fit equals the components mmb_sif_embedding_host /
mmb_sif_embedding take, and so fit-then-transform on the same utterances is get_sentence_embeddings."""
import os

import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu

EMB_RTOL = 1e-5     # embeddings within 1e-5 relative, as the other SIF tests


@pytest.fixture(scope='module')
def mods():
    import torch
    import _native
    import sif_functions
    import sif
    assert torch.cuda.is_available()
    return _native, sif_functions, sif


def dev_inputs(n, L, V, d, seed, zero_w=None, neg=True):
    """Table, SIF weights and Zipf ids (pad runs, some negative ids, row 1 all negative: an all-zero-weight row)
    as CUDA tensors."""
    import torch
    rng = np.random.default_rng(seed)
    We = cases.table(V, d, seed=seed)
    ids, p = cases.zipf_ids(rng, n, L, V)
    if neg and n > 4:
        flat = ids.reshape(-1)
        pos = rng.choice(flat.size, size=max(2, flat.size // 50), replace=False)
        flat[pos] = -rng.integers(1, V + 1, size=pos.size)
        ids[1, :] = -1
    w = cases.sif_weights(p).astype(np.float32)
    if zero_w is not None:
        w[zero_w] = 0.0
    t = lambda a: torch.as_tensor(a, device='cuda')
    return t(We), t(w), t(ids), ids


def components(npc, d, seed=7):
    """npc unit rows, float32 (CUDA tensor)."""
    import torch
    rng = np.random.default_rng(seed)
    pc = rng.standard_normal((npc, d))
    pc /= np.linalg.norm(pc, axis=1, keepdims=True) if npc else 1.0
    return torch.as_tensor(pc.astype(np.float32), device='cuda')


def two_pass(nv, table_t, w_t, ids_t, pc_t):
    """mmb_sif_embed_ws + mmb_remove_pc with the workspace sif_transform_device allocates."""
    import torch
    n, L = ids_t.shape
    V, d = table_t.shape
    npc = pc_t.shape[0]
    emb = torch.empty((n, d), dtype=torch.float32, device='cuda')
    st = torch.zeros(1, dtype=torch.int32, device='cuda')
    nbytes = nv.lib.mmb_sif_embed_workspace_bytes(V, d, n, L)
    ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda') if nbytes else None
    nv.check(nv.lib.mmb_sif_embed_ws(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.ptr(ids_t), n, L, nv.ptr(emb), nv.ptr(st),
                                     nv.ptr(ws), nbytes, nv.stream_ptr()))
    nv.raise_on_status(st, V)
    if npc:
        nv.check(nv.lib.mmb_remove_pc(nv.ptr(emb), n, d, nv.ptr(pc_t), npc, nv.ptr(emb), nv.stream_ptr()))
    return emb


def same_bits(a, b):
    a = a.cpu().numpy() if hasattr(a, 'cpu') else a
    b = b.cpu().numpy() if hasattr(b, 'cpu') else b
    assert a.shape == b.shape and a.dtype == b.dtype
    return np.array_equal(a.view(np.int32 if a.dtype == np.float32 else np.int64),
                          b.view(np.int32 if b.dtype == np.float32 else np.int64))


def fused_vs_two_pass(mods, table_t, w_t, ids_t, npc, d, kernel=None):
    nv, sf, _ = mods
    pc_t = components(npc, d)
    got = sf.sif_transform_device(table_t, w_t, ids_t, pc_t)
    name = nv.lib.mmb_last_kernel(0).decode()
    want = two_pass(nv, table_t, w_t, ids_t, pc_t)
    assert same_bits(got, want), (d, npc, name)
    if kernel is not None:
        assert kernel in name, name
    if npc:
        assert name.endswith(' +pc f32'), name
    return name


# ---- 1. fused = two passes, bit for bit ----------------------------------------------------------------------
@pytest.mark.parametrize('d', [4, 128, 300, 512, 1024])
@pytest.mark.parametrize('npc', [0, 1, 3, 32])
def test_fused_equals_two_pass_general(mods, d, npc):
    table_t, w_t, ids_t, _ = dev_inputs(300, 20, 1000, d, seed=d + npc)      # N L < 8 V: no pre-scaled table
    fused_vs_two_pass(mods, table_t, w_t, ids_t, npc, d, kernel='sif_embed_warp')
    out = mods[1].sif_transform_device(table_t, w_t, ids_t, components(npc, d))
    assert bool(out[1].isnan().all())                    # the all-zero-weight row: 0 / 0, as NumPy


@pytest.mark.parametrize('d', [128, 300, 512])
@pytest.mark.parametrize('npc', [1, 3])
def test_fused_equals_two_pass_prescaled(mods, d, npc):
    table_t, w_t, ids_t, _ = dev_inputs(4096, 32, 2000, d, seed=3, neg=False)
    fused_vs_two_pass(mods, table_t, w_t, ids_t, npc, d, kernel='sif_embed_prescaled_kernel')


@pytest.mark.parametrize('d', [128, 300])
def test_fused_equals_two_pass_prescaled_standby(mods, d):
    """A zero vocabulary weight: the pre-scaled kernel stands down and the general kernel behind it runs."""
    table_t, w_t, ids_t, _ = dev_inputs(4096, 32, 2000, d, seed=4, zero_w=5)
    fused_vs_two_pass(mods, table_t, w_t, ids_t, 3, d)


@pytest.mark.parametrize('d', [300, 1024])
@pytest.mark.parametrize('npc', [0, 1, 32])
def test_fused_equals_two_pass_cta(mods, d, npc):
    table_t, w_t, ids_t, _ = dev_inputs(100, 300, 800, d, seed=5)
    fused_vs_two_pass(mods, table_t, w_t, ids_t, npc, d, kernel='sif_embed_cta_kernel')


def test_fused_equals_two_pass_wide_table(mods):
    """V * d * 4 >= 4 GiB: 64-bit row offsets."""
    import torch
    d, V = 128, (1 << 23) + 5
    g = torch.Generator(device='cuda')
    g.manual_seed(0)
    table_t = torch.randn((V, d), device='cuda', generator=g)
    w_t = torch.rand(V, device='cuda', generator=g) + 0.01
    ids_t = torch.randint(-V, V, (2000, 16), device='cuda', generator=g)
    ids_t[:, :4] = torch.randint(V - 1000, V, (2000, 4), device='cuda', generator=g)     # rows past 4 GiB
    fused_vs_two_pass(mods, table_t, w_t, ids_t, 1, d, kernel='true>')
    del table_t
    torch.cuda.empty_cache()


def test_fused_bad_index_raises(mods):
    nv, sf, _ = mods
    table_t, w_t, ids_t, _ = dev_inputs(64, 20, 500, 300, seed=6)
    ids_t[3, 2] = 500
    with pytest.raises(IndexError):
        sf.sif_transform_device(table_t, w_t, ids_t, components(1, 300))
    ids_t[3, 2] = -501
    with pytest.raises(IndexError):
        sf.sif_transform_device(table_t, w_t, ids_t, components(1, 300))


# ---- 2. host transform = device transform ----------------------------------------------------------------------
def transform_host(nv, table_t, w_t, ids, pc_t, f64, chunk_rows):
    n, L = ids.shape
    V, d = table_t.shape
    out = np.full((n, d), np.nan, dtype=np.float64 if f64 else np.float32)
    pc = np.ascontiguousarray(pc_t.cpu().numpy())
    rc = nv.lib.mmb_sif_transform_host(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.np_ptr(ids), n, L, nv.np_ptr(pc),
                                       pc.shape[0], nv.np_ptr(out), int(f64), chunk_rows)
    nv.check(rc)
    return out


@pytest.mark.parametrize('shape', [(600, 24, 2000, 300, 3, None), (4096, 32, 2000, 300, 1, None),
                                   (4096, 32, 2000, 300, 2, 5), (500, 12, 300, 1024, 2, None),
                                   (3000, 16, 500, 512, 1, None)],
                         ids=['general', 'prescaled', 'prescaled_standby', 'd1024', 'd512'])
def test_host_transform_equals_device(mods, shape):
    nv, sf, _ = mods
    n, L, V, d, npc, zero_w = shape
    table_t, w_t, ids_t, ids = dev_inputs(n, L, V, d, seed=8, zero_w=zero_w, neg=zero_w is not None or n != 4096)
    pc_t = components(npc, d)
    want = sf.sif_transform_device(table_t, w_t, ids_t, pc_t)
    for chunk_rows in (n, n // 4, n // 3 + 7, 1):
        for f64 in (False, True):
            got = transform_host(nv, table_t, w_t, ids, pc_t, f64, chunk_rows)
            ref = want.double() if f64 else want
            assert same_bits(got, ref), (chunk_rows, f64)


def test_host_transform_npc0_f64_is_widened_embed(mods):
    nv, sf, _ = mods
    table_t, w_t, ids_t, ids = dev_inputs(300, 20, 500, 300, seed=9)
    pc_t = components(0, 300)
    emb = two_pass(nv, table_t, w_t, ids_t, pc_t)
    assert same_bits(transform_host(nv, table_t, w_t, ids, pc_t, True, 77), emb.double())
    assert same_bits(transform_host(nv, table_t, w_t, ids, pc_t, False, 77), emb)


def pom(golden_dir, split):
    g = np.load(os.path.join(golden_dir, 'sif_pom_full.npz'))
    return cases.table(7763, 300, seed=11), g['weights'], g[split + '_ids'].astype(np.int64)


def test_host_transform_pom_chunked_stays_on_cta(mods, golden_dir):
    import torch
    nv, sf, sif = mods
    We, w, ids = pom(golden_dir, 'test')
    table_t = torch.as_tensor(We, device='cuda')
    w_t = torch.as_tensor(w.astype(np.float32), device='cuda')
    pc_t = torch.as_tensor(sif.fit_sentence_components(We, w, ids).astype(np.float32), device='cuda')
    want = sf.sif_transform_device(table_t, w_t, torch.as_tensor(ids, device='cuda'), pc_t)
    assert 'sif_embed_cta_kernel' in nv.lib.mmb_last_kernel(0).decode()
    for chunk_rows in (16, 203, 1):
        for f64 in (False, True):
            got = transform_host(nv, table_t, w_t, ids, pc_t, f64, chunk_rows)
            assert 'sif_embed_cta_kernel' in nv.lib.mmb_last_kernel(0).decode()
            assert same_bits(got, want.double() if f64 else want), (chunk_rows, f64)


def test_host_transform_bad_index(mods):
    nv, sf, _ = mods
    table_t, w_t, ids_t, ids = dev_inputs(300, 20, 500, 300, seed=10)
    ids[250, 3] = 500
    with pytest.raises(IndexError):
        transform_host(nv, table_t, w_t, ids, components(1, 300), False, 64)
    ids[250, 3] = 1
    transform_host(nv, table_t, w_t, ids, components(1, 300), False, 64)     # the next call is clean


# ---- 3. fit from host = the existing host path's components -----------------------------------------------------
def fit_host(nv, sf, table_t, w_t, ids, npc, chunk_rows):
    n, L = ids.shape
    V, d = table_t.shape
    omega = np.ascontiguousarray(sf.start_block(d if n >= d else n, npc))
    pc = np.full((npc, d), np.nan, dtype=np.float32)
    nv.check(nv.lib.mmb_sif_fit_host(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.np_ptr(ids), n, L, npc, nv.np_ptr(omega),
                                     nv.np_ptr(pc), nv.GRAM_AUTO, chunk_rows))
    return pc


def embedding_host_pc(nv, sf, table_t, w_t, ids, npc, chunk_rows):
    n, L = ids.shape
    V, d = table_t.shape
    omega = np.ascontiguousarray(sf.start_block(d if n >= d else n, npc))
    pc = np.full((npc, d), np.nan, dtype=np.float32)
    emb = np.empty((n, d), dtype=np.float32)
    nv.check(nv.lib.mmb_sif_embedding_host(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.np_ptr(ids), n, L, npc,
                                           nv.np_ptr(omega), nv.np_ptr(emb), 0, nv.np_ptr(pc), nv.GRAM_AUTO,
                                           chunk_rows))
    return pc


@pytest.mark.parametrize('shape', [(3000, 24, 500, 300, 1), (3000, 24, 500, 300, 3), (8192, 32, 2000, 300, 1),
                                   (2000, 16, 400, 128, 2)], ids=['npc1', 'npc3', 'prescaled_tc_gram', 'd128'])
def test_fit_host_equals_embedding_host(mods, shape):
    nv, sf, _ = mods
    n, L, V, d, npc = shape
    table_t, w_t, ids_t, ids = dev_inputs(n, L, V, d, seed=12, neg=n != 8192)
    for chunk_rows in (n // 3, 700, 4096):
        assert same_bits(fit_host(nv, sf, table_t, w_t, ids, npc, chunk_rows),
                         embedding_host_pc(nv, sf, table_t, w_t, ids, npc, chunk_rows)), chunk_rows
    _, pc_dev = sf.sif_embedding_device(table_t, w_t, ids_t, npc=npc, return_pc=True)
    assert same_bits(fit_host(nv, sf, table_t, w_t, ids, npc, n), pc_dev)
    assert same_bits(fit_host(nv, sf, table_t, w_t, ids, npc, 0), pc_dev)      # default chunk: 2^18 rows > N


def test_fit_host_few_rows_runs_as_one_chunk(mods):
    """N < d: the start block needs every row, so any chunk_rows gives mmb_sif_embedding's components."""
    nv, sf, _ = mods
    table_t, w_t, ids_t, ids = dev_inputs(100, 24, 500, 300, seed=13)
    _, pc_dev = sf.sif_embedding_device(table_t, w_t, ids_t, npc=2, return_pc=True)
    for chunk_rows in (10, 33, 100):
        assert same_bits(fit_host(nv, sf, table_t, w_t, ids, 2, chunk_rows), pc_dev), chunk_rows


# ---- 4. fit then transform is the reference function ------------------------------------------------------------
@pytest.mark.parametrize('split', ['valid', 'test'])
def test_fit_transform_is_get_sentence_embeddings_pom(mods, golden_dir, split):
    import torch
    nv, sf, sif = mods
    We, w, ids = pom(golden_dir, split)
    want = sif.get_sentence_embeddings(We, w, ids)
    pc = sif.fit_sentence_components(We, w, ids)
    assert pc.dtype == np.float64 and pc.shape == (1, 300)
    assert same_bits(sif.transform_sentence_embeddings(We, w, ids, pc), want)
    # CUDA ids: against the device-resident path
    ids_t = torch.as_tensor(ids, device='cuda')
    pc_t = sif.fit_sentence_components(We, w, ids_t)
    assert pc_t.dtype == torch.float32 and pc_t.is_cuda
    assert same_bits(sif.transform_sentence_embeddings(We, w, ids_t, pc_t), sif.get_sentence_embeddings(We, w, ids_t))


def test_fit_transform_is_get_sentence_embeddings_bench_shape(mods):
    """2 M utterances of bench.py's shape (L = 64, Zipf ids over 400 k words, d = 300): several chunks, the
    pre-scaled kernel and the tensor-core Gram."""
    import torch
    import bench
    nv, sf, sif = mods
    dev = torch.device('cuda', 0)
    table, w_t, p = bench.make_table_and_weights(dev)
    ids = bench.make_ids(dev, 2_000_000, bench.L_TOK, p, seed=3).cpu().numpy()
    We = table.cpu().numpy()
    w = w_t.cpu().numpy()
    want = sif.get_sentence_embeddings(We, w, ids)
    got = sif.transform_sentence_embeddings(We, w, ids, sif.fit_sentence_components(We, w, ids))
    assert same_bits(got, want)
    del want, got
    ids_t = torch.as_tensor(ids[:300_000], device='cuda')
    assert same_bits(sif.transform_sentence_embeddings(We, w, ids_t, sif.fit_sentence_components(We, w, ids_t)),
                     sif.get_sentence_embeddings(We, w, ids_t))


# ---- 5. out of sample, against the float64 oracle ---------------------------------------------------------------
def test_out_of_sample_matches_oracle(mods, golden_dir):
    from oracle import sif_oracle as so
    _, _, sif = mods
    We, w, ids_a = pom(golden_dir, 'valid')
    _, _, ids_b = pom(golden_dir, 'test')
    pc = sif.fit_sentence_components(We, w, ids_a)
    got = sif.transform_sentence_embeddings(We, w, ids_b, pc)
    avg_b = so.get_weighted_average(We, ids_b, so.seq2weight(ids_b, np.ones(ids_b.shape), w))
    want = so.remove_pc_with(avg_b, pc)
    scale = np.abs(want).max(axis=-1, keepdims=True)
    assert float(np.max(np.abs(got - want) / scale)) < EMB_RTOL
    # out= in float32, pinned
    nv = mods[0]
    pin = nv.PinnedArray(got.shape, np.float32)
    assert sif.transform_sentence_embeddings(We, w, ids_b, pc, out=pin.array) is pin.array
    assert same_bits(pin.array.astype(np.float64), got)
    pin.free()


# ---- 6. arguments -----------------------------------------------------------------------------------------------
def test_arguments(mods):
    import torch
    nv, sf, sif = mods
    We = cases.table(50, 16, seed=1)
    w = np.linspace(0.1, 1, 50)
    ids = np.random.default_rng(0).integers(0, 50, size=(20, 6))
    pc = sif.fit_sentence_components(We, w, ids, npc=2)
    with pytest.raises(ValueError):
        sif.transform_sentence_embeddings(We, w, ids, np.zeros((1, 12)))                 # wrong d
    with pytest.raises(ValueError):
        sif.transform_sentence_embeddings(We, w, ids, np.zeros((33, 16)))                # npc > 32
    with pytest.raises(ValueError):
        sif.transform_sentence_embeddings(We, w, ids, pc, out=np.zeros((16, 20)).T)      # not C-contiguous
    with pytest.raises(ValueError):
        sif.transform_sentence_embeddings(We, w, ids, pc, out=np.zeros((20, 15)))        # wrong shape
    with pytest.raises(ValueError):
        sif.transform_sentence_embeddings(We, w, ids, pc, out=np.zeros((20, 16), dtype=np.int64))
    rag = sf.to_ragged(ids)
    with pytest.raises(ValueError):
        sif.transform_sentence_embeddings(We, w, rag, pc)
    with pytest.raises(ValueError):
        sif.fit_sentence_components(We, w, rag)
    with pytest.raises(ValueError):
        sif.fit_sentence_components(We, w, ids, npc=23)
    with pytest.raises(IndexError):                                                      # id beyond a short w
        sif.transform_sentence_embeddings(We, w[:40], np.full((2, 3), 45), pc)
    short = sif.transform_sentence_embeddings(We, w[:40], np.minimum(ids, 39), pc)       # zero-padded w
    assert same_bits(short, sif.transform_sentence_embeddings(We, np.concatenate([w[:40], np.zeros(10)]),
                                                              np.minimum(ids, 39), pc))
    # N = 0 is a no-op
    empty = sif.transform_sentence_embeddings(We, w, np.zeros((0, 6), dtype=np.int64), pc)
    assert empty.shape == (0, 16)
    e_t = sif.transform_sentence_embeddings(We, w, torch.zeros((0, 6), dtype=torch.int64, device='cuda'), pc)
    assert tuple(e_t.shape) == (0, 16)
    with pytest.raises(ValueError):
        sif.fit_sentence_components(We, w, np.zeros((0, 6), dtype=np.int64))
    dev_args = (torch.as_tensor(We, device='cuda'), torch.as_tensor(w.astype(np.float32), device='cuda'),
                torch.as_tensor(ids, device='cuda'), torch.as_tensor(pc.astype(np.float32), device='cuda'))
    for bad in (torch.empty((20, 15), device='cuda'), torch.empty((20, 16), dtype=torch.float64, device='cuda'),
                torch.empty((16, 20), device='cuda').t(), torch.empty((20, 16))):
        with pytest.raises(ValueError):
            sf.sif_transform_device(*dev_args, out=bad)
    # components of either float type, npc = 0 is the plain weighted average
    assert same_bits(sif.transform_sentence_embeddings(We, w, ids, pc.astype(np.float32)),
                     sif.transform_sentence_embeddings(We, w, ids, pc))
    plain = sif.transform_sentence_embeddings(We, w, ids, np.zeros((0, 16)))
    avg = sf.get_weighted_average(We, ids, sf.seq2weight(ids, np.ones(ids.shape), w))
    assert float(np.max(np.abs(plain - avg))) <= 1e-6 * float(np.abs(avg).max())
    # the C entry points reject what Python would not pass
    out = torch.empty((20, 16), device='cuda')
    st = torch.zeros(1, dtype=torch.int32, device='cuda')
    t = lambda a, dt: torch.as_tensor(a, dtype=dt, device='cuda')
    rc = nv.lib.mmb_sif_transform(nv.ptr(t(We, torch.float32)), 50, 16, nv.ptr(t(w, torch.float32)),
                                  nv.ptr(t(ids, torch.int64)), 20, 6, nv.ptr(t(pc, torch.float32)), 33, nv.ptr(out),
                                  nv.ptr(st), None, 0, nv.stream_ptr())
    assert rc == nv.MMB_E_INVALID
