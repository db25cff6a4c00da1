"""The SIF sweep from host buffers (mmb_sif_embedding_sweep_host, and sif.get_sentence_embeddings_sweep on NumPy ids).

The contract is bit identity: every out[k, j], float32 or float64, equals the device sweep
sif_functions.sif_embedding_sweep(table, W, ids, npcs)[k, j] (widened for float64) at every chunk size: the
chunked embed keeps the variant of the whole batch, the Grams are taken over the whole emb[k], and the projection
only widens on its store."""
import ctypes as C
import os

import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mods():
    import torch
    import _native
    import sif_functions
    import sif
    assert torch.cuda.is_available()
    return _native, sif_functions, sif


def group_size(d):
    """Weight vectors per gather pass of the K-vector embed."""
    return 8 if d <= 256 else (4 if d <= 512 else 2)


def inputs(n, L, V, d, K, seed):
    """Zipf ids with pad runs and some negative ids, K SIF weight vectors for different `a`."""
    rng = np.random.default_rng(seed)
    We = cases.table(V, d, seed=seed)
    ids, p = cases.zipf_ids(rng, n, L, V)
    flat = ids.reshape(-1)
    if flat.size >= 8:
        pos = rng.choice(flat.size, size=max(2, flat.size // 60), replace=False)
        flat[pos] = -rng.integers(1, V + 1, size=pos.size)
    W = np.stack([cases.sif_weights(p, a) for a in np.geomspace(1e-4, 3e-2, K)]).astype(np.float32)
    return We, ids, W


def sweep_host(nv, table_t, W_t, ids, npcs, chunk_rows, f64, out=None, omegas=None):
    """mmb_sif_embedding_sweep_host -> (rc, out)."""
    import sif_functions as sf
    V, d = table_t.shape
    K = W_t.shape[0]
    n, L = ids.shape
    P = len(npcs)
    if out is None:
        out = np.full((K, P, n, d), np.nan, dtype=np.float64 if f64 else np.float32)
    if omegas is None:
        omegas = [np.ascontiguousarray(sf.start_block(d if n >= d else n, p)) if p else None for p in npcs]
    omega_arr = (C.c_void_p * P)(*[o.ctypes.data if o is not None else None for o in omegas])
    rc = nv.lib.mmb_sif_embedding_sweep_host(nv.ptr(table_t), V, d, nv.ptr(W_t), K, nv.np_ptr(ids), n, L, P,
                                             (C.c_int * P)(*npcs), omega_arr, nv.np_ptr(out), int(f64),
                                             nv.GRAM_AUTO, chunk_rows)
    return rc, out


def device_sweep(sf, table_t, W_t, ids, npcs):
    import torch
    return sf.sif_embedding_sweep(table_t, W_t, torch.as_tensor(ids, device=table_t.device), npcs=npcs)


def assert_same_bits(got, ref, what):
    """got: host float32 / float64 array; ref: the device sweep's float32 CUDA tensor."""
    if got.dtype == np.float64:
        want = ref.double().cpu().numpy()
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), what
    else:
        want = ref.cpu().numpy()
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), what


def check(nv, sf, table_t, W_t, ids, npcs, chunks, what):
    torch_ref = device_sweep(sf, table_t, W_t, ids, npcs)
    for chunk_rows in chunks:
        for f64 in (True, False):
            rc, out = sweep_host(nv, table_t, W_t, ids, npcs, chunk_rows, f64)
            nv.check(rc)
            assert_same_bits(out, torch_ref, what + (chunk_rows, f64))


@pytest.mark.parametrize('d', [100, 300, 512, 1024])
def test_bit_identical_at_every_chunk_size(mods, d):
    """chunk_rows in {0 (default), 1, 257, 700, N} with K = Kg + 3 (a full and a partial gather group) and
    npcs (0, 1, 2); then K in {1, Kg} with npcs (0,), (1,) and (0, 1, 2).  The component solve stops at d = 512,
    so d = 1024 removes none."""
    import torch
    nv, sf, _ = mods
    n, L, V = 1100, 20, 3000
    kg = group_size(d)
    npc_sets = [(0,), (1,), (0, 1, 2)] if d <= 512 else [(0,), (0, 0)]
    We, ids, W = inputs(n, L, V, d, kg + 3, seed=d)
    table_t = torch.as_tensor(We, device='cuda')
    W_t = torch.as_tensor(W, device='cuda')
    check(nv, sf, table_t, W_t, ids, npc_sets[-1], (0, 1, 257, 700, n), ('K=Kg+3', d))
    for K in (1, kg):
        Wk = W_t[:K].contiguous()
        for npcs in npc_sets:
            check(nv, sf, table_t, Wk, ids, npcs, (257,), (K, npcs, d))


def test_many_component_sets(mods):
    """P = 10: mmb_remove_pc_multi needs two groups of sets, and one staging chunk holds all ten."""
    import torch
    nv, sf, _ = mods
    We, ids, W = inputs(1500, 24, 2000, 300, 3, seed=7)
    npcs = tuple(j % 4 for j in range(9)) + (22,)
    check(nv, sf, torch.as_tensor(We, device='cuda'), torch.as_tensor(W, device='cuda'), ids, npcs, (0, 700),
          ('P=10',))


def test_fewer_utterances_than_dimensions(mods):
    """N < d: each component solve starts from emb[k]^T Omega over the whole emb[k], not a chunk of it."""
    import torch
    nv, sf, _ = mods
    We, ids, W = inputs(150, 30, 800, 300, 5, seed=8)
    check(nv, sf, torch.as_tensor(We, device='cuda'), torch.as_tensor(W, device='cuda'), ids, (0, 1, 3),
          (0, 1, 64), ('N<d',))


def test_real_pom_split_on_the_cta_kernel(mods, golden_dir):
    """The POM test split (203 utterances of 1357 tokens) takes the CTA-per-utterance embed; in chunks of 16
    utterances it must stay on it, because the variant is decided on the whole batch."""
    import torch
    nv, sf, _ = mods
    g = np.load(os.path.join(golden_dir, 'sif_pom_full.npz'))
    ids = np.ascontiguousarray(g['test_ids'].astype(np.int64))
    assert ids.shape == (203, 1357)
    We = cases.table(7763, 300, seed=11)
    w = np.asarray(g['weights'], dtype=np.float64).reshape(-1)
    W = np.stack([w, 0.5 * w, np.where(np.arange(w.size) % 5 == 0, 0.0, w)]).astype(np.float32)
    table_t, W_t = torch.as_tensor(We, device='cuda'), torch.as_tensor(W, device='cuda')
    ref = device_sweep(sf, table_t, W_t, ids, (0, 1, 2))
    for chunk_rows in (16, 0):
        for f64 in (True, False):
            rc, out = sweep_host(nv, table_t, W_t, ids, (0, 1, 2), chunk_rows, f64)
            nv.check(rc)
            assert nv.lib.mmb_last_kernel(1).decode().startswith('sif_embed_multi_cta_kernel<3,'), chunk_rows
            assert_same_bits(out, ref, ('pom', chunk_rows, f64))


def test_empty_bad_ids_and_argument_errors(mods):
    import torch
    nv, sf, sif = mods
    We, ids, W = inputs(300, 16, 500, 300, 3, seed=9)
    table_t, W_t = torch.as_tensor(We, device='cuda'), torch.as_tensor(W, device='cuda')
    # N = 0: returns at once, nothing written
    empty = np.zeros((0, 16), dtype=np.int64)
    rc, out = sweep_host(nv, table_t, W_t, empty, (0, 1), 0, True)
    assert rc == nv.MMB_OK and out.shape == (3, 2, 0, 300)
    got = sif.get_sentence_embeddings_sweep(We, W, empty, npcs=(0, 1))
    assert got.shape == (3, 2, 0, 300) and got.dtype == np.float64
    # a bad id (>= V, then < -V) is an IndexError after the call has drained, and the next call succeeds
    for bad_id in (500, -501):
        bad = ids.copy()
        bad[200, 3] = bad_id
        rc, _ = sweep_host(nv, table_t, W_t, bad, (0, 1), 64, True)
        assert rc == nv.MMB_E_INDEX, bad_id
        with pytest.raises(IndexError):
            sif.get_sentence_embeddings_sweep(We, W, bad, npcs=(1,))
        check(nv, sf, table_t, W_t, ids, (0, 1), (64,), ('after bad id', bad_id))
    # argument errors
    omegas = [None, np.ascontiguousarray(sf.start_block(300, 1))]

    def rc_of(**kw):
        args = dict(table_t=table_t, W_t=W_t, ids=ids, npcs=(0, 1), chunk_rows=0, f64=True, omegas=omegas)
        args.update(kw)
        return sweep_host(nv, **args)[0]

    assert rc_of(W_t=W_t[:0].contiguous()) == nv.MMB_E_INVALID                          # K = 0
    assert rc_of(npcs=(), omegas=[]) == nv.MMB_E_INVALID                                 # P = 0
    assert rc_of(npcs=(23,), omegas=[np.zeros((300, 33))]) == nv.MMB_E_INVALID          # npc > 22
    assert rc_of(omegas=[None, None]) == nv.MMB_E_INVALID                                # no Omega for npc 1
    t298 = table_t[:, :298].contiguous()
    assert rc_of(table_t=t298, out=np.zeros((3, 2, 300, 298))) == nv.MMB_E_INVALID     # d % 4 != 0
    with pytest.raises(ValueError):
        nv.check(rc_of(npcs=(23,), omegas=[np.zeros((300, 33))]))
    with pytest.raises(ValueError):                                                      # wrong out shape
        sif.get_sentence_embeddings_sweep(We, W, ids, npcs=(1,), out=np.empty((3, 2, 300, 300)))
    with pytest.raises(ValueError):                                                      # out with device ids
        sif.get_sentence_embeddings_sweep(We, W, torch.as_tensor(ids, device='cuda'), npcs=(1,),
                                          out=np.empty((3, 1, 300, 300)))


def test_numpy_entry_fills_a_pinned_out(mods):
    """sif.get_sentence_embeddings_sweep(..., out=PinnedArray) fills and returns that array, float64 and
    float32, with the device sweep's bits; without out it returns a new float64 array with the same bits."""
    import torch
    nv, sf, sif = mods
    We, ids, W = inputs(2500, 32, 4000, 300, 4, seed=10)
    npcs = (0, 1, 3)
    ref = sf.sif_embedding_sweep(torch.as_tensor(We, device='cuda'), torch.as_tensor(W, device='cuda'),
                                 torch.as_tensor(ids, device='cuda'), npcs=npcs)
    for dt in (np.float64, np.float32):
        pinned = nv.PinnedArray((4, 3, 2500, 300), dt)
        try:
            got = sif.get_sentence_embeddings_sweep(We, list(W), ids, npcs=npcs, out=pinned.array)
            assert got is pinned.array
            assert_same_bits(got, ref, ('pinned', dt))
        finally:
            pinned.free()
    plain = sif.get_sentence_embeddings_sweep(We, W, ids, npcs=npcs)
    assert plain.dtype == np.float64
    assert_same_bits(plain, ref, ('plain',))
