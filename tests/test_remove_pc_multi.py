"""mmb_remove_pc_multi (P component sets against one read of X) and the sweep stages built on it.

The contract is bit identity: out[j] equals mmb_remove_pc(X, pc[j], npc[j]) bit for bit, and X itself for
npc[j] = 0, for every row-chunk class of the kernel, every grouping of the sets into launches and in place
at P = 1.  sif_dist.sharded_sif_embedding_sweep without a process group is the single-GPU sweep bit for bit."""
import ctypes as C

import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mods():
    import torch
    import _native
    import sif_functions
    import sif_dist
    assert torch.cuda.is_available()
    return _native, sif_functions, sif_dist


def same_bits(a, b):
    import torch
    return a.shape == b.shape and bool(torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)))


def components(rng, npc, d, dev):
    import torch
    pc = rng.standard_normal((max(npc, 1), d))
    pc /= np.linalg.norm(pc, axis=1, keepdims=True)
    return torch.as_tensor(pc[:npc].astype(np.float32), device=dev) if npc else None


def remove_pc_multi(nv, X, pcs, npcs, outs):
    n, d = X.shape
    P = len(npcs)
    pc_arr = (C.c_void_p * P)(*[p.data_ptr() if p is not None else None for p in pcs])
    out_arr = (C.c_void_p * P)(*[o.data_ptr() if o is not None else None for o in outs])
    return nv.lib.mmb_remove_pc_multi(nv.ptr(X), n, d, P, pc_arr, (C.c_int * P)(*npcs), out_arr, nv.stream_ptr())


def single(nv, X, pc):
    import torch
    out = torch.empty_like(X)
    nv.check(nv.lib.mmb_remove_pc(nv.ptr(X), X.shape[0], X.shape[1], nv.ptr(pc), pc.shape[0], nv.ptr(out),
                                  nv.stream_ptr()))
    return out


def check_sets(nv, X, npcs, seed, want_launches=None):
    import torch
    rng = np.random.default_rng(seed)
    pcs = [components(rng, p, X.shape[1], X.device) for p in npcs]
    outs = [torch.full_like(X, float('nan')) for _ in npcs]
    before = nv.lib.mmb_launch_count()
    nv.check(remove_pc_multi(nv, X, pcs, npcs, outs))
    launches = nv.lib.mmb_launch_count() - before
    if want_launches is not None:
        assert launches == want_launches, (npcs, launches)
    for j, p in enumerate(npcs):
        want = X if p == 0 else single(nv, X, pcs[j])
        assert same_bits(outs[j], want), (X.shape, npcs, j)


@pytest.mark.parametrize('d', [128, 256, 300, 512, 1024])
def test_bit_identical_to_single_calls(mods, d):
    """Every NCH class (1, 2, 3, 4, 8 float4 chunks per lane), npc sets mixing 0 with 1..22."""
    import torch
    nv, _, _ = mods
    X = torch.as_tensor(cases.table(3001, d, seed=d), device='cuda')
    X[5] = -0.0                                          # signed zeros pass through the npc = 0 column
    for npcs in [(0, 1, 3), (1,), (22, 0, 2, 5), (0,), (0, 0)]:
        check_sets(nv, X, npcs, seed=d + len(npcs))


def test_in_place_at_one_set(mods):
    import torch
    nv, _, _ = mods
    rng = np.random.default_rng(1)
    for d, npc in ((300, 1), (300, 3), (1024, 22), (300, 0)):
        X = torch.as_tensor(cases.table(2000, d, seed=d + npc), device='cuda')
        pc = components(rng, npc, d, X.device)
        want = X.clone() if npc == 0 else single(nv, X, pc)
        nv.check(remove_pc_multi(nv, X, [pc], [npc], [X]))
        assert same_bits(X, want), (d, npc)


def test_several_groups(mods):
    """More than 8 sets, and sets whose components overflow one launch's 128 KB of shared memory at d = 1024:
    the entry point splits them into consecutive groups, one launch each, with the same bits."""
    import torch
    nv, _, _ = mods
    X = torch.as_tensor(cases.table(1500, 300, seed=3), device='cuda')
    check_sets(nv, X, tuple(j % 4 for j in range(11)), seed=4, want_launches=2)
    check_sets(nv, X, tuple([2] * 17), seed=5, want_launches=3)
    X = torch.as_tensor(cases.table(1500, 1024, seed=6), device='cuda')
    check_sets(nv, X, (22, 22, 22), seed=7, want_launches=3)     # 88 KB each: one set per launch
    check_sets(nv, X, (32, 0, 32), seed=8, want_launches=2)      # 128 KB + an empty set, then 128 KB
    check_sets(nv, X, (1, 3, 22), seed=9, want_launches=1)


def test_empty_and_argument_errors(mods):
    import torch
    nv, _, _ = mods
    X = torch.zeros((0, 300), device='cuda')
    before = nv.lib.mmb_launch_count()
    assert remove_pc_multi(nv, X, [None, None], [0, 0], [X.clone(), X.clone()]) == nv.MMB_OK
    assert nv.lib.mmb_launch_count() == before
    X = torch.randn((64, 300), device='cuda')
    pc = torch.randn((2, 300), device='cuda')
    o1, o2 = torch.empty_like(X), torch.empty_like(X)
    bad = [
        (X, [pc], [33], [o1]),                     # npc > 32
        (X, [pc], [-1], [o1]),                     # npc < 0
        (X, [None], [2], [o1]),                    # components missing
        (X, [pc, pc], [2, 2], [o1, None]),         # output missing
        (X, [pc, pc], [2, 1], [o1, X]),            # in place needs P == 1
        (X[:, :298].contiguous(), [pc[:, :298].contiguous()], [1], [o1]),   # d % 4
    ]
    for args in bad:
        assert remove_pc_multi(nv, *args) == nv.MMB_E_INVALID, args[2]
    big = torch.zeros((4, 1028), device='cuda')
    assert remove_pc_multi(nv, big, [None], [0], [big.clone()]) == nv.MMB_E_INVALID       # d > 1024
    assert nv.lib.mmb_remove_pc_multi(nv.ptr(X), 64, 300, 0, (C.c_void_p * 1)(), (C.c_int * 1)(),
                                      (C.c_void_p * 1)(), nv.stream_ptr()) == nv.MMB_E_INVALID   # P = 0
    assert nv.lib.mmb_remove_pc_multi(None, 64, 300, 1, (C.c_void_p * 1)(pc.data_ptr()), (C.c_int * 1)(1),
                                      (C.c_void_p * 1)(o1.data_ptr()), nv.stream_ptr()) == nv.MMB_E_INVALID
    with pytest.raises(ValueError):
        nv.check(remove_pc_multi(nv, X, [pc, pc], [2, 1], [o1, X]))
    assert nv.lib.mmb_comm_slot_bytes() == 4 * 1024 * 1024


def sweep_case(n, L, V, d, K, seed):
    import torch
    rng = np.random.default_rng(seed)
    We = cases.table(V, d, seed=seed)
    ids, p = cases.zipf_ids(rng, n, L, V)
    W = np.stack([cases.sif_weights(p, a) for a in np.geomspace(1e-4, 3e-2, K)]).astype(np.float32)
    return (torch.as_tensor(We, device='cuda'), torch.as_tensor(W, device='cuda'),
            torch.as_tensor(ids, device='cuda'))


@pytest.mark.parametrize('n,npcs', [(3000, (0, 1, 3)), (5000, (2,)), (157, (0, 1, 3)), (157, (1,)), (800, (0,)),
                                    (0, (0, 1))])
def test_sharded_sweep_without_group_equals_single_gpu_sweep(mods, n, npcs):
    """No process group: the exchange is the identity and n_global = n, so every stage is the single-GPU
    sweep's (N < d through the summed start block, N >= 4096 through the tcgen05 Gram), padded and ragged."""
    nv, sf, sd = mods
    table, W, ids = sweep_case(n, 40, 2000, 300, 3, seed=n + len(npcs))
    marks = []
    for x in (ids, sf.to_ragged(ids)):
        want = sf.sif_embedding_sweep(table, W, x, npcs=npcs)
        got, pcs, st = sd.sharded_sif_embedding_sweep(table, W, x, n, 0, npcs=npcs, timers=marks.append)
        nv.raise_on_status(st, table.shape[0])
        assert same_bits(got, want), (n, npcs)
        assert len(pcs) == 3 and all(len(row) == len(npcs) for row in pcs)
        for row in pcs:
            for p, pc in zip(npcs, row):
                assert pc is None if (p == 0 or n == 0) else tuple(pc.shape) == (p, 300)
    if n == 0:      # nothing to sum, solve or project: the call ends after the embed
        assert marks == ['embed', 'embed']
    elif any(npcs):
        assert marks[:5] == ['embed', 'gram', 'allreduce', 'pc', 'project']
    else:           # npc = 0 only: no Gram and no exchange
        assert marks == ['embed', 'pc', 'project'] * 2


def test_sharded_sweep_components_match_single_vector_solve(mods):
    """pcs[k][j] is the component sharded_sif_embedding solves for vocab_w[k] and npcs[j]."""
    nv, sf, sd = mods
    table, W, ids = sweep_case(600, 30, 3000, 300, 2, seed=11)    # N L < 8 V: both embeds on the general kernel
    out, pcs, st = sd.sharded_sif_embedding_sweep(table, W, ids, 600, 0, npcs=(1, 4))
    for k in range(2):
        for j, p in enumerate((1, 4)):
            emb, pc, _ = sd.sharded_sif_embedding(table, W[k].contiguous(), ids, 600, 0, npc=p)
            assert same_bits(pcs[k][j], pc) and same_bits(out[k, j], emb), (k, p)


def test_sharded_sweep_bad_id_is_a_status_bit(mods):
    nv, sf, sd = mods
    table, W, ids = sweep_case(300, 20, 1000, 300, 2, seed=12)
    ids[7, 3] = 1000
    out, pcs, st = sd.sharded_sif_embedding_sweep(table, W, ids, 300, 0, npcs=(0, 1))
    with pytest.raises(IndexError):
        nv.raise_on_status(st, 1000)
    with pytest.raises(ValueError):
        sd.sharded_sif_embedding_sweep(table, W, ids, 300, 0, npcs=(23,))
    with pytest.raises(ValueError):
        sd.sharded_sif_embedding_sweep(table, W[:, :999].contiguous(), ids, 300, 0, npcs=(1,))
