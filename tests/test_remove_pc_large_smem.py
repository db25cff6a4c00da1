"""mmb_remove_pc with more than 48 KB of components at d <= 512 (npc * d > 12288, e.g. npc = 32 at d = 512): the
kernel needs the dynamic shared-memory opt-in at every row width, not only for d > 512."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('d,npc', [(512, 32), (400, 31), (1024, 32)])
def test_remove_pc_many_components_matches_oracle(d, npc):
    import torch
    import _native as nv
    from oracle import sif_oracle as so
    rng = np.random.default_rng(d + npc)
    X = rng.standard_normal((777, d)).astype(np.float32)
    pc = np.linalg.qr(rng.standard_normal((d, npc)))[0].T.astype(np.float32)
    X_t, pc_t = torch.as_tensor(X, device='cuda'), torch.as_tensor(np.ascontiguousarray(pc), device='cuda')
    out = torch.empty_like(X_t)
    nv.check(nv.lib.mmb_remove_pc(nv.ptr(X_t), X.shape[0], d, nv.ptr(pc_t), npc, nv.ptr(out), nv.stream_ptr()))
    want = so.remove_pc_with(X.astype(np.float64), pc.astype(np.float64))
    got = out.cpu().numpy().astype(np.float64)
    assert float(np.max(np.abs(got - want))) < 1e-4 * float(np.abs(want).max())
