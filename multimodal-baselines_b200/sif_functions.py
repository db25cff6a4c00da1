"""Drop-in for the reference's ``sif_functions.py`` on B200 (SURVEY.md §8 rows A1-A5).

Same names, argument order, dtypes and error behaviour as the reference module
(``from sif_functions import Params, seq2weight, SIF_embedding`` -- reference sif.py:6);
the arithmetic runs in libmmb_b200.so (hand-written sm_100a CUDA behind the C ABI of
include/mmb_b200.h).  NumPy in -> NumPy out, like the reference; every function also takes
CUDA torch tensors and then returns a CUDA tensor without touching the host.

``sif_embedding_sweep`` (no reference counterpart) embeds with K word-weight vectors over one gather and
removes several numbers of principal components: a sweep over SIF's ``a`` and ``npc``.

There is no CPU fallback: without the built library or without a CUDA device these raise.
"""
import numpy as np
import torch

import _native as nv
from _native import lib

__all__ = ['seq2weight', 'Params', 'get_weighted_average', 'compute_pc', 'remove_pc',
           'SIF_embedding', 'start_block', 'gram', 'pc_from_gram', 'project_out',
           'sif_embedding_device', 'sif_embedding_sweep', 'RaggedIds', 'to_ragged', 'sif_embedding_ragged']


def _is_np(*xs):
    return not any(isinstance(x, torch.Tensor) for x in xs)


def _status(dev):
    return torch.zeros(1, dtype=torch.int32, device=dev)


# --------------------------------------------------------------------------- A1
def seq2weight(seq, mask, weight4ind):
    """reference sif_functions.py:8-15 -- ``w[i,j] = weight4ind[seq[i,j]]`` where
    ``mask[i,j] > 0 and seq[i,j] >= 0`` else 0; float32 (N, L).  ``IndexError`` for ids
    ``>= len(weight4ind)`` like NumPy."""
    dev = nv.require_cuda()
    as_np = _is_np(seq, mask, weight4ind)
    seq_t = nv.to_device(seq, torch.int64, dev)
    if seq_t.dim() != 2:
        raise ValueError('seq must be 2-D (n_samples, seq_len)')
    n, L = seq_t.shape
    w4i = nv.to_device(weight4ind, torch.float32, dev).reshape(-1)
    mask_t = None
    if mask is not None:
        m = np.asarray(mask) if not isinstance(mask, torch.Tensor) else mask
        if not (as_np and m.size and bool((m > 0).all())):      # all-ones mask: NULL (sif.py:82)
            mask_t = nv.to_device((m > 0), torch.float32, dev)   # only the sign test matters (line 12)
            if tuple(mask_t.shape) != (n, L):
                raise IndexError('mask shape %s does not match seq shape %s' % (tuple(mask_t.shape), (n, L)))
    out = torch.empty((n, L), dtype=torch.float32, device=dev)
    st = _status(dev)
    nv.check(lib.mmb_seq2weight(nv.ptr(seq_t), nv.ptr(mask_t), nv.ptr(w4i), w4i.numel(), n, L,
                                nv.ptr(out), nv.ptr(st), nv.stream_ptr()))
    nv.raise_on_status(st, w4i.numel())
    return out.cpu().numpy() if as_np else out


class Params(object):
    """reference sif_functions.py:17-26."""

    def __init__(self):
        self.LW = 1e-5
        self.LC = 1e-5
        self.eta = 0.05

    def __str__(self):
        t = "LW", self.LW, ", LC", self.LC, ", eta", self.eta
        t = map(str, t)
        return ' '.join(t)


# --------------------------------------------------------------------------- A2
def _weighted_average_device(We_t, x_t, w_t):
    n, L = x_t.shape
    V, d = We_t.shape
    emb = torch.empty((n, d), dtype=torch.float32, device=We_t.device)
    st = _status(We_t.device)
    nv.check(lib.mmb_weighted_average(nv.ptr(We_t), V, d, nv.ptr(x_t), nv.ptr(w_t), n, L,
                                      nv.ptr(emb), nv.ptr(st), nv.stream_ptr()))
    nv.raise_on_status(st, V)
    return emb


def get_weighted_average(We, x, w):
    """reference sif_functions.py:28-56 -- ``emb[i] = w[i,:].dot(We[x[i,:],:]) /
    count_nonzero(w[i,:])``.  Returns float64 (n_samples, d) like the reference's
    ``np.zeros`` (line 37); the sum itself is FP32 in token order (the reference's own
    accumulation type when ``w`` and ``We`` are float32)."""
    dev = nv.require_cuda()
    as_np = _is_np(We, x, w)
    We_t = nv.to_device(We, torch.float32, dev)
    x_t = nv.to_device(x, torch.int64, dev)
    w_t = nv.to_device(w, torch.float32, dev)
    if x_t.dim() != 2 or tuple(w_t.shape) != tuple(x_t.shape):
        raise ValueError('x and w must both be (n_samples, seq_len)')
    emb = _weighted_average_device(We_t, x_t, w_t)
    return emb.double().cpu().numpy() if as_np else emb


# --------------------------------------------------------------------------- A3
def start_block(n_rows, npc, seed=0):
    """The seeded Gaussian start block of sklearn's randomized range finder that
    ``TruncatedSVD(n_iter=7, random_state=0)`` (reference sif_functions.py:65) draws:
    ``RandomState(0).normal(size=(n_rows, npc + 10))``; ``n_rows`` = d when N >= d, else N."""
    return np.random.RandomState(seed).normal(size=(int(n_rows), int(npc) + 10))


_START_BLOCK_CACHE = {}


def start_block_device(n_rows, npc, device):
    """``start_block`` as a float64 CUDA tensor, cached per (rows, npc, device): it is a constant
    of the algorithm (sklearn's ``random_state=0``), so it is generated and uploaded once."""
    key = (int(n_rows), int(npc), str(device))
    t = _START_BLOCK_CACHE.get(key)
    if t is None:
        if len(_START_BLOCK_CACHE) > 64:
            _START_BLOCK_CACHE.clear()
        t = torch.as_tensor(start_block(n_rows, npc)).to(device)
        _START_BLOCK_CACHE[key] = t
    return t


def gram(X_t, mode=nv.GRAM_AUTO, return_ws=False):
    """``G = X^T X`` (d, d) float32 on the device (first half of compute_pc)."""
    n, d = X_t.shape
    G = torch.empty((d, d), dtype=torch.float32, device=X_t.device)
    nbytes = lib.mmb_gram_workspace_bytes(n, d, mode)
    ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=X_t.device)
    nv.check(lib.mmb_gram(nv.ptr(X_t), n, d, nv.ptr(G), nv.ptr(ws), nbytes, mode, nv.stream_ptr()))
    return (G, ws) if return_ws else G


def pc_from_gram(G_t, npc, n_rows, X_t=None, S0_t=None, n_iter=7):
    """Components (npc, d) float32 from the Gram and the seeded start block (second half of
    compute_pc).  ``n_rows`` is the GLOBAL number of rows N of X (decides sklearn's
    transpose rule N < d).  For N < d the start block is ``X^T Omega``: pass ``X_t`` (single
    device) or a ready ``S0_t`` (multi-GPU: summed over ranks by the caller)."""
    d = G_t.shape[0]
    k = npc + 10
    dev = G_t.device
    transposed = n_rows < d
    if S0_t is None:
        if transposed:
            omega = start_block_device(n_rows, npc, dev)
            S0_t = torch.empty((d, k), dtype=torch.float64, device=dev)
            nv.check(lib.mmb_start_block_xt(nv.ptr(X_t), n_rows, d, nv.ptr(omega), k, nv.ptr(S0_t),
                                            nv.stream_ptr()))
        else:
            S0_t = start_block_device(d, npc, dev)
    pc = torch.empty((npc, d), dtype=torch.float32, device=dev)
    nbytes = lib.mmb_pc_workspace_bytes(d, k)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    nv.check(lib.mmb_pc_from_gram(nv.ptr(G_t), d, nv.ptr(S0_t.contiguous()), k, npc, int(transposed), n_iter,
                                  nv.ptr(pc), nv.ptr(ws), nbytes, nv.stream_ptr()))
    return pc


def _compute_pc_device(X_t, npc, mode=nv.GRAM_AUTO):
    n, d = X_t.shape
    if npc + 10 > 32:
        raise ValueError('npc must be <= 22')
    return pc_from_gram(gram(X_t, mode), npc, n, X_t=X_t)


def compute_pc(X, npc=1):
    """reference sif_functions.py:58-67 -- the ``components_`` of scikit-learn's
    ``TruncatedSVD(n_components=npc, n_iter=7, random_state=0).fit(X)`` (no centring),
    computed from the d x d Gram on the device; float64 (npc, d).

    Precision note: the reference keeps X in float64 end to end (sif_functions.py:58-81 receive the
    float64 array of line 37); here X is rounded to float32 on upload, the Gram is accumulated in
    FP32 / 3xTF32 and only the d x (npc+10) solve runs in FP64.  The result is returned as float64 for
    type parity, but carries float32 input rounding (cos > 0.9999 against sklearn's float64 output is
    what the parity tests assert, north_star's tolerance)."""
    dev = nv.require_cuda()
    as_np = _is_np(X)
    X_t = nv.to_device(X, torch.float32, dev)
    pc = _compute_pc_device(X_t, npc)
    return pc.double().cpu().numpy() if as_np else pc


# --------------------------------------------------------------------------- A4
def project_out(X_t, pc_t, out=None):
    """``X - (X pc^T) pc`` on the device (reference sif_functions.py:78/80)."""
    n, d = X_t.shape
    out = torch.empty_like(X_t) if out is None else out
    nv.check(lib.mmb_remove_pc(nv.ptr(X_t), n, d, nv.ptr(pc_t), pc_t.shape[0], nv.ptr(out), nv.stream_ptr()))
    return out


def remove_pc(X, npc=1):
    """reference sif_functions.py:69-81.  Like compute_pc, X is rounded to float32 on upload and the
    projection is evaluated in FP32 (the reference works in float64); returned as float64."""
    dev = nv.require_cuda()
    as_np = _is_np(X)
    X_t = nv.to_device(X, torch.float32, dev)
    pc = _compute_pc_device(X_t, npc)
    XX = project_out(X_t, pc)
    return XX.double().cpu().numpy() if as_np else XX


# --------------------------------------------------------------------------- A5
def SIF_embedding(We, x, w, params):
    """reference sif_functions.py:84-96 -- weighted average, then PC removal iff
    ``params.rmpc > 0``."""
    dev = nv.require_cuda()
    as_np = _is_np(We, x, w)
    We_t = nv.to_device(We, torch.float32, dev)
    x_t = nv.to_device(x, torch.int64, dev)
    w_t = nv.to_device(w, torch.float32, dev)
    emb = _weighted_average_device(We_t, x_t, w_t)
    if params.rmpc > 0:
        pc = _compute_pc_device(emb, params.rmpc)
        project_out(emb, pc, out=emb)
    return emb.double().cpu().numpy() if as_np else emb


def sif_embedding_device(table_t, vocab_w_t, ids_t, npc=1, gram_mode=nv.GRAM_AUTO, omega_t=None,
                         return_pc=False, check=True):
    """The fused device-resident path (seq2weight folded into the gather; embed -> Gram ->
    components -> projection with no host round trip): ``mmb_sif_embedding``.
    All arguments are CUDA tensors: table (V, d) f32, vocab_w (V,) f32, ids (N, L) int64."""
    n, L = ids_t.shape
    V, d = table_t.shape
    dev = table_t.device
    emb = torch.empty((n, d), dtype=torch.float32, device=dev)
    st = _status(dev)
    pc = torch.empty((max(npc, 1), d), dtype=torch.float32, device=dev)
    if npc > 0 and omega_t is None:
        omega_t = start_block_device(d if n >= d else n, npc, dev)
    nbytes = lib.mmb_sif_workspace_bytes(n, d, npc)
    extra = lib.mmb_sif_embed_workspace_bytes(V, d, n, L)     # large batches: scratch for the pre-scaled table
    if extra:
        nbytes = (nbytes + 255) // 256 * 256 + extra
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    nv.check(lib.mmb_sif_embedding(nv.ptr(table_t), V, d, nv.ptr(vocab_w_t), nv.ptr(ids_t), n, L, npc,
                                   nv.ptr(omega_t), nv.ptr(emb), nv.ptr(pc), None, nv.ptr(ws), nbytes,
                                   gram_mode, nv.ptr(st), nv.stream_ptr()))
    if check:
        nv.raise_on_status(st, V)
    return (emb, pc) if return_pc else emb


def sif_embedding_sweep(table_t, vocab_w_t, ids_t, npcs=(1,), gram_mode=nv.GRAM_AUTO):
    """SIF embeddings for K word-weight vectors x P principal-component counts (a sweep over the smoothing
    constant ``a`` of ``a / (a + p(w))`` and over ``npc``).  All arguments are CUDA tensors: table (V, d) f32,
    vocab_w (K, V) f32, ids (N, L) int64.  Returns float32 (K, P, N, d), P = ``len(npcs)``.

    One ``mmb_sif_embed_multi`` call gathers every token's row once for all K weight vectors (``emb[k]`` is bit
    for bit ``mmb_sif_embed`` with ``vocab_w[k]``); then per k one Gram, and per (k, npc) one ``pc_from_gram``
    (with that k's own start block when N < d) and one projection.  ``npc = 0`` is the raw weighted average.
    With a single ``npc`` the projection runs in place: peak memory is the (K, N, d) output."""
    npcs = tuple(int(p) for p in npcs)
    if not npcs:
        raise ValueError('npcs must name at least one number of components')
    for p in npcs:
        if p < 0 or p + 10 > 32:
            raise ValueError('npc must be in 0..22')
    if vocab_w_t.dim() != 2 or ids_t.dim() != 2:
        raise ValueError('vocab_w must be (K, V) and ids (n_samples, seq_len)')
    n, L = ids_t.shape
    V, d = table_t.shape
    K = vocab_w_t.shape[0]
    if vocab_w_t.shape[1] != V:
        raise ValueError('vocab_w has %d columns, the table %d rows' % (vocab_w_t.shape[1], V))
    dev = table_t.device
    emb = torch.empty((K, n, d), dtype=torch.float32, device=dev)
    st = _status(dev)
    nbytes = lib.mmb_sif_embed_multi_workspace_bytes(V, K)
    ws = torch.empty(max(nbytes, 32), dtype=torch.uint8, device=dev)
    nv.check(lib.mmb_sif_embed_multi(nv.ptr(table_t), V, d, nv.ptr(vocab_w_t), K, nv.ptr(ids_t), n, L, nv.ptr(emb),
                                     nv.ptr(st), nv.ptr(ws), nbytes, nv.stream_ptr()))
    nv.raise_on_status(st, V)
    del ws
    in_place = len(npcs) == 1
    out = emb.unsqueeze(1) if in_place else torch.empty((K, len(npcs), n, d), dtype=torch.float32, device=dev)
    if n == 0:
        return out
    for k in range(K):
        E = emb[k]
        G = gram(E, gram_mode) if any(npcs) else None
        for j, p in enumerate(npcs):
            if p == 0:
                if not in_place:
                    out[k, j].copy_(E)
                continue
            pc = pc_from_gram(G, p, n, X_t=E)
            project_out(E, pc, out=out[k, j])
    return out


# --------------------------------------------------------------------------- ragged ids (SURVEY.md 8f N3)
class RaggedIds(object):
    """Token ids in CSR form on the device: utterance i is ``tokens[offsets[i]:offsets[i+1]]`` (int64 CUDA
    tensors; ``offsets`` has N + 1 entries), standing for row i of the right-padded ``(N, L_pad)`` id matrix
    the reference builds (utils.py:77-80), i.e. followed by ``L_pad - length_i`` copies of ``pad_id``.  The
    pad tokens stay part of the arithmetic (they are ordinary tokens to sif_functions.py:28-56: summed with
    their weight, counted in the divisor) but are neither stored, moved nor walked."""

    def __init__(self, tokens, offsets, L_pad, pad_id=0):
        self.tokens, self.offsets, self.L_pad, self.pad_id = tokens, offsets, int(L_pad), int(pad_id)

    @property
    def shape(self):
        return (int(self.offsets.numel()) - 1, self.L_pad)

    def lengths(self):
        return self.offsets[1:] - self.offsets[:-1]

    def to_padded(self):
        """The (N, L_pad) matrix back (testing / interop)."""
        n, L = self.shape
        out = torch.full((n, L), self.pad_id, dtype=torch.int64, device=self.tokens.device)
        lens = self.lengths()
        pos = torch.arange(L, device=out.device)[None, :]
        out[pos < lens[:, None]] = self.tokens
        return out


def to_ragged(ids, pad_id=0, device=None):
    """Padded ``(N, L)`` ids (NumPy or tensor) -> ``RaggedIds`` on the device (``mmb_ids_lengths`` +
    ``mmb_ids_compact``): length = 1 + index of the last token that is not ``pad_id``; interior pad ids
    (MOSI's shared OOV row 0) stay tokens."""
    dev = device or nv.require_cuda()
    ids_t = nv.to_device(ids, torch.int64, dev)
    if ids_t.dim() != 2:
        raise ValueError('ids must be (n_samples, seq_len)')
    n, L = ids_t.shape
    lengths = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nv.check(lib.mmb_ids_lengths(nv.ptr(ids_t), n, L, int(pad_id), nv.ptr(lengths), nv.ptr(offsets), nv.stream_ptr()))
    total = int(offsets[-1].item())
    tokens = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
    nv.check(lib.mmb_ids_compact(nv.ptr(ids_t), n, L, nv.ptr(offsets), nv.ptr(tokens), nv.stream_ptr()))
    return RaggedIds(tokens[:total], offsets, L, pad_id)


def sif_embedding_ragged(table_t, vocab_w_t, ragged, npc=1, gram_mode=nv.GRAM_AUTO, return_pc=False, check=True):
    """``sif_embedding_device`` on ``RaggedIds``: ``mmb_sif_embed_ragged`` -> Gram -> components ->
    projection, all on the device.  Equal to the padded call on ``ragged.to_padded()``."""
    n, _ = ragged.shape
    V, d = table_t.shape
    dev = table_t.device
    emb = torch.empty((n, d), dtype=torch.float32, device=dev)
    st = _status(dev)
    nv.check(lib.mmb_sif_embed_ragged(nv.ptr(table_t), V, d, nv.ptr(vocab_w_t), nv.ptr(ragged.tokens),
                                      nv.ptr(ragged.offsets), n, ragged.L_pad, ragged.pad_id, nv.ptr(emb), nv.ptr(st),
                                      nv.stream_ptr()))
    if check:
        nv.raise_on_status(st, V)
    pc = None
    if npc > 0 and n > 0:
        pc = _compute_pc_device(emb, npc, gram_mode)
        project_out(emb, pc, out=emb)
    return (emb, pc) if return_pc else emb
