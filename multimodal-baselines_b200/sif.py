"""Drop-in for the reference's ``sif.py`` (SURVEY.md §2 #2, §8 row A5): word weights and
``get_sentence_embeddings``, the call ``simplesif.main`` makes per split (reference
simplesif.py:296-311).  The embedding itself runs through ``mmb_sif_embedding_host`` /
``mmb_sif_embedding`` of libmmb_b200.so.  ``get_sentence_embeddings_sweep`` (no reference counterpart) does the
same for K word-weight vectors and several numbers of removed components in one gather
(``mmb_sif_embedding_sweep_host`` for NumPy ids; ``mmb_sif_embed_multi`` / ``mmb_sif_embed_multi_ragged`` for ids
on the device).  ``fit_sentence_components`` and ``transform_sentence_embeddings`` split the same call into
TruncatedSVD's fit and transform: components fitted on one set of utterances (``mmb_sif_fit_host``), then removed
from the embeddings of any other (``mmb_sif_transform_host`` / ``mmb_sif_transform``, one fused pass).
"""
import ctypes as C
import os

import numpy as np
import torch

import _native as nv
from _native import lib
from sif_functions import Params, seq2weight, SIF_embedding, start_block, sif_embedding_device  # noqa: F401
from sif_functions import sif_transform_device  # noqa: F401
from sif_functions import sif_embedding_sweep, sweep_npcs  # noqa: F401
from sif_functions import RaggedIds, sif_embedding_ragged, to_ragged  # noqa: F401

# ---- word weights a / (a + p(w)) (host-side file handling; the arithmetic that matters runs in the kernels) ----

def get_word_weights(word_freq_file, a=1e-3):
    """reference sif.py:14-32.  ``{word: a / (a + count / total)}`` from a text file of ``word count``
    pairs; lines that do not have exactly two fields are echoed and skipped, blank lines ignored."""
    counts = {}
    with open(word_freq_file, 'r') as fh:
        for raw in fh:
            fields = raw.split()
            if not fields:
                continue
            if len(fields) != 2:
                print(fields)
                continue
            counts[fields[0]] = float(fields[1])
    total = float(sum(counts.values()))
    return {word: a / (a + c / total) for word, c in counts.items()}


_WEIGHT_FILES = {'pom': 'pom/pom_word_weights.npy', 'iemocap': 'iemocap/iemocap_word_weights.npy'}


def _load_weight_vector(path):
    vec = np.load(path).squeeze()
    print(vec.shape)
    return vec


def load_pom_weights():
    """reference sif.py:44-47 -- the per-vocabulary weight vector shipped with the POM ids."""
    return _load_weight_vector(_WEIGHT_FILES['pom'])


def load_iemocap_weights():
    """reference sif.py:49-52."""
    return _load_weight_vector(_WEIGHT_FILES['iemocap'])


def load_mosi_weights(word2ix=None):
    """reference sif.py:54-76 -- the cached ``word_weights.npy`` if present, else built from the enwiki
    counts: index i gets the weight of its (lower-cased) word, 1.0 when the word has no count.  The
    reference's rebuild branch reads a global ``word2ix`` that is never defined (line 63: NameError);
    here the mapping is an optional argument and its absence raises the same NameError."""
    cache = 'word_weights.npy'
    if os.path.isfile(cache):
        return np.load(cache, allow_pickle=False).squeeze()
    if word2ix is None:
        raise NameError("name 'word2ix' is not defined")
    by_word = get_word_weights('SIF/auxiliary_data/enwiki_vocab_min200.txt')
    weights = np.zeros(max(word2ix.values()) + 1)
    missing = 0
    for word, ix in word2ix.items():
        w = by_word.get(word.lower())
        if w is None:
            w, missing = 1., missing + 1
        weights[ix] = w
    print("# of words with unknown weight", missing)
    print(weights[:5])
    np.save(cache, weights, allow_pickle=False)
    return weights


def load_weights(args):
    """reference sif.py:34-42 -- the weight vector of ``args['dataset']``; unknown names raise
    NotImplementedError like the reference's final ``else``."""
    loaders = {'mosi': load_mosi_weights, 'pom': load_pom_weights, 'iemocap': load_iemocap_weights}
    if args['dataset'] not in loaders:
        raise NotImplementedError
    return loaders[args['dataset']]()


def get_sentence_word_weights(text, weights):
    """reference sif.py:78-82 -- weights for each word in each sentence (mask of ones)."""
    return seq2weight(text, np.ones(np.shape(text)), weights)


def _prepare(word_embeddings, weights, text, dev):
    """``(table_t, w_t, ids)`` for the single-vector calls: the table and the weight vector as float32 CUDA tensors,
    and the ids as they came, a C-contiguous int64 NumPy array or a contiguous CUDA tensor, either (N, L).  A weight
    vector shorter than the table is padded with zeros; an id beyond it raises ``IndexError``, as NumPy's
    ``weights[ids]`` would."""
    if isinstance(text, torch.Tensor) and text.is_cuda:
        ids = text.contiguous()
    else:
        ids = np.ascontiguousarray(np.asarray(text), dtype=np.int64)
    if ids.ndim != 2:
        raise ValueError('text must be (n_samples, seq_len)')
    table_t = nv.to_device(word_embeddings, torch.float32, dev)
    w_t = nv.to_device(weights if isinstance(weights, torch.Tensor) else np.asarray(weights).reshape(-1),
                       torch.float32, dev).reshape(-1)
    V = table_t.shape[0]
    if w_t.numel() < V:
        id_max = int(ids.max()) if ids.shape[0] * ids.shape[1] else None     # only here: a pass over the ids
        if id_max is not None and id_max >= w_t.numel():
            raise IndexError('index %d is out of bounds for axis 0 with size %d' % (id_max, w_t.numel()))
        w_t = torch.cat([w_t, w_t.new_zeros(V - w_t.numel())])
    return table_t, w_t, ids


def get_sentence_embeddings(word_embeddings, weights, text, out=None):
    """reference sif.py:84-94 -- SIF embedding of every utterance with the first principal
    component removed (``RMPC = 1``, line 88).

    NumPy in -> float64 NumPy out, as the reference; CUDA tensors in -> float32 CUDA tensor
    out (device-resident fused path).  ``out`` may be a preallocated (N, d) float64/float32
    host array (e.g. ``_native.PinnedArray(...).array``) to receive the result.
    """
    RMPC = 1
    dev = nv.require_cuda()
    if isinstance(text, RaggedIds):
        # SURVEY.md 8f N3: CSR ids on the device -- the padded matrix's result without its padding
        table_t = nv.to_device(word_embeddings, torch.float32, dev)
        w_t = nv.to_device(weights, torch.float32, dev).reshape(-1)
        return sif_embedding_ragged(table_t, w_t, text, npc=RMPC)
    if isinstance(text, torch.Tensor) and text.is_cuda:
        table_t = nv.to_device(word_embeddings, torch.float32, dev)
        w_t = nv.to_device(weights, torch.float32, dev).reshape(-1)
        return sif_embedding_device(table_t, w_t, text.contiguous(), npc=RMPC)

    table_t, w_t, ids = _prepare(word_embeddings, weights, text, dev)
    n, L = ids.shape
    V, d = table_t.shape
    if out is None:
        out = np.empty((n, d), dtype=np.float64)
    assert out.shape == (n, d) and out.flags['C_CONTIGUOUS'] and out.dtype in (np.float64, np.float32)
    omega = np.ascontiguousarray(start_block(d if n >= d else n, RMPC))
    torch.cuda.current_stream().synchronize()      # table / weights uploads are done
    nv.check(lib.mmb_sif_embedding_host(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.np_ptr(ids), n, L, RMPC,
                                        nv.np_ptr(omega), nv.np_ptr(out), int(out.dtype == np.float64),
                                        None, nv.GRAM_AUTO, 0))
    return out


def get_sentence_embeddings_sweep(word_embeddings, weights, text, npcs=(1,), out=None):
    """``get_sentence_embeddings`` for K word-weight vectors at once (e.g. ``get_word_weights(file, a)`` for
    several ``a``) and P numbers of removed principal components: ``out[k, j]`` is the SIF embedding with
    ``weights[k]`` and ``npcs[j]`` components removed (0 = the raw weighted average).  The table rows are
    gathered once for all K vectors.

    ``weights`` is a (K, V) array or a sequence of K vectors; a vector shorter than the table is padded with
    zeros, and an id beyond it raises ``IndexError``, as in ``get_sentence_embeddings``.  CUDA tensors or
    ``RaggedIds`` in -> float32 CUDA tensor out (``sif_functions.sif_embedding_sweep``).  NumPy in -> float64
    (K, P, N, d) NumPy out through ``mmb_sif_embedding_sweep_host``: the ids stream to the device in chunks, only
    the K embeddings stay resident there, and each projected chunk is written straight into the host result,
    bit for bit the device sweep's values.  ``out`` may be a preallocated C-contiguous (K, P, N, d) float64 or
    float32 host array (e.g. ``_native.PinnedArray(...).array``, for full PCIe rate) to receive the result; it is
    returned.  For ``RaggedIds`` the ids are those of the padded matrix they stand for: the tokens, and
    ``pad_id`` when an utterance is shorter than ``L_pad``."""
    dev = nv.require_cuda()
    ragged = isinstance(text, RaggedIds)
    as_np = not (ragged or (isinstance(text, torch.Tensor) and text.is_cuda))
    if out is not None and not as_np:
        raise ValueError('out= takes host ids; with CUDA ids or RaggedIds the result is a CUDA tensor')
    table_t = nv.to_device(word_embeddings, torch.float32, dev)
    V, d = table_t.shape
    if isinstance(weights, torch.Tensor):
        vecs = [weights.reshape(-1)] if weights.dim() == 1 else list(weights)
    elif isinstance(weights, np.ndarray) and weights.ndim == 2:
        vecs = list(weights)
    else:
        vecs = [weights] if np.ndim(weights[0]) == 0 else list(weights)
    if as_np:
        ids = np.ascontiguousarray(np.asarray(text), dtype=np.int64)
        if ids.ndim != 2:
            raise ValueError('text must be (n_samples, seq_len)')
        id_max = int(ids.max()) if ids.size else None
    elif ragged:
        ids_t = text
        n, L = text.shape
        id_max = int(text.tokens.max().item()) if text.tokens.numel() else None
        if n and bool((text.lengths() < L).any()):
            id_max = text.pad_id if id_max is None else max(id_max, text.pad_id)
    else:
        ids_t = text.contiguous()
        id_max = int(ids_t.max().item()) if ids_t.numel() else None
    rows = []
    for vec in vecs:
        w_t = nv.to_device(vec if isinstance(vec, torch.Tensor) else np.asarray(vec).reshape(-1),
                           torch.float32, dev).reshape(-1)
        if w_t.numel() < V:
            if id_max is not None and id_max >= w_t.numel():
                raise IndexError('index %d is out of bounds for axis 0 with size %d' % (id_max, w_t.numel()))
            w_t = torch.cat([w_t, w_t.new_zeros(V - w_t.numel())])
        rows.append(w_t[:V])
    W_t = torch.stack(rows).contiguous()
    if not as_np:
        return sif_embedding_sweep(table_t, W_t, ids_t, npcs=npcs)
    npcs = sweep_npcs(npcs)
    K, P = W_t.shape[0], len(npcs)
    n, L = ids.shape
    if out is None:
        out = np.empty((K, P, n, d), dtype=np.float64)
    if (tuple(out.shape) != (K, P, n, d) or not out.flags['C_CONTIGUOUS']
            or out.dtype not in (np.float64, np.float32)):
        raise ValueError('out must be a C-contiguous (%d, %d, %d, %d) float64 or float32 array' % (K, P, n, d))
    omegas = [np.ascontiguousarray(start_block(d if n >= d else n, p)) if p else None for p in npcs]
    omega_arr = (C.c_void_p * P)(*[o.ctypes.data if o is not None else None for o in omegas])
    torch.cuda.current_stream().synchronize()      # table / weights uploads are done
    nv.check(lib.mmb_sif_embedding_sweep_host(nv.ptr(table_t), V, d, nv.ptr(W_t), K, nv.np_ptr(ids), n, L, P,
                                              (C.c_int * P)(*npcs), omega_arr, nv.np_ptr(out),
                                              int(out.dtype == np.float64), nv.GRAM_AUTO, 0))
    return out


def fit_sentence_components(word_embeddings, weights, text, npc=1):
    """The first half of ``get_sentence_embeddings`` as an estimator's fit: the ``npc`` principal components
    (reference sif_functions.py:58-67, ``TruncatedSVD.fit``) of the SIF embeddings of ``text``, for
    ``transform_sentence_embeddings`` to remove from these or any other utterances' embeddings.

    NumPy ids -> float64 (npc, d) NumPy array, like ``compute_pc`` (``mmb_sif_fit_host``: the ids stream to the
    device in chunks and only the Gram stays there, so N is not bounded by device memory); CUDA ids -> the float32
    (npc, d) CUDA tensor ``mmb_sif_embedding`` computes.  npc in 1..22."""
    dev = nv.require_cuda()
    if isinstance(text, RaggedIds):
        raise ValueError('fit_sentence_components takes padded (N, L) ids, not RaggedIds')
    npc = int(npc)
    if npc < 1 or npc + 10 > 32:
        raise ValueError('npc must be in 1..22')
    table_t, w_t, ids = _prepare(word_embeddings, weights, text, dev)
    n, L = ids.shape
    V, d = table_t.shape
    if n == 0:
        raise ValueError('fitting components needs at least one utterance')
    if isinstance(ids, torch.Tensor):
        return sif_embedding_device(table_t, w_t, ids, npc=npc, return_pc=True)[1]
    omega = np.ascontiguousarray(start_block(d if n >= d else n, npc))
    pc = np.empty((npc, d), dtype=np.float32)
    torch.cuda.current_stream().synchronize()      # table / weights uploads are done
    nv.check(lib.mmb_sif_fit_host(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.np_ptr(ids), n, L, npc, nv.np_ptr(omega),
                                  nv.np_ptr(pc), nv.GRAM_AUTO, 0))
    return pc.astype(np.float64)


def transform_sentence_embeddings(word_embeddings, weights, text, components, out=None):
    """The second half of ``get_sentence_embeddings`` as an estimator's transform: the SIF embedding of every
    utterance of ``text`` minus its projection on ``components`` (reference sif_functions.py:69-81 with the
    components given), embedded and projected in one pass.  ``components`` is a float32 or float64 (npc, d) array
    or tensor, npc in 0..32 (0: the plain weighted average), rounded to float32 -- exact for what
    ``fit_sentence_components`` returns, so ``transform_sentence_embeddings(We, w, X,
    fit_sentence_components(We, w, X))`` is ``get_sentence_embeddings(We, w, X)`` bit for bit.

    NumPy ids -> float64 (N, d) NumPy out (``mmb_sif_transform_host``: ids in, embedding and D2H overlap chunk by
    chunk, and nothing of size N is kept on the device).  ``out`` may be a preallocated C-contiguous (N, d) float64
    or float32 host array (e.g. ``_native.PinnedArray(...).array``, for full PCIe rate); it is filled and returned.
    CUDA ids -> float32 (N, d) CUDA tensor (``sif_functions.sif_transform_device``)."""
    dev = nv.require_cuda()
    if isinstance(text, RaggedIds):
        raise ValueError('transform_sentence_embeddings takes padded (N, L) ids, not RaggedIds')
    table_t, w_t, ids = _prepare(word_embeddings, weights, text, dev)
    n, L = ids.shape
    V, d = table_t.shape
    pc_t = nv.to_device(components, torch.float32, dev)
    if pc_t.dim() != 2 or pc_t.shape[1] != d or pc_t.shape[0] > 32:
        raise ValueError('components must be (npc, %d) with npc in 0..32, got %s' % (d, tuple(pc_t.shape)))
    if isinstance(ids, torch.Tensor):
        if out is not None:
            raise ValueError('out= takes host ids; with CUDA ids the result is a CUDA tensor')
        return sif_transform_device(table_t, w_t, ids, pc_t)
    if out is None:
        out = np.empty((n, d), dtype=np.float64)
    if tuple(out.shape) != (n, d) or not out.flags['C_CONTIGUOUS'] or out.dtype not in (np.float64, np.float32):
        raise ValueError('out must be a C-contiguous (%d, %d) float64 or float32 array' % (n, d))
    pc = pc_t.cpu().numpy()
    torch.cuda.current_stream().synchronize()      # table / weights uploads are done
    nv.check(lib.mmb_sif_transform_host(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.np_ptr(ids), n, L, nv.np_ptr(pc),
                                        pc.shape[0], nv.np_ptr(out), int(out.dtype == np.float64), 0))
    return out
