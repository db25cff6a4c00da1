"""Drop-in for the reference's ``sif.py`` (SURVEY.md §2 #2, §8 row A5): word weights and
``get_sentence_embeddings``, the call ``simplesif.main`` makes per split (reference
simplesif.py:296-311).  The embedding itself runs through ``mmb_sif_embedding_host`` /
``mmb_sif_embedding`` of libmmb_b200.so.  ``get_sentence_embeddings_sweep`` (no reference counterpart) does the
same for K word-weight vectors and several numbers of removed components in one gather (``mmb_sif_embed_multi``).
"""
import ctypes as C
import os

import numpy as np
import torch

import _native as nv
from _native import lib
from sif_functions import Params, seq2weight, SIF_embedding, start_block, sif_embedding_device  # noqa: F401
from sif_functions import sif_embedding_sweep  # noqa: F401
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

    ids = np.ascontiguousarray(np.asarray(text), dtype=np.int64)
    if ids.ndim != 2:
        raise ValueError('text must be (n_samples, seq_len)')
    n, L = ids.shape
    table_t = nv.to_device(word_embeddings, torch.float32, dev)
    w_t = nv.to_device(np.asarray(weights).reshape(-1), torch.float32, dev)
    V, d = table_t.shape
    if w_t.numel() < V:
        if ids.size and ids.max() >= w_t.numel():
            raise IndexError('index %d is out of bounds for axis 0 with size %d' % (ids.max(), w_t.numel()))
        w_t = torch.cat([w_t, w_t.new_zeros(V - w_t.numel())])
    if out is None:
        out = np.empty((n, d), dtype=np.float64)
    assert out.shape == (n, d) and out.flags['C_CONTIGUOUS'] and out.dtype in (np.float64, np.float32)
    omega = np.ascontiguousarray(start_block(d if n >= d else n, RMPC))
    torch.cuda.current_stream().synchronize()      # table / weights uploads are done
    nv.check(lib.mmb_sif_embedding_host(nv.ptr(table_t), V, d, nv.ptr(w_t), nv.np_ptr(ids), n, L, RMPC,
                                        nv.np_ptr(omega), nv.np_ptr(out), int(out.dtype == np.float64),
                                        None, nv.GRAM_AUTO, 0))
    return out


def get_sentence_embeddings_sweep(word_embeddings, weights, text, npcs=(1,)):
    """``get_sentence_embeddings`` for K word-weight vectors at once (e.g. ``get_word_weights(file, a)`` for
    several ``a``) and P numbers of removed principal components: ``out[k, j]`` is the SIF embedding with
    ``weights[k]`` and ``npcs[j]`` components removed (0 = the raw weighted average).  The table rows are
    gathered once for all K vectors (``sif_functions.sif_embedding_sweep``).

    ``weights`` is a (K, V) array or a sequence of K vectors; a vector shorter than the table is padded with
    zeros, and an id beyond it raises ``IndexError``, as in ``get_sentence_embeddings``.  NumPy in -> float64
    (K, P, N, d) NumPy out; CUDA tensors in -> float32 CUDA tensor out.  The ids are uploaded once and the
    result downloaded once."""
    dev = nv.require_cuda()
    as_np = not (isinstance(text, torch.Tensor) and text.is_cuda)
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
        ids_t = nv.to_device(ids, torch.int64, dev)
        id_max = int(ids.max()) if ids.size else None
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
    out = sif_embedding_sweep(table_t, torch.stack(rows).contiguous(), ids_t, npcs=npcs)
    return out.double().cpu().numpy() if as_np else out
