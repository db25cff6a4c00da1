"""Utterance-sharded SIF embedding over the GPUs of one box (SURVEY.md §8e).

The reference has no distributed code; this is the one data-parallel strategy the path
admits.  Utterances are split into contiguous blocks, one per rank (one process per GPU);
the table and the vocabulary weights are replicated.  Per split of the data:

    rank-local:  emb_r = weighted average of its block              (no communication)
                 G_r   = emb_r^T emb_r                               (d x d float32)
    exchange:    G = sum_r G_r            ONE all-reduce of d*d floats (360 KB at d = 300)
                 (N < d only: the start block S0 = X^T Omega is summed the same way)
    replicated:  components from (G, seeded start block) -- same bits on every rank, so no
                 broadcast is needed
    rank-local:  emb_r -= (emb_r pc^T) pc

The exchange has two implementations:
  * ``PeerComm`` (default on one box, world <= 8): libmmb_b200.so's own one-shot all-reduce over
    NVLink peer memory (CUDA IPC buffers), fused into the kernel that finishes the Gram
    (``mmb_gram_allreduce_peer``) -- ranks add in rank order, so every rank holds identical bits;
  * ``torch.distributed.all_reduce`` (NCCL on GPUs, gloo on CPU): the fallback for any other
    topology or backend, the path a caller selects with ``comm=None``, and what
    tests/test_dist_cpu.py exercises for the partition / reduction arithmetic.
"""
import ctypes as C
import os

import numpy as np
import torch
import torch.distributed as dist


def shard_bounds(n_global, world_size, rank):
    """Contiguous block [lo, hi) of rank `rank`; the first n_global % world_size ranks get
    one extra row (same rule as numpy.array_split)."""
    base, rem = divmod(int(n_global), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def allreduce_sum_(t, group=None):
    """In-place sum over ranks (no-op without an initialised process group)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


_NUMA_NOTE = 'not bound (single process)'


def _gpu_numa_node(local_rank):
    """NUMA node of GPU `local_rank` from sysfs (None when the guest hides it: numa_node = -1)."""
    try:
        prop = torch.cuda.get_device_properties(local_rank)
        bdf = '%04x:%02x:%02x.0' % (getattr(prop, 'pci_domain_id', 0), prop.pci_bus_id, prop.pci_device_id)
        with open('/sys/bus/pci/devices/%s/numa_node' % bdf) as fh:
            node = int(fh.read().strip())
        return node if node >= 0 else None
    except Exception:
        return None


def _node_cpus(node):
    with open('/sys/devices/system/node/node%d/cpulist' % node) as fh:
        cpus = set()
        for part in fh.read().strip().split(','):
            if '-' in part:
                a, b = part.split('-')
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
    return cpus


def bind_to_gpu_numa_node(local_rank):
    """One process per GPU: pin this process's threads (and, by first touch, the pinned host buffers it
    allocates afterwards) to the NUMA node its GPU hangs off, so that eight ranks' H2D/D2H streams do not
    all cross one socket's memory controller.  A no-op, recorded in ``numa_note()``, when the box shows a
    single node or hides the GPU's node (virtualised guests report numa_node = -1)."""
    global _NUMA_NOTE
    try:
        n_nodes = len([d for d in os.listdir('/sys/devices/system/node') if d.startswith('node') and d[4:].isdigit()])
    except Exception:
        n_nodes = 0
    node = _gpu_numa_node(local_rank)
    if n_nodes <= 1 or node is None:
        _NUMA_NOTE = 'no placement possible: %d NUMA node(s) visible, GPU %d reports node %s' % (n_nodes, local_rank, node)
        return None
    try:
        allowed = os.sched_getaffinity(0)
        cpus = _node_cpus(node) & allowed
        if not cpus:
            _NUMA_NOTE = 'GPU %d is on node %d but none of its CPUs are in this cpuset' % (local_rank, node)
            return None
        os.sched_setaffinity(0, cpus)
        # MPOL_PREFERRED on the GPU's node for every later allocation of this process (set_mempolicy, x86-64 238)
        try:
            libc = C.CDLL(None, use_errno=True)
            mask = C.c_ulong(1 << node)
            libc.syscall(C.c_long(238), C.c_int(1), C.byref(mask), C.c_ulong(64))
        except Exception:
            pass
        _NUMA_NOTE = 'rank bound to NUMA node %d of GPU %d (%d CPUs, MPOL_PREFERRED)' % (node, local_rank, len(cpus))
        return node
    except Exception as e:
        _NUMA_NOTE = 'binding failed: %s' % e
        return None


def numa_note():
    return _NUMA_NOTE


class PeerComm(object):
    """NVLink exchange buffers of the ranks of one box (one process per GPU).

    Every rank allocates one buffer in libmmb_b200.so, the 64-byte CUDA IPC handles travel
    through ``torch.distributed.all_gather_object`` once, and each rank maps its peers' buffers.
    ``epoch`` advances by one per collective call; all ranks must issue the same sequence."""

    def __init__(self, group=None):
        import _native as nv
        self.nv, self.lib = nv, nv.lib
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        if self.world > 8:
            raise ValueError('PeerComm supports at most 8 ranks (one NVLink box)')
        self.dev = torch.device('cuda', torch.cuda.current_device())
        own = C.c_void_p()
        nv.check(self.lib.mmb_comm_alloc(C.byref(own)))
        self.own = own
        handle = (C.c_char * 64)()
        nv.check(self.lib.mmb_comm_export(own, handle))
        handles = [None] * self.world
        dist.all_gather_object(handles, (os.uname().nodename, bytes(handle.raw)), group=group)
        if len(set(h[0] for h in handles)) != 1:
            raise ValueError('PeerComm needs all ranks on one host')
        self.opened = []
        bufs = []
        for r, (_, raw) in enumerate(handles):
            if r == self.rank:
                bufs.append(own.value)
            else:
                p = C.c_void_p()
                nv.check(self.lib.mmb_comm_open(C.create_string_buffer(raw, 64), C.byref(p)))
                self.opened.append(p)
                bufs.append(p.value)
        self.bufs = (C.c_void_p * self.world)(*bufs)
        self.epoch = 0
        self.status = torch.zeros(1, dtype=torch.int32, device=self.dev)
        dist.barrier(group=group)        # every rank has mapped every buffer before the first use

    def _next(self):
        self.epoch += 1
        return C.c_uint64(self.epoch)

    def allreduce_(self, t):
        """In-place sum over ranks of a float32 / float64 CUDA tensor (<= 4 MiB), rank order, identical bits."""
        nv = self.nv
        assert t.is_cuda and t.is_contiguous() and t.dtype in (torch.float32, torch.float64)
        nv.check(self.lib.mmb_allreduce_peer(nv.ptr(t), t.numel(), int(t.dtype == torch.float64), self.rank,
                                             self.world, self.bufs, self._next(), nv.ptr(self.status),
                                             nv.stream_ptr()))
        return t

    def gram_allreduce(self, emb, mode=0):
        """G = sum over ranks of emb_r^T emb_r: local tcgen05 Gram, then ONE kernel that reduces
        its partials and exchanges them over NVLink."""
        nv = self.nv
        n, d = emb.shape
        G = torch.empty((d, d), dtype=torch.float32, device=emb.device)
        nbytes = self.lib.mmb_gram_workspace_bytes(max(n, 1), d, mode)
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=emb.device)
        nv.check(self.lib.mmb_gram_allreduce_peer(nv.ptr(emb), n, d, nv.ptr(G), nv.ptr(ws), nbytes, mode, self.rank,
                                                  self.world, self.bufs, self._next(), nv.ptr(self.status),
                                                  nv.stream_ptr()))
        return G

    def sif_embedding_host(self, table_t, vocab_w_t, ids_host, out_host, n_global, npc=1, gram_mode=0,
                           chunk_rows=0):
        """This rank's block through the host-buffer pipeline (``mmb_sif_embedding_host_peer``):
        ``ids_host`` (n_local, L) int64 and ``out_host`` (n_local, d) float32/float64 are NumPy
        arrays (pinned for full PCIe rate); H2D, embed and per-chunk Gram overlap, the Gram is summed
        over the ranks through NVLink peer memory, the projection overlaps the D2H.  Synchronous."""
        import sif_functions as sf
        nv = self.nv
        n_local, L = ids_host.shape
        V, d = table_t.shape
        omega = np.ascontiguousarray(sf.start_block(d, npc))
        nv.check(self.lib.mmb_sif_embedding_host_peer(
            nv.ptr(table_t), V, d, nv.ptr(vocab_w_t), nv.np_ptr(ids_host), n_local, L, npc, nv.np_ptr(omega),
            nv.np_ptr(out_host), int(out_host.dtype == np.float64), None, gram_mode, chunk_rows, int(n_global),
            self.rank, self.world, self.bufs, self._next()))
        return out_host

    def check(self):
        """Synchronises; raises if a peer never arrived."""
        if int(self.status.item()) & self.nv.STATUS_COMM_TIMEOUT:
            raise self.nv.MMBError('peer all-reduce timed out: a rank never raised its flag')

    def close(self):
        """Unmap the peers' buffers, then (after a barrier) free this rank's own: CUDA requires that
        every importer has closed its mapping before the exporter frees the allocation."""
        torch.cuda.synchronize()
        for p in self.opened:
            self.lib.mmb_comm_close(p)
        self.opened = []
        if dist.is_initialized():
            dist.barrier(group=self.group)
            torch.cuda.synchronize()
        if self.own is not None:
            self.lib.mmb_comm_free(self.own)
            self.own = None


_DEFAULT_COMM = {}


def default_comm(group=None):
    """The process-wide PeerComm of `group` (created on first use), or None when the exchange
    goes through torch.distributed: no process group, one rank, a non-NCCL backend, more than
    8 ranks or more than one host.  To use torch.distributed on purpose, pass ``comm=None`` to
    the sharded entry points instead of the default ``'auto'``."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) < 2:
        return None
    if dist.get_backend(group) != 'nccl':
        return None
    key = id(group)
    if key not in _DEFAULT_COMM:
        try:
            _DEFAULT_COMM[key] = PeerComm(group)
        except ValueError:
            _DEFAULT_COMM[key] = None
    return _DEFAULT_COMM[key]


def close_default_comms():
    for c in _DEFAULT_COMM.values():
        if c is not None:
            c.close()
    _DEFAULT_COMM.clear()


def local_omega_rows(n_global, lo, n_local, npc, start_block_fn):
    """Rows [lo, lo + n_local) of the global seeded Omega (N_global x (npc+10), float64): the host-side
    partition rule of the N < d case (each rank multiplies ITS rows of X^T with ITS rows of Omega)."""
    return np.ascontiguousarray(start_block_fn(n_global, npc)[lo:lo + n_local])


def local_start_block(emb_local, n_global, lo, npc, start_block_fn):
    """N_global < d: this rank's share of S0 = X^T Omega, using rows [lo, hi) of the global
    seeded Omega (float64, d x (npc+10)); the caller all-reduces it."""
    import _native as nv
    n_local, d = emb_local.shape
    k = npc + 10
    S0 = torch.zeros((d, k), dtype=torch.float64, device=emb_local.device)
    if n_local > 0:
        omega = torch.as_tensor(local_omega_rows(n_global, lo, n_local, npc, start_block_fn)).to(emb_local.device)
        nv.check(nv.lib.mmb_start_block_xt(nv.ptr(emb_local), n_local, d, nv.ptr(omega), k, nv.ptr(S0), nv.stream_ptr()))
    return S0


_EMBED_SCRATCH = {}


def _embed_scratch(nbytes, dev):
    """One scratch buffer per device for the pre-scaled table of mmb_sif_embed_ws (reused across calls: the
    same stream orders its uses)."""
    t = _EMBED_SCRATCH.get(str(dev))
    if t is None or t.numel() < nbytes:
        t = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _EMBED_SCRATCH[str(dev)] = t
    return t


def sharded_sif_embedding(table_t, vocab_w_t, ids_local_t, n_global, lo, npc=1, group=None, gram_mode=0,
                          timers=None, comm='auto'):
    """SIF embedding + PC removal of this rank's block of a split of `n_global` utterances.

    table_t (V, d) f32, vocab_w_t (V,) f32, ids_local_t (n_local, L) int64 -- CUDA tensors on
    this rank's device.  Returns (emb_local (n_local, d) f32, pc (npc, d) f32).
    `timers`, if given, is a callable mark(name) invoked between stages (bench.py records
    CUDA events there)."""
    import _native as nv
    import sif_functions as sf
    from _native import lib

    mark = timers or (lambda name: None)
    n_local, L = ids_local_t.shape
    V, d = table_t.shape
    dev = table_t.device
    emb = torch.empty((n_local, d), dtype=torch.float32, device=dev)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = lib.mmb_sif_embed_workspace_bytes(V, d, n_local, L)   # > 0: large batch, weights folded into a scratch table
    ws = _embed_scratch(ws_bytes, dev) if ws_bytes else None
    nv.check(lib.mmb_sif_embed_ws(nv.ptr(table_t), V, d, nv.ptr(vocab_w_t), nv.ptr(ids_local_t), n_local, L,
                                  nv.ptr(emb), nv.ptr(st), nv.ptr(ws), ws_bytes, nv.stream_ptr()))
    mark('embed')
    if npc <= 0:
        return emb, None, st
    if comm == 'auto':
        comm = default_comm(group)
    S0 = None
    if comm is not None:
        # Gram partial reduction + NVLink exchange in one kernel ('gram' then covers both stages)
        G = comm.gram_allreduce(emb, gram_mode)
        mark('gram')
        if n_global < d:
            S0 = comm.allreduce_(local_start_block(emb, n_global, lo, npc, sf.start_block).contiguous())
    else:
        if n_local > 0:
            G = sf.gram(emb, gram_mode)
        else:
            G = torch.zeros((d, d), dtype=torch.float32, device=dev)
        mark('gram')
        allreduce_sum_(G, group)
        if n_global < d:
            S0 = local_start_block(emb, n_global, lo, npc, sf.start_block)
            allreduce_sum_(S0, group)
    mark('allreduce')
    pc = sf.pc_from_gram(G, npc, n_global, S0_t=S0)
    mark('pc')
    if n_local > 0:
        sf.project_out(emb, pc, out=emb)
    mark('project')
    return emb, pc, st


def exchange_sweep_(G, S0_blocks=(), comm=None, group=None, slot_bytes=None):
    """Sum the sweep's stacked Grams G (K, d, d) float32 and its float64 start blocks over the ranks, in place.
    With a ``PeerComm`` the Grams go in groups of floor(slot / (4 d^2)) (11 at d = 300) and the start blocks
    (flattened back to back) in slot-sized pieces, one ``allreduce_`` per group; otherwise one
    ``torch.distributed`` all-reduce for each of the two stacks.  The group sizes depend only on the shapes,
    so every rank issues the same exchange sequence.  ``slot_bytes`` defaults to ``mmb_comm_slot_bytes()``."""
    S0_blocks = list(S0_blocks)
    flat = torch.cat([b.reshape(-1) for b in S0_blocks]) if S0_blocks else None
    if comm is None:
        allreduce_sum_(G, group)
        if flat is not None:
            allreduce_sum_(flat, group)
    else:
        if slot_bytes is None:
            import _native as nv
            slot_bytes = nv.lib.mmb_comm_slot_bytes()
        K, d, _ = G.shape
        per = slot_bytes // (4 * d * d)
        if per < 1:
            raise ValueError('a %d x %d Gram does not fit the %d-byte exchange slot' % (d, d, slot_bytes))
        for k in range(0, K, per):
            comm.allreduce_(G[k:k + per])
        if flat is not None:
            step = slot_bytes // 8
            for i in range(0, flat.numel(), step):
                comm.allreduce_(flat[i:i + step])
    if flat is not None:
        i = 0
        for b in S0_blocks:
            b.copy_(flat[i:i + b.numel()].view_as(b))
            i += b.numel()
    return G


def sharded_sif_embedding_sweep(table_t, vocab_w_t, ids_local, n_global, lo, npcs=(1,), group=None, gram_mode=0,
                                timers=None, comm='auto'):
    """The SIF sweep (``sif_functions.sif_embedding_sweep``: K word-weight vectors x P component counts) on this
    rank's block of a split of `n_global` utterances.

    table_t (V, d) f32, vocab_w_t (K, V) f32, ids_local (n_local, L) int64 or ``RaggedIds`` of this rank's
    block -- CUDA tensors on this rank's device.  Returns ``(out, pcs, st)``: out (K, P, n_local, d) float32
    (in place over the embeddings when P = 1), ``pcs[k][j]`` the (npcs[j], d) components (None for npc = 0,
    identical bits on every rank) and the status word, which this call does not read: check it afterwards
    (``_native.raise_on_status(st, V)`` raises ``IndexError`` for a bad id), so that a bad id on one rank never
    leaves its peers waiting in the exchange.

    Stages (each followed by ``timers(name)`` when given, as in ``sharded_sif_embedding``): 'embed' (one
    multi-vector gather), 'gram' (K local Grams), 'allreduce' (the stacked Grams, and for n_global < d the K x P
    start blocks, summed over the ranks -- see ``exchange_sweep_``), 'pc' (replicated solves with the global
    N), 'project' (one ``mmb_remove_pc_multi`` per k).  With the peer exchange ``out[k, j]`` is bit for bit
    ``sharded_sif_embedding(table_t, vocab_w_t[k], ids_local, n_global, lo, npc=npcs[j])``'s result on padded
    ids.  Every rank, an empty block included, must make the call with the same K, d and npcs."""
    import sif_functions as sf

    mark = timers or (lambda name: None)
    npcs = sf.sweep_npcs(npcs)
    emb, st = sf.sweep_embed(table_t, vocab_w_t, ids_local)
    mark('embed')
    out = sf.sweep_output(emb, npcs)
    K, n_local, d = emb.shape
    if n_global == 0:
        return out, [[None] * len(npcs) for _ in range(K)], st
    G = S0 = None
    if any(npcs):
        if comm == 'auto':
            comm = default_comm(group)
        G = sf.sweep_grams(emb, gram_mode)
        mark('gram')
        if n_global < d:
            S0 = [[local_start_block(emb[k], n_global, lo, p, sf.start_block) if p else None for p in npcs]
                  for k in range(K)]
        exchange_sweep_(G, [b for row in S0 for b in row if b is not None] if S0 else (), comm, group)
        mark('allreduce')
    pcs = sf.sweep_solve_project(emb, G, npcs, n_global, out, S0=S0, mark=mark)
    return out, pcs, st


def cpu_reference_partition(X_blocks):
    """Host-side statement of the exchange step used by the CPU tests: the sum of per-shard
    Grams equals the Gram of the concatenation."""
    return sum(np.asarray(b, dtype=np.float64).T @ np.asarray(b, dtype=np.float64) for b in X_blocks)
