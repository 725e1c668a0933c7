"""Tensor-level wrappers over the C ABI (``include/dcb200.h``) and the ``dcb200::`` torch ops.

Every function takes CUDA tensors, allocates outputs / workspaces with the torch caching
allocator, enqueues on torch's current stream and returns immediately (no host sync except
where a data-dependent output size must be read back: ``knn_graph`` / ``radius_graph``).
PyTorch is plumbing here: device memory and streams.  No eager fallback exists.
"""
import collections
import copy
import ctypes as C
import weakref

import torch

from . import _abi
from ._abi import GEMM_AUTO, GEMM_FP32, GEMM_TF32X3, GEMM_PREFER_TC  # noqa: F401

_i32, _i64, _f32 = torch.int32, torch.int64, torch.float32

# Optional live profiling (bench.py): when set to a list, every spmm / gemm call is bracketed by
# CUDA events on the launching stream and a record with its algorithmic bytes / flops is appended.
PROFILER = None


def _prof_begin():
    if PROFILER is None:
        return None
    e0 = torch.cuda.Event(enable_timing=True)
    e0.record()
    return e0


def _prof_end(e0, **rec):
    if e0 is None:
        return
    e1 = torch.cuda.Event(enable_timing=True)
    e1.record()
    PROFILER.append(dict(e0=e0, e1=e1, **rec))


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise _abi.DcError(f"{name}: expected a CUDA tensor (libdcb200 has no CPU path)")
    if t.dtype != dtype:
        raise _abi.DcError(f"{name}: expected dtype {dtype}, got {t.dtype}")


def _rows(t, name):
    """2-D tensor with unit inner stride -> (tensor, leading dimension)."""
    if t.dim() != 2 or (t.shape[1] > 1 and t.stride(1) != 1):
        raise _abi.DcError(f"{name}: expected a 2-D tensor with contiguous rows")
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def _workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)


# Page-locked staging for host-built tables (dc_gemm_batched): the library fills the buffer and enqueues an asynchronous
# upload, so the buffer must outlive the copy.  Eager: a buffer returns to the free list once an event recorded behind
# the copy has completed.  Under CUDA-graph capture the copy becomes a node that re-reads the buffer on every replay:
# buffers are handed to ``CAPTURE_KEEPALIVE`` (set by step.CapturedTrainStep, which owns them as long as its graph).
_STAGE_FREE = {}
_STAGE_BUSY = collections.deque()
CAPTURE_KEEPALIVE = None


def _capturing():
    return torch.cuda.is_current_stream_capturing()


def _staging_get(nbytes):
    if not _capturing():
        while _STAGE_BUSY and _STAGE_BUSY[0][0].query():
            _, t = _STAGE_BUSY.popleft()
            _STAGE_FREE.setdefault(t.numel(), []).append(t)
    size = max(4096, 1 << (int(nbytes) - 1).bit_length())
    free = _STAGE_FREE.get(size)
    if free:
        return free.pop()
    return torch.empty(size, dtype=torch.uint8, pin_memory=True)


def _staging_put(t):
    if _capturing():
        if CAPTURE_KEEPALIVE is None:
            raise _abi.DcError("stream capture of a host-staged call needs ops.CAPTURE_KEEPALIVE (use step.CapturedTrainStep)")
        CAPTURE_KEEPALIVE.append(t)
    else:
        ev = torch.cuda.Event()
        ev.record()
        _STAGE_BUSY.append((ev, t))


# ----------------------------------------------------------------------------- K5
def csr_build(edge_index, num_nodes, group_by=0, drop_self_loops=False):
    """-> (rowptr int32 [N+1], nbr int32 [E], eid int32 [E]); see dc_csr_build."""
    _need(edge_index, _i64, "edge_index")
    if edge_index.dim() != 2 or edge_index.shape[0] != 2:
        raise _abi.DcError("edge_index must be int64 [2, E]")
    ei = edge_index.contiguous()
    E, dev = ei.shape[1], ei.device
    rowptr = torch.empty(num_nodes + 1, dtype=_i32, device=dev)
    nbr = torch.empty(E, dtype=_i32, device=dev)
    eid = torch.empty(E, dtype=_i32, device=dev)
    nb = _abi.lib().dc_csr_build_workspace_bytes(num_nodes, E)
    ws = _workspace(nb, dev)
    _abi.call("dc_csr_build", _ptr(ei), E, num_nodes, int(group_by), int(bool(drop_self_loops)), _ptr(rowptr), _ptr(nbr),
              _ptr(eid), _ptr(ws), ws.numel(), _stream())
    return rowptr, nbr, eid


def deg_inv_sqrt(rowptr, num_nodes, add_self_loop=False):
    dis = torch.empty(num_nodes, dtype=_f32, device=rowptr.device)
    _abi.call("dc_deg_inv_sqrt", _ptr(rowptr), num_nodes, int(bool(add_self_loop)), _ptr(dis), _stream())
    return dis


import os

TILE_NODES = 2048      # receivers per K1 tile (one graph of the batch where possible)
# K1 variant (all bit-identical): "generic" (warp per receiver, full rows through L2), "tiled"
# (tile x 128-B slice, 4 lanes x 2 float4), "tiled8" (tile x slice, 8 lanes x float4, full-line
# gathers), "tiled_prefetch" (tiled8 + streaming L1 prefetch pass).  B200 r01 (C5, F=256, k=8):
# generic 0.531 / 0.587 ms (fwd / transposed), tiled 0.533 / 0.705, tiled8 0.465 / 0.562,
# tiled_prefetch 0.462 / 0.548  ->  tiled8 is the default where the layout allows.
# B200 r01 late (scripts/k1_lab.py, same config): lean 0.386 / 0.585, blocks (flags 28) 0.391 / 0.495  ->  "auto" =
# lean for the forward structure (uniform kNN degrees, no extra build), edge blocks for the transposed one (ragged
# degrees: the degree-sorted units remove the divergence).
K1_VARIANT = os.environ.get("DCB200_K1", "auto")
# dc_spmm_blocks flags: 1 = persistent grid, 2 = L1 record prefetch, 4 = 768-thread CTAs, 8/16 = L2 prefetch stream
# (24 = the CTA's own tile slice), 32 = one prefetch per sector.  28 = 768 threads, one-shot grid, in-CTA L2 stream.
K1_FLAGS = int(os.environ.get("DCB200_K1_FLAGS", "28"))
# hop chain (K1 v9): 0 = one launch per hop; 1 = chain the forward hops of a layer; 2 = forward and backward chains
K1_CHAIN = int(os.environ.get("DCB200_K1_CHAIN", "2"))
# K1 v10: hop chains with the tile slice staged in shared memory by TMA (dc_spmm_stage) where the tile fits; 0 = v9 chain.
# Measured r02 (C5, F=256, 2000-node graphs): 0.519 ms per forward hop against 0.348 for the L1 chain (the load and gather phases
# of the one resident CTA do not overlap, and a 227 KB carve-out leaves ~28 KB of L1 for the edge records) -> off by default.
K1_STAGE = int(os.environ.get("DCB200_K1_STAGE", "0"))
# K1 v11: hop chains as per-group edge streams with a rolling gather window (dc_spmm_stream; no self loops, F % 32 == 0).
K1_STREAM = int(os.environ.get("DCB200_K1_STREAM", "0"))


# Small host-built index tables (tile boundaries) uploaded once per distinct content and kept on the device: batches of a
# training run repeat a handful of shapes, and a pageable upload inside the step would block the host — and cannot be
# stream-captured (step.CapturedTrainStep warms the cache before it captures).
_TABLE_CACHE = collections.OrderedDict()
_TABLE_CACHE_MAX = 64


def _device_table(key, build, device):
    dev = torch.device(device)
    full = (key, dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    hit = _TABLE_CACHE.get(full)
    if hit is not None:
        _TABLE_CACHE.move_to_end(full)
        return hit
    if _capturing():
        raise _abi.DcError("index table missing from the device cache during stream capture (run the step once eagerly first)")
    t = build().to(dev)
    _TABLE_CACHE[full] = t
    if len(_TABLE_CACHE) > _TABLE_CACHE_MAX:
        _TABLE_CACHE.popitem(last=False)
    return t


TILE_WHOLE_MAX = int(os.environ.get("DCB200_TILE_WHOLE_MAX", "3600"))     # largest graph kept as ONE tile (3600: what dc_spmm_stage can hold in shared memory, 4 float4 lanes)


def make_tiles(ptr_host, num_nodes, target=TILE_NODES, whole_max=TILE_WHOLE_MAX):
    """Tile boundaries for the K1 kernels: whole graphs of the block-diagonal batch (a tile that is a union of whole graphs is
    closed under the edges, which the hop-chain kernels need), small graphs merged up to ~target receivers, graphs of more than
    ``whole_max`` rows split into target-sized chunks (those tiles are not closed: one launch per hop, L1 gathers)."""
    if ptr_host is None:
        return None
    tiles, cur = [0], 0
    for lo, hi in zip(ptr_host[:-1], ptr_host[1:]):
        n = hi - lo
        if n > max(target + target // 4, whole_max):
            if cur != lo:
                tiles.append(lo)
            k = -(-n // target)
            step = -(-n // k)
            tiles.extend(range(lo + step, hi, step))
            tiles.append(hi)
            cur = hi
        else:
            if hi - cur > target + target // 4 and cur != lo:
                tiles.append(lo)
                cur = lo
            if n > target + target // 4:      # a large graph that still fits: a tile of its own
                tiles.append(hi)
                cur = hi
        # else: keep merging
    if tiles[-1] != num_nodes:
        tiles.append(num_nodes)
    return tiles


# Node reordering for ONE large graph (no block-diagonal structure to tile by): the hops of a graph whose node order
# is spatially random fetch every source row slice from L2 / DRAM.  When the edge builder knows the positions (knn_graph /
# radius_graph on a single large cloud) it registers the grid-cell order of the points for the edge_index it returns; the
# structure is then built on relabelled nodes and the layer runs its hops in that order (features permuted in and out,
# dc_permute_rows).  Per-receiver sums keep their original edge order, so hop results are bit-identical.
REORDER = os.environ.get("DCB200_REORDER", "1") != "0"
REORDER_MIN_NODES = 32768
_ORDER_HINTS = {}


def _hint_key(edge_index):
    return (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, edge_index.device.index)


def register_order_hint(edge_index, order):
    """``order`` int32 [N]: a spatially coherent permutation of the nodes (new position -> node id) for this edge_index.
    The table holds only a weak reference: the hint lives exactly as long as the tensor (while it is alive its storage
    address cannot be recycled, so the key is unambiguous; nothing is pinned)."""
    for k in [k for k, (ref, _) in _ORDER_HINTS.items() if ref() is None]:
        del _ORDER_HINTS[k]
    _ORDER_HINTS[_hint_key(edge_index)] = (weakref.ref(edge_index), order)


def _order_hint(edge_index, num_nodes):
    hit = _ORDER_HINTS.get(_hint_key(edge_index))
    if hit is None or hit[0]() is None or hit[1].numel() != num_nodes:
        return None
    return hit[1]


def _eligible_order(edge_index, num_nodes, mode, ptr_host):
    """The registered spatial order if this structure qualifies for relabelling (one large TAG/GCN graph), else None."""
    if not (REORDER and mode in ("tag", "gcn") and num_nodes >= REORDER_MIN_NODES and (ptr_host is None or len(ptr_host) <= 2)):
        return None
    return _order_hint(edge_index, num_nodes)


def _need_pos(pos):
    """The C ABI reads 3 floats per point and has no dimension argument: anything but fp32 [N, 3] is an error."""
    _need(pos, _f32, "pos")
    if pos.dim() != 2 or pos.shape[1] != 3:
        raise _abi.DcError(f"pos: expected [N, 3] points, got {tuple(pos.shape)}")


def cell_order(pos):
    """int32 [N]: point indices in grid-cell order (dc_cell_order)."""
    _need_pos(pos)
    pos = pos.contiguous()
    N = pos.shape[0]
    order = torch.empty(N, dtype=_i32, device=pos.device)
    nb = _abi.lib().dc_knn_grid_workspace_bytes(N)
    ws = _workspace(nb, pos.device)
    _abi.call("dc_cell_order", _ptr(pos), N, _ptr(order), _ptr(ws), nb, _stream())
    return order


def permute_rows(x, perm, out=None):
    """out[i, :] = x[perm[i], :] (perm int32)."""
    _need(x, _f32, "x"); _need(perm, _i32, "perm")
    N, F = x.shape
    if out is None:
        out = torch.empty((N, F), dtype=_f32, device=x.device)
    _abi.call("dc_permute_rows", _ptr(x), _rows(x, "x"), _ptr(perm), _ptr(out), _rows(out, "out"), N, F, _stream())
    return out


class GraphCSR:
    """Device-resident structure of one (batched) graph: CSR by target for the forward
    aggregation, CSR by source for its transpose (built lazily, used by backward), the
    symmetric-normalisation vector ``dis = deg^-1/2`` and the per-edge weights in CSR order.

    mode "tag": PyG ``gcn_norm(add_self_loops=False)`` (TAGConv) — loops kept as ordinary edges.
    mode "gcn": ``add_remaining_self_loops`` — existing loops dropped, one appended per node.
    mode "gat": ``remove_self_loops`` + ``add_self_loops`` — same structure as "gcn", no dis.
    ``ptr_host`` (python list, ``Batch.ptr``) lets K1 align its tiles with graph boundaries.
    ``weighted_view`` gives a per-call copy carrying the norms of a per-edge weight (``weighted`` True).
    """

    weighted = False

    def __init__(self, edge_index, num_nodes, mode="tag", ptr_host=None, reorder=True):
        if mode not in ("tag", "gcn", "gat", "plain"):
            raise ValueError(mode)
        self.mode, self.N, self.E = mode, int(num_nodes), int(edge_index.shape[1])
        # the caller's tensor: graph_csr keys its cache on this tensor's address, so the entry must keep it alive (also on the
        # relabelling path below, which otherwise stores only the relabelled copy) or the allocator could hand the same
        # address to a different edge list of the same shape
        self._src_edge_index = edge_index
        # one large graph with a registered spatial order: build everything on relabelled nodes (see REORDER above)
        self.order = _eligible_order(edge_index, self.N, mode, ptr_host) if reorder else None
        self.rank = None
        if self.order is not None:
            rank = torch.empty(self.N, dtype=_i64, device=edge_index.device)
            rank[self.order.long()] = torch.arange(self.N, dtype=_i64, device=edge_index.device)
            edge_index = rank[edge_index]                      # same edges, same order, new node labels
            self.rank = rank.to(_i32)
        self.edge_index = edge_index.contiguous()     # dense [2, E]: the kernels that read edge_index index it as such
        self.self_loops = mode in ("gcn", "gat")
        self.rowptr, self.nbr, self.eid = csr_build(edge_index, self.N, 0, self.self_loops)
        self.dis = deg_inv_sqrt(self.rowptr, self.N, mode == "gcn") if mode in ("tag", "gcn") else None
        self.w, self.self_w = (edge_weights(self.rowptr, self.nbr, self.dis, self.N, mode == "gcn")
                               if self.dis is not None else (None, None))
        self.edges = pack_edges(self.nbr, self.w) if mode in ("tag", "gcn") else None
        self._t = None
        self._wt = None
        self._edges_t = None
        tiles = make_tiles(ptr_host, self.N)
        self.tile_ptr = (_device_table(("tiles", tuple(tiles)), lambda: torch.tensor(tiles, dtype=_i32), edge_index.device)
                         if tiles is not None else None)
        self.n_tiles = len(tiles) - 1 if tiles is not None else 0
        self._tiles_host = tiles
        # every tile boundary is a graph boundary <=> tiles are closed under the edges (needed by the hop chain)
        self.tiles_closed = tiles is not None and set(tiles) <= set(ptr_host)
        self._blocks = {}
        self._max_tile = max((b - a for a, b in zip(tiles[:-1], tiles[1:])), default=0) if tiles is not None else TILE_NODES
        self._view = None
        self._att = None

    def internal_view(self):
        """The same structure seen as a graph whose nodes ARE numbered in this structure's order (``order`` None).  A stack of
        layers on one relabelled graph permutes its input once, runs every layer on the view and permutes the result back
        once (``stack_enter`` / ``stack_exit``) instead of twice per layer."""
        if self.order is None:
            return self
        if self._view is None:
            v = copy.copy(self)
            v.order, v.rank, v._view = None, None, None
            v._src_edge_index = self.edge_index      # the relabelled edge list: the tensor the view is cached under
            v._blocks = {}
            self._view = v
        return self._view

    def blocks(self, transpose=False, unit=4):
        """K1 v7/v8 edge blocks (sliced-ELL copy of the CSR) of the forward / transposed structure, built lazily."""
        key = (bool(transpose), unit)
        if key not in self._blocks:
            rp = self.t[0] if transpose else self.rowptr
            self._blocks[key] = EdgeBlocks(rp, self._edges_t if transpose else self.edges, self.N, self.E, self._tiles_host, unit)
        return self._blocks[key]

    def attention_edges(self):
        """(keep, edge_index_sl) of a "gat" structure, built on first use and kept: ``keep`` int64 [E_nl], the ids of the edges
        that are not self loops, in edge order, or None when no edge is one (then alpha's edge rows are alpha_e[:E] as they
        stand, a copy instead of a gather); ``edge_index_sl`` int64 [2, E_nl + N] = ``add_self_loops(remove_self_loops(
        edge_index), N)``, PyG GATConv's attention edges, in the labels of the tensor the structure was built from.  The first
        call reads E_nl back to the host (one synchronisation); later calls launch nothing, so they can be captured."""
        if self.mode != "gat":
            raise _abi.DcError(f"attention_edges: needs a 'gat' structure, got {self.mode!r}")
        if self._att is None:
            ei = self._src_edge_index.to(_i64)
            keep = torch.nonzero(ei[0] != ei[1]).squeeze(1)
            loops = torch.arange(self.N, dtype=_i64, device=ei.device)
            edges = ei[:, keep] if keep.shape[0] < self.E else ei
            self._att = (keep if keep.shape[0] < self.E else None, torch.cat([edges, loops.expand(2, -1)], 1))
        return self._att

    @property
    def t(self):
        """(rowptr, nbr, eid) grouped by source — the transposed structure."""
        if self._t is None:
            if self.weighted:
                raise _abi.DcError("weighted view built without its by-source structure (weighted_view(..., transpose=True))")
            self._t = csr_build(self.edge_index, self.N, 1, self.self_loops)
            if self.dis is not None:
                self._wt = edge_weights(self._t[0], self._t[1], self.dis, self.N, False)[0]
                self._edges_t = pack_edges(self._t[1], self._wt)
        return self._t

    def to_internal(self, x):
        """Rows of ``x`` in the structure's node order (identity unless the graph was relabelled)."""
        return x if self.order is None else permute_rows(x, self.order)

    def from_internal(self, y, out=None):
        if self.order is None:
            return y
        return permute_rows(y, self.rank, out=out)

    def propagate(self, h, transpose=False, add=None, out=None, bias=None, relu=False, internal=False):
        """out = act(add + A_hat h + bias) (A_hat^T when ``transpose``); A_hat per ``mode``.
        Uses the tiled L1-reuse kernel when the layout allows, else the generic kernel; both give
        bit-identical results.  ``internal``: operands are already in the structure's node order."""
        if self.order is not None and not internal:
            res = self.propagate(self.to_internal(h), transpose=transpose, add=None if add is None else self.to_internal(add),
                                 bias=bias, relu=relu, internal=True)
            return self.from_internal(res, out=out)
        rp, nb, _ = self.t if transpose else (self.rowptr, self.nbr, self.eid)
        w = self._wt if transpose else self.w
        self_loop = self.mode == "gcn"
        variant = K1_VARIANT if K1_VARIANT != "auto" else ("blocks" if transpose else "lean")
        if variant == "blocks" and self.weighted:
            variant = "lean"      # edge blocks are a host-planned copy per structure; a weighted view lives for one call
        if variant == "blocks" and self.mode in ("tag", "gcn") and _tiled_ok(h, out, add, bias):
            return spmm_blocks(self.blocks(transpose), rp, self._edges_t if transpose else self.edges,
                               self.self_w if self_loop else None, h, add=add, self_loop=self_loop, bias=bias, relu=relu, out=out)
        if variant == "lean" and self.mode in ("tag", "gcn") and _tiled_ok(h, out, add, bias):
            return spmm_lean(rp, self._edges_t if transpose else self.edges, self.self_w if self_loop else None, h, add=add,
                             self_loop=self_loop, bias=bias, relu=relu, out=out, tile_ptr=self.tile_ptr, n_tiles=self.n_tiles)
        if variant != "generic" and self.mode in ("tag", "gcn") and _tiled_ok(h, out, add, bias):
            return spmm_tiled(rp, nb, w, self.self_w if self_loop else None, h, add=add, self_loop=self_loop, bias=bias,
                              relu=relu, out=out, tile_ptr=self.tile_ptr, n_tiles=self.n_tiles)
        if self.weighted:
            return spmm(rp, nb, h, edge_w=w, self_w=self.self_w if self_loop else None, add=add, self_loop=self_loop, bias=bias,
                        relu=relu, out=out)
        return spmm(rp, nb, h, dis=self.dis, add=add, self_loop=self_loop, bias=bias, relu=relu, out=out)


def weighted_view(g, edge_weight, normalize=True, fill_value=1.0, transpose=False):
    """The structure ``g`` ("tag" or "gcn", as built and cached for ``edge_index``) with the norms of ``edge_weight`` (fp32 [E] in
    the order of the ``edge_index`` ``g`` was built from): a shallow copy like ``internal_view()`` carrying its own ``dis``,
    ``w`` / ``edges`` (by target) and, with ``transpose``, ``_wt`` / ``_edges_t`` (by source), plus ``self_w``, ``loop_w`` and
    ``loop_eid`` for "gcn" (``add_remaining_self_loops(fill_value)``).  PyG's weighted gcn_norm, computed on the device for every
    call (dc_gcn_norm_weighted); the view is never cached and ``g`` is not modified.  ``normalize=False`` ("tag"): norm_e = w_e.
    ``propagate`` / ``propagate_chain`` run on the view unchanged, on the packed-record kernels."""
    if g.mode not in ("tag", "gcn"):
        raise _abi.DcError(f"weighted_view: needs a 'tag' or 'gcn' structure, got {g.mode!r}")
    _need(edge_weight, _f32, "edge_weight")
    if edge_weight.dim() != 1 or edge_weight.shape[0] != g.E:
        raise _abi.DcError(f"edge_weight: expected [{g.E}] (one weight per edge), got {tuple(edge_weight.shape)}")
    if edge_weight.device != g.rowptr.device:
        raise _abi.DcError(f"edge_weight is on {edge_weight.device}, the graph on {g.rowptr.device}")
    ew = edge_weight.contiguous()
    rpt, nbt, eidt = g.t if transpose else (None, None, None)
    N, E, dev = g.N, g.E, ew.device
    loops = g.mode == "gcn"
    v = copy.copy(g)
    v.weighted, v._blocks, v._view, v._t = True, {}, None, g._t if transpose else None
    v.edge_weight = ew
    v.dis = torch.empty(N, dtype=_f32, device=dev) if normalize else None
    v.loop_w = torch.empty(N, dtype=_f32, device=dev) if loops else None
    v.loop_eid = torch.empty(N, dtype=_i32, device=dev) if loops else None
    v.self_w = torch.empty(N, dtype=_f32, device=dev) if loops else None
    v.w = torch.empty(max(E, 1), dtype=_f32, device=dev)
    v.edges = torch.empty((max(E, 1), 2), dtype=_i32, device=dev)
    v._wt = torch.empty(max(E, 1), dtype=_f32, device=dev) if transpose else None
    v._edges_t = torch.empty((max(E, 1), 2), dtype=_i32, device=dev) if transpose else None
    _abi.call("dc_gcn_norm_weighted", _ptr(g.edge_index), E, N, _ptr(g.rowptr), _ptr(g.nbr), _ptr(g.eid), _ptr(rpt), _ptr(nbt),
              _ptr(eidt), _ptr(ew), float(fill_value), int(bool(normalize)), int(loops), _ptr(v.dis), _ptr(v.loop_w),
              _ptr(v.loop_eid), _ptr(v.self_w), _ptr(v.w), _ptr(v.edges), _ptr(v._wt), _ptr(v._edges_t), _stream())
    return v


def edge_sddmm(g, pairs, self_term=False):
    """s[e] = sum_k <G_k[dst_e], H_k[src_e]> by original edge id over ``g``'s by-target rows (and the self term
    s_self[i] = sum_k <G_k[i], H_k[i]>) for ``pairs`` = [(G_k, H_k)], all [N, F] in the structure's node order -> (s [E],
    s_self [N] or None); see dc_edge_sddmm.  More than ``_abi.MAX_CHAIN`` pairs are added in groups, in order."""
    N, F = pairs[0][0].shape
    s = torch.empty(max(g.E, 1), dtype=_f32, device=pairs[0][0].device)
    s_self = torch.empty(N, dtype=_f32, device=s.device) if self_term else None
    # the ABI wants the neighbour and edge-id arrays even without edges; an edgeless graph has empty ones (null pointers), and
    # then every row is empty and the stand-in is never read
    nbr, eid = (g.nbr, g.eid) if g.E else (g.rowptr, g.rowptr)
    for i0 in range(0, len(pairs), _abi.MAX_CHAIN):
        grp = pairs[i0:i0 + _abi.MAX_CHAIN]
        arr = (_abi.SddmmPair * len(grp))()
        for i, (G, H) in enumerate(grp):
            _need(G, _f32, "G"), _need(H, _f32, "H")
            if G.shape != (N, F) or H.shape != (N, F):
                raise _abi.DcError("edge_sddmm: every pair needs [N, F] operands")
            arr[i] = _abi.SddmmPair(_ptr(G), _rows(G, "G"), _ptr(H), _rows(H, "H"))
        e0 = _prof_begin()
        _abi.call("dc_edge_sddmm", _ptr(g.rowptr), _ptr(nbr), _ptr(eid), arr, len(grp), N, F, int(i0 > 0), _ptr(s),
                  _ptr(s_self), _stream())
        _prof_end(e0, op="sddmm", F=F, N=N, E=g.E, bytes=sddmm_bytes(N, g.E, F, len(grp), self_term))
    return (s if g.E else s.new_empty(0)), s_self


def sddmm_bytes(N, E, F, pairs, self_term):
    """Algorithmic DRAM bytes of one dc_edge_sddmm launch: every G_k and H_k row once, the row pointers, neighbour and edge ids,
    the outputs."""
    return 4 * (2 * pairs * N * F + (N + 1) + 2 * E + E + (N if self_term else 0))


def gcn_norm_backward(v, s, s_self=None):
    """dL/dedge_weight [E] (original edge order) from s = dL/dnorm of a weighted view built with ``normalize`` and ``transpose``;
    see dc_gcn_norm_weighted_backward.  ``s_self``: dL/dself_w of a "gcn" view."""
    rpt, nbt, eidt = v.t
    dw = torch.empty(max(v.E, 1), dtype=_f32, device=s.device)
    loops = s_self is not None
    _abi.call("dc_gcn_norm_weighted_backward", _ptr(v.rowptr), _ptr(v.nbr), _ptr(v.eid), _ptr(rpt), _ptr(nbt), _ptr(eidt),
              _ptr(v.edge_weight), _ptr(v.dis), _ptr(v.loop_w if loops else None), _ptr(v.loop_eid if loops else None), _ptr(s),
              _ptr(s_self), v.N, v.E, _ptr(dw), _stream())
    return dw if v.E else dw.new_empty(0)


def _al16(t):
    return t is None or (t.data_ptr() % 16 == 0)


def propagate_chain(g, hops, transpose=False, internal=False):
    """Consecutive hops of one layer: ``hops`` = [(in, add or None, out)], ``in`` of hop k normally the ``out`` of hop
    k-1.  One dc_spmm_chain launch when the structure allows it (block-diagonal batch with whole-graph tiles, F % 32 == 0,
    TAG/GCN weights), else one ``propagate`` per hop; both give bit-identical results."""
    if g.order is not None and not internal:
        return [g.propagate(h, transpose=transpose, add=a, out=o) for h, a, o in hops]
    F = hops[0][0].shape[1]
    ok = (K1_CHAIN and g.mode in ("tag", "gcn") and g.tiles_closed and len(hops) <= _abi.MAX_CHAIN
          and K1_VARIANT in ("auto", "lean", "blocks") and all(_tiled_ok(h, o, a, None) for h, a, o in hops))
    staged = ok and K1_STAGE and g.E > 0 and _abi.lib().dc_spmm_stage_supported(g._max_tile, F)
    if not (staged or (ok and F % 32 == 0)):
        return [g.propagate(h, transpose=transpose, add=a, out=o, internal=True) for h, a, o in hops]
    rp = g.t[0] if transpose else g.rowptr
    return spmm_chain(rp, g._edges_t if transpose else g.edges, g.self_w if g.mode == "gcn" else None, hops,
                      self_loop=g.mode == "gcn", tile_ptr=g.tile_ptr, n_tiles=g.n_tiles, max_tile_rows=g._max_tile if staged else 0)


def _tiled_ok(h, out, add, bias):
    F = h.shape[1]
    if any(t is not None and t.shape[0] * t.stride(0) >= 2 ** 32 for t in (h, out, add)):
        return False   # the tiled kernels index with 32-bit element offsets
    if F % 4 or h.dim() != 2 or h.stride(1) != 1 or h.stride(0) % 4 or not _al16(h) or not _al16(bias):
        return False
    for t in (out, add):
        if t is not None and (t.stride(1) != 1 or t.stride(0) % 4 or not _al16(t)):
            return False
    return True


_CSR_CACHE = {}
_CSR_CACHE_MAX = 16


def graph_csr(edge_index, num_nodes, mode="tag", ptr_host=None, reorder=True):
    """Structure cache: ``conv(x, edge_index)`` (models/model.py:71,77) passes the same
    ``edge_index`` tensor to every layer and hop, so the CSR pair is built once per batch.
    Keyed on storage identity + version; the entry pins the caller's tensor (``GraphCSR._src_edge_index``) so
    the address cannot be recycled while cached.  Writes to ``edge_index`` that bypass torch's version counter (raw
    pointer writes by a kernel through ``out=``) are not seen: call ``clear_csr_cache()`` after such a write."""
    if isinstance(edge_index, GraphCSR):
        return edge_index
    reorder = bool(reorder) and _eligible_order(edge_index, int(num_nodes), mode, ptr_host) is not None
    key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, int(num_nodes), mode,
           edge_index.device.index, reorder)
    hit = _CSR_CACHE.get(key)
    if hit is not None and hit._src_edge_index.data_ptr() == edge_index.data_ptr():
        return hit
    g = GraphCSR(edge_index, num_nodes, mode, ptr_host, reorder=reorder)
    if len(_CSR_CACHE) >= _CSR_CACHE_MAX:
        _CSR_CACHE.pop(next(iter(_CSR_CACHE)))
    _CSR_CACHE[key] = g
    return g


def adopt_csr(g):
    """Put a structure that was built directly (``GraphCSR(...)``) into the cache under the key of the tensor it was built
    from, so that the ``dcb200::`` custom ops — which take ``edge_index`` tensors — find it; returns that tensor."""
    ei = g._src_edge_index
    key = (ei.data_ptr(), tuple(ei.shape), ei._version, g.N, g.mode, ei.device.index, g.order is not None)
    if _CSR_CACHE.get(key) is not g:
        if len(_CSR_CACHE) >= _CSR_CACHE_MAX:
            _CSR_CACHE.pop(next(iter(_CSR_CACHE)))
        _CSR_CACHE[key] = g
    return ei


def clear_csr_cache():
    _CSR_CACHE.clear()


class _PermuteRows(torch.autograd.Function):
    """out[i] = x[perm[i]] with its exact adjoint (dx = dout[inverse]); both through dc_permute_rows."""

    @staticmethod
    def forward(ctx, x, perm, inverse):
        ctx.inverse = inverse
        return permute_rows(x.contiguous(), perm)

    @staticmethod
    def backward(ctx, dout):
        return permute_rows(dout.contiguous(), ctx.inverse), None, None


class _AttentionWeights(torch.autograd.Function):
    """alpha in the order of ``edge_index_sl``: cat(alpha_e[keep], alpha_s) [E_nl + N, H].  The backward writes the gradient
    back to [max(E, 1), H] by edge id (zeros at self-loop edges; ``keep`` holds each id once, so a plain index copy) and [N, H]."""

    @staticmethod
    def forward(ctx, alpha_e, alpha_s, keep, E):
        ctx.keep, ctx.rows, ctx.E = keep, alpha_e.shape[0], E
        return torch.cat([alpha_e[:E] if keep is None else alpha_e.index_select(0, keep), alpha_s], 0)

    @staticmethod
    def backward(ctx, dalpha):
        keep, E = ctx.keep, ctx.E
        n_keep = E if keep is None else keep.shape[0]
        dalpha_e = dalpha.new_zeros((ctx.rows, dalpha.shape[1]))
        if keep is None:
            dalpha_e[:E] = dalpha[:E]
        else:
            dalpha_e.index_copy_(0, keep, dalpha[:n_keep])
        return dalpha_e, dalpha[n_keep:], None, None


def attention_weights(alpha_e, alpha_s, keep, E):
    """PyG GATConv's ``alpha`` [E_nl + N, H] from the per-edge-id ``alpha_e`` [max(E, 1), H] and the loops' ``alpha_s`` [N, H]
    of ``dcb200::gat_conv_heads``, differentiable; ``keep`` from ``GraphCSR.attention_edges()``, E the number of edges."""
    return _AttentionWeights.apply(alpha_e, alpha_s, keep, E)


def stack_enter(x, edge_index, mode="tag", ptr_host=None):
    """Entry of a stack of layers that all run on ``edge_index`` (models/model.py:69-78).  For a relabelled large graph
    (``GraphCSR.order``) returns the features in the structure's node order, the relabelled edge list (with the structure's
    internal view adopted into the cache, so the layers neither rebuild nor permute) and the structure to leave through;
    otherwise the arguments unchanged and None."""
    g = edge_index if isinstance(edge_index, GraphCSR) else graph_csr(edge_index, x.shape[0], mode, ptr_host)
    if g.order is None:
        return x, edge_index, None
    return _PermuteRows.apply(x, g.order, g.rank), adopt_csr(g.internal_view()), g


def stack_exit(y, g):
    """Back to the caller's node order (identity when ``stack_enter`` returned None)."""
    return y if g is None else _PermuteRows.apply(y, g.rank, g.order)


# ----------------------------------------------------------------------------- K1
def spmm(rowptr, nbr, h, dis=None, edge_w=None, edge_w_index=None, self_w=None, add=None, self_loop=False, bias=None,
         relu=False, out=None):
    """out[i] = act(add[i] + sum_e w_e h[nbr[e]] (+ self term) + bias); see dc_spmm."""
    _need(h, _f32, "h")
    ldh = _rows(h, "h")
    N, F = h.shape
    if out is None:
        out = torch.empty((N, F), dtype=_f32, device=h.device)
    ldo = _rows(out, "out")
    ldadd = _rows(add, "add") if add is not None else 0
    for t, n in ((dis, "dis"), (edge_w, "edge_w"), (self_w, "self_w"), (add, "add"), (bias, "bias")):
        _need(t, _f32, n)
    e0 = _prof_begin()
    _abi.call("dc_spmm", _ptr(rowptr), _ptr(nbr), _ptr(dis), _ptr(edge_w), _ptr(edge_w_index), _ptr(self_w), _ptr(h), ldh,
              _ptr(out), ldo, _ptr(add), ldadd, N, F, int(bool(self_loop)), _ptr(bias), int(bool(relu)), _stream())
    if e0 is not None:
        E = nbr.numel()
        _prof_end(e0, op="spmm", F=F, N=N, E=E,
                  bytes=8 * N * F + 4 * E + 8 * N + 4 + (4 * N * F if add is not None else 0))
    return out


def edge_weights(rowptr, nbr, dis, num_nodes, want_self):
    """(w [E] in CSR order, self_w [N] or None): w[p] = fl(dis[nbr[p]] * dis[i]); see dc_edge_weights."""
    w = torch.empty(nbr.numel(), dtype=_f32, device=dis.device)
    self_w = torch.empty(num_nodes, dtype=_f32, device=dis.device) if want_self else None
    _abi.call("dc_edge_weights", _ptr(rowptr), _ptr(nbr), _ptr(dis), num_nodes, _ptr(w), _ptr(self_w), _stream())
    return w, self_w


def pack_edges(nbr, w):
    """int32 [E, 2] packed {neighbour, weight bits} records in CSR order; see dc_pack_edges."""
    E = nbr.numel()
    out = torch.empty((max(E, 1), 2), dtype=_i32, device=nbr.device)
    _abi.call("dc_pack_edges", _ptr(nbr), _ptr(w), E, _ptr(out), _stream())
    return out


class EdgeBlocks:
    """Sliced-ELL (SELL-4-sigma) copy of a CSR for dc_spmm_blocks; see include/dcb200.h (K1 v7)."""

    def __init__(self, rowptr, edges, num_nodes, num_edges, tiles_host=None, unit=4):
        import numpy as np
        self.unit = unit
        dev = rowptr.device
        N = int(num_nodes)
        if tiles_host is None:
            tp = np.arange(0, N + TILE_NODES, TILE_NODES, dtype=np.int64)[: -(-N // TILE_NODES) + 1] if N else np.zeros(1, np.int64)
            tp[-1] = N
        else:
            tp = np.asarray(tiles_host, dtype=np.int64)
        tup = np.zeros_like(tp)
        np.cumsum((np.diff(tp) + unit - 1) // unit, out=tup[1:])
        self.max_tile_rows = int(np.diff(tp).max()) if len(tp) > 1 else 0
        self.n_tiles, self.n_units = len(tp) - 1, int(tup[-1])
        both = _device_table(("blocks", unit, tp.tobytes()), lambda: torch.from_numpy(np.stack([tp, tup]).astype(np.int32)), dev)
        self.tile_ptr, self.tile_unit_ptr = both[0], both[1]
        cap = int(_abi.lib().dc_blocks_record_capacity(N, int(num_edges), self.n_tiles))
        self.slots = torch.empty((max(self.n_units, 1) * unit, 4), dtype=_i32, device=dev)
        self.recs = torch.empty((cap, 2), dtype=_i32, device=dev)
        self.status = torch.zeros(1, dtype=_i32, device=dev)
        self.tile_rec_ptr = torch.zeros(self.n_tiles + 1, dtype=_i32, device=dev)
        ws = _workspace(_abi.lib().dc_blocks_workspace_bytes(self.n_units), dev)
        _abi.call("dc_blocks_build", _ptr(rowptr), _ptr(edges), _ptr(self.tile_ptr), _ptr(self.tile_unit_ptr), self.n_tiles,
                  self.n_units, unit, _ptr(self.slots), _ptr(self.recs), cap, _ptr(self.tile_rec_ptr), _ptr(self.status), _ptr(ws), ws.numel(), _stream())


def spmm_blocks(blocks, rowptr, edges, self_w, h, add=None, self_loop=False, bias=None, relu=False, out=None, flags=None):
    """K1 v7 (edge blocks); see dc_spmm_blocks."""
    _need(h, _f32, "h")
    ldh = _rows(h, "h")
    N, F = h.shape
    if out is None:
        out = torch.empty((N, F), dtype=_f32, device=h.device)
    ldo = _rows(out, "out")
    ldadd = _rows(add, "add") if add is not None else 0
    e0 = _prof_begin()
    _abi.call("dc_spmm_blocks", _ptr(blocks.slots), _ptr(blocks.recs), _ptr(rowptr), _ptr(edges), _ptr(blocks.tile_ptr),
              _ptr(blocks.tile_unit_ptr), _ptr(blocks.tile_rec_ptr), blocks.n_tiles, _ptr(self_w), _ptr(h), ldh, _ptr(out), ldo, _ptr(add), ldadd, F, int(bool(self_loop)), _ptr(bias),
              int(bool(relu)), K1_FLAGS if flags is None else int(flags), _stream())
    if e0 is not None:
        E = edges.shape[0]
        _prof_end(e0, op="spmm", F=F, N=N, E=E,
                  bytes=8 * N * F + 4 * E + 8 * N + 4 + (4 * N * F if add is not None else 0))
    return out


def spmm_lean(rowptr, edges, self_w, h, add=None, self_loop=False, bias=None, relu=False, out=None, tile_ptr=None, n_tiles=0,
              tile_nodes=TILE_NODES):
    """K1 v6 (lean tile x slice kernel on packed edge records); see dc_spmm_lean."""
    _need(h, _f32, "h")
    ldh = _rows(h, "h")
    N, F = h.shape
    if out is None:
        out = torch.empty((N, F), dtype=_f32, device=h.device)
    ldo = _rows(out, "out")
    ldadd = _rows(add, "add") if add is not None else 0
    e0 = _prof_begin()
    _abi.call("dc_spmm_lean", _ptr(rowptr), _ptr(edges), _ptr(self_w), _ptr(h), ldh, _ptr(out), ldo, _ptr(add), ldadd, N, F,
              int(bool(self_loop)), _ptr(bias), int(bool(relu)), _ptr(tile_ptr), int(n_tiles), int(tile_nodes), _stream())
    if e0 is not None:
        E = edges.shape[0]
        _prof_end(e0, op="spmm", F=F, N=N, E=E,
                  bytes=8 * N * F + 4 * E + 8 * N + 4 + (4 * N * F if add is not None else 0))
    return out


def spmm_chain(rowptr, edges, self_w, hops, self_loop=False, tile_ptr=None, n_tiles=0, tile_nodes=TILE_NODES, max_tile_rows=0):
    """K1 v9 / v10: ``hops`` = [(in, add or None, out), ...] consecutive hops of one layer in ONE launch; every tile must be
    closed under the edges (``GraphCSR.tiles_closed``).  ``max_tile_rows`` > 0 selects the TMA-staged kernel
    (dc_spmm_stage: tile slice in shared memory, any F % 4 == 0), else dc_spmm_chain (L1 gathers, F % 32 == 0)."""
    arr = (_abi.Hop * len(hops))()
    N, F = hops[0][0].shape
    nbytes = 0
    for i, (h, add, out) in enumerate(hops):
        _need(h, _f32, "in"); _need(add, _f32, "add"); _need(out, _f32, "out")
        if h.shape != (N, F) or out.shape != (N, F) or (add is not None and add.shape != (N, F)):
            raise _abi.DcError("spmm_chain: every hop needs [N, F] operands")
        arr[i] = _abi.Hop(_ptr(h), _rows(h, "in"), _ptr(add), _rows(add, "add") if add is not None else 0, _ptr(out),
                          _rows(out, "out"))
        nbytes += 8 * N * F + 4 * edges.shape[0] + 8 * N + 4 + (4 * N * F if add is not None else 0)
    e0 = _prof_begin()
    if max_tile_rows:
        _abi.call("dc_spmm_stage", _ptr(rowptr), _ptr(edges), _ptr(self_w), arr, len(hops), N, F, int(bool(self_loop)),
                  _ptr(tile_ptr), int(n_tiles), int(tile_nodes), int(max_tile_rows), _stream())
    elif K1_STREAM and not self_loop and F % 32 == 0:
        _abi.call("dc_spmm_stream", _ptr(rowptr), _ptr(edges), arr, len(hops), N, F, _ptr(tile_ptr), int(n_tiles), int(tile_nodes),
                  _stream())
    else:
        _abi.call("dc_spmm_chain", _ptr(rowptr), _ptr(edges), _ptr(self_w), arr, len(hops), N, F, int(bool(self_loop)), _ptr(tile_ptr),
                  int(n_tiles), int(tile_nodes), _stream())
    if e0 is not None:
        _prof_end(e0, op="spmm", F=F, N=N, E=edges.shape[0], bytes=nbytes, hops=len(hops))
    return [h[2] for h in hops]


def spmm_tiled(rowptr, nbr, w, self_w, h, add=None, self_loop=False, bias=None, relu=False, out=None, tile_ptr=None,
               n_tiles=0, tile_nodes=TILE_NODES):
    """K1 v2 (tile x slice, L1 reuse); see dc_spmm_tiled."""
    _need(h, _f32, "h")
    ldh = _rows(h, "h")
    N, F = h.shape
    if out is None:
        out = torch.empty((N, F), dtype=_f32, device=h.device)
    ldo = _rows(out, "out")
    ldadd = _rows(add, "add") if add is not None else 0
    e0 = _prof_begin()
    _abi.call("dc_spmm_tiled", _ptr(rowptr), _ptr(nbr), _ptr(w), _ptr(self_w), _ptr(h), ldh, _ptr(out), ldo, _ptr(add), ldadd,
              N, F, int(bool(self_loop)), _ptr(bias), int(bool(relu)), _ptr(tile_ptr), int(n_tiles), int(tile_nodes),
              {"tiled": 0, "tiled_prefetch": 1, "tiled8": 2, "smem": 3}.get(K1_VARIANT, 2), _stream())
    if e0 is not None:
        E = nbr.numel()
        _prof_end(e0, op="spmm", F=F, N=N, E=E,
                  bytes=8 * N * F + 4 * E + 8 * N + 4 + (4 * N * F if add is not None else 0))
    return out


def edge_relu(rowptr, nbr, p, q, r=None, mode=0):
    """Fused per-edge relu-sum and its backward gathers (A9 layer); see dc_edge_relu."""
    N, F = p.shape
    out = torch.empty((N, F), dtype=_f32, device=p.device)
    for t in (p, q, r):
        if t is not None and (t.stride(0) != F or t.stride(1) != 1):
            raise _abi.DcError("edge_relu: operands must be contiguous [N, F]")
    _abi.call("dc_edge_relu", _ptr(rowptr), _ptr(nbr), _ptr(p), _ptr(q), _ptr(r), _ptr(out), F, N, F, int(mode), _stream())
    return out


# ----------------------------------------------------------------------------- K2 / K3
# accuracy lab (scripts/acc_lab.py): DCB200_GEMM=fp32 forces the exact-fp32 FFMA kernel for every product
FORCE_GEMM_PRECISION = {"fp32": GEMM_FP32, "tc": GEMM_PREFER_TC}.get(os.environ.get("DCB200_GEMM", ""))


def gemm(segs, M, N, trans_a=False, trans_b=True, bias=None, relu=False, out=None, accumulate=False,
         precision=GEMM_AUTO):
    """C[M,N] = act(sum_s opA(A_s) opB(B_s) + bias) (+C); segs = [(A_s, B_s), ...]; see dc_gemm.
    More than ``_abi.MAX_SEGS`` segments (a decoder fed by >= 4 attention heads, TAGConv with K >= 4) are chained
    in groups with ``accumulate``; bias and ReLU are applied by the last group."""
    if FORCE_GEMM_PRECISION is not None:
        precision = FORCE_GEMM_PRECISION
    if len(segs) > _abi.MAX_SEGS:
        groups = [segs[i:i + _abi.MAX_SEGS] for i in range(0, len(segs), _abi.MAX_SEGS)]
        for gi, grp in enumerate(groups):
            last = gi == len(groups) - 1
            out = gemm(grp, M, N, trans_a=trans_a, trans_b=trans_b, bias=bias if last else None, relu=relu and last, out=out,
                       accumulate=accumulate or gi > 0, precision=precision)
        return out
    arr = (_abi.GemmSeg * len(segs))()
    ktot = 0
    dev = segs[0][0].device
    for i, (A, B) in enumerate(segs):
        _need(A, _f32, "A"), _need(B, _f32, "B")
        lda, ldb = _rows(A, "A"), _rows(B, "B")
        K = A.shape[0] if trans_a else A.shape[1]
        Kb = B.shape[1] if trans_b else B.shape[0]
        Ma = A.shape[1] if trans_a else A.shape[0]
        Nb = B.shape[0] if trans_b else B.shape[1]
        if K != Kb or Ma != M or Nb != N:
            raise _abi.DcError(f"gemm: segment {i} shapes {tuple(A.shape)} x {tuple(B.shape)} do not give [{M},{N}]")
        arr[i] = _abi.GemmSeg(A.data_ptr(), lda, B.data_ptr(), ldb, K)
        ktot += K
    if out is None:
        out = torch.empty((M, N), dtype=_f32, device=dev)
    ldc = _rows(out, "out")
    nb = _abi.lib().dc_gemm_workspace_bytes(M, N, ktot, int(trans_a), int(trans_b))
    ws = _workspace(nb, dev) if nb else None
    e0 = _prof_begin()
    _abi.call("dc_gemm", arr, len(segs), int(trans_a), int(trans_b), M, N, _ptr(out), ldc, _ptr(bias), int(bool(relu)),
              int(bool(accumulate)), int(precision), _ptr(ws), nb, _stream())
    _prof_end(e0, op="gemm", M=M, N=N, K=ktot, flops=2.0 * M * N * ktot)
    return out


def gemm_batched(problems, trans_a=False, trans_b=True, relu=False, accumulate=False):
    """problems = [(A, B, C), ...]: C_i = act(opA(A_i) opB(B_i)) (+C_i) for all i in one tensor-core launch; see
    dc_gemm_batched.  A problem may carry a fused epilogue (A, B, C, E, rowv): C = E o (acc - rowv[:, None]).
    Falls back to one dc_gemm per problem when a problem does not fit the tensor path.  The fused epilogue excludes
    ``relu`` and ``accumulate``, as in dc_gemm_batched."""
    if (relu or accumulate) and any(len(q) > 3 for q in problems):
        raise _abi.DcError("gemm_batched: the fused epilogue operand E excludes relu and accumulate")
    problems = [q for q in problems if q[2].numel() > 0]
    if not problems:
        return
    arr = (_abi.GemmProblem * len(problems))()
    flops = 0.0
    ok = True
    for i, q in enumerate(problems):
        A, B, Cm = q[:3]
        E, rowv = (q[3], q[4]) if len(q) > 3 else (None, None)
        _need(A, _f32, "A"), _need(B, _f32, "B"), _need(Cm, _f32, "C"), _need(E, _f32, "E"), _need(rowv, _f32, "rowv")
        lda, ldb, ldc = _rows(A, "A"), _rows(B, "B"), _rows(Cm, "C")
        K = A.shape[0] if trans_a else A.shape[1]
        Kb = B.shape[1] if trans_b else B.shape[0]
        M = A.shape[1] if trans_a else A.shape[0]
        N = B.shape[0] if trans_b else B.shape[1]
        if K != Kb or tuple(Cm.shape) != (M, N):
            raise _abi.DcError(f"gemm_batched: problem {i}: {tuple(A.shape)} x {tuple(B.shape)} -> {tuple(Cm.shape)}")
        ok = ok and K > 0 and lda % 4 == 0 and ldb % 4 == 0 and A.data_ptr() % 16 == 0 and B.data_ptr() % 16 == 0
        arr[i] = _abi.GemmProblem(A.data_ptr(), lda, B.data_ptr(), ldb, Cm.data_ptr(), ldc, M, N, K, _ptr(E),
                                  _rows(E, "E") if E is not None else 0, _ptr(rowv))
        flops += 2.0 * M * N * K
    if not ok or FORCE_GEMM_PRECISION == GEMM_FP32:
        for q in problems:
            A, B, Cm = q[:3]
            gemm([(A, B)], Cm.shape[0], Cm.shape[1], trans_a=trans_a, trans_b=trans_b, relu=relu, out=Cm, accumulate=accumulate)
            if len(q) > 3:
                Cm.copy_(q[3] * (Cm - q[4][:, None]))
        return
    nb = _abi.lib().dc_gemm_batched_workspace_bytes(len(problems))
    ws = _workspace(nb, problems[0][0].device)
    stage = _staging_get(nb)
    e0 = _prof_begin()
    _abi.call("dc_gemm_batched", arr, len(problems), int(trans_a), int(trans_b), int(bool(relu)), int(bool(accumulate)), _ptr(ws), nb,
              stage.data_ptr(), stage.numel(), _stream())
    _prof_end(e0, op="gemm", M=0, N=0, K=0, flops=flops)
    _staging_put(stage)


def rowdot(A, B):
    """out[m] = sum_n A[m, n] * B[m, n]; see dc_rowdot."""
    _need(A, _f32, "A"), _need(B, _f32, "B")
    M, N = A.shape
    out = torch.empty(M, dtype=_f32, device=A.device)
    _abi.call("dc_rowdot", _ptr(A), _rows(A, "A"), _ptr(B), _rows(B, "B"), M, N, _ptr(out), _stream())
    return out


def colsum(X):
    _need(X, _f32, "X")
    ldx = _rows(X, "X")
    M, N = X.shape
    out = torch.empty(N, dtype=_f32, device=X.device)
    nb = _abi.lib().dc_colsum_workspace_bytes(M, N)
    ws = _workspace(nb, X.device)
    _abi.call("dc_colsum", _ptr(X), ldx, M, N, _ptr(out), _ptr(ws), nb, _stream())
    return out


def relu_bwd(Y, dY):
    Y, dY = Y.contiguous(), dY.contiguous()
    dX = torch.empty_like(dY)
    _abi.call("dc_relu_bwd", _ptr(Y), _ptr(dY), _ptr(dX), Y.numel(), _stream())
    return dX


def relu_bwd_colsum(Y, dY):
    """(dX, colsum(dX)) with dX = dY * (Y > 0) in one pass; see dc_relu_bwd_colsum."""
    _need(Y, _f32, "Y"), _need(dY, _f32, "dY")
    M, N = Y.shape
    ldy, lddy = _rows(Y, "Y"), _rows(dY, "dY")
    dX = torch.empty((M, N), dtype=_f32, device=Y.device)
    out = torch.empty(N, dtype=_f32, device=Y.device)
    nb = _abi.lib().dc_colsum_workspace_bytes(M, N)
    ws = _workspace(nb, Y.device)
    _abi.call("dc_relu_bwd_colsum", _ptr(Y), ldy, _ptr(dY), lddy, _ptr(dX), N, M, N, _ptr(out), _ptr(ws), nb, _stream())
    return dX, out


def relu_bwd_db(Y, dY, relu, need_db):
    """The head of every layer backward: undo the fused ReLU and take the bias gradient -> (dY', db or None)."""
    if relu and need_db:
        return relu_bwd_colsum(Y, dY)
    if relu:
        dY = relu_bwd(Y, dY)
    return dY, (colsum(dY) if need_db else None)


# ----------------------------------------------------------------------------- K4
def _ptr_tensor(num_points, batch, ptr, device):
    if ptr is not None:
        return ptr.to(device=device, dtype=_i64).contiguous()
    if batch is None:
        return torch.tensor([0, num_points], dtype=_i64, device=device)
    counts = torch.bincount(batch.to(device))
    return torch.cat([counts.new_zeros(1), counts.cumsum(0)]).to(_i64)


# Neighbour search strategy: "auto" = uniform grid (K4g) for a single point cloud of at least KNN_GRID_MIN points and
# one grid per graph for a batch of at least KNN_GRID_MIN points whose clouds average at least KNN_GRID_BATCH_MIN (dc_knn_grid_batched), tiled brute force
# (K4) otherwise; "brute" / "grid" force one.  Results are bit-identical.
KNN_MODE = os.environ.get("DCB200_KNN", "auto")
KNN_GRID_MIN = 16384
RADIUS_GRID_BATCH_MIN = 1024   # the radius scan has no insertion path: its brute-force form holds out until ~1000 points per graph
KNN_GRID_BATCH_MIN = int(os.environ.get("DCB200_KNN_GRID_BATCH_MIN", "256"))   # measured: 2x faster than brute force from 250 points per graph up


def _use_grid(N, batch, ptr, width):
    single = batch is None and (ptr is None or ptr.numel() == 2)
    return single and width <= 128 and (KNN_MODE == "grid" or (KNN_MODE == "auto" and N >= KNN_GRID_MIN))


def _use_grid_batched(N, B, width, per_graph_min=None):
    """One grid per graph (dc_knn_grid_batched / dc_radius_grid_batched) for a batch of B >= 2 clouds."""
    per_graph_min = KNN_GRID_BATCH_MIN if per_graph_min is None else per_graph_min
    return (B >= 2 and width <= 128 and B < (1 << 24)
            and (KNN_MODE == "grid" or (KNN_MODE == "auto" and N >= KNN_GRID_MIN and N >= B * per_graph_min)))


def knn_table(pos, k, batch=None, ptr=None, loop=False):
    """int32 [N, k (+1 if not loop)] neighbour table, ascending (distance, index), -1 padded."""
    _need_pos(pos)
    pos = pos.contiguous()
    N = pos.shape[0]
    W = k + (0 if loop else 1)
    tab = torch.empty((N, W), dtype=_i32, device=pos.device)
    if _use_grid(N, batch, ptr, W):
        nb = _abi.lib().dc_knn_grid_workspace_bytes(N)
        ws = _workspace(nb, pos.device)
        order = torch.empty(N, dtype=_i32, device=pos.device) if REORDER and N >= REORDER_MIN_NODES else None
        _abi.call("dc_knn_grid", _ptr(pos), N, k, int(bool(loop)), _ptr(tab), _ptr(order), _ptr(ws), nb, _stream())
        tab._cell_order = order     # the search's own counting sort doubles as the spatial node order (ops.REORDER)
        tab._grid_ws = ws           # tests read the device-side grid / brute-force decision out of it (grid_took_it)
        return tab
    p = _ptr_tensor(N, batch, ptr, pos.device)
    B = p.numel() - 1
    if _use_grid_batched(N, B, W):
        nb = _abi.lib().dc_knn_grid_batched_workspace_bytes(N, B)
        ws = _workspace(nb, pos.device)
        _abi.call("dc_knn_grid_batched", _ptr(pos), _ptr(p), B, N, k, int(bool(loop)), _ptr(tab), _ptr(ws), nb, _stream())
        tab._grid_ws = ws
        return tab
    _abi.call("dc_knn", _ptr(pos), _ptr(p), B, N, k, int(bool(loop)), _ptr(tab), _stream())
    return tab


def radius_table(pos, r, batch=None, ptr=None, loop=False, max_num_neighbors=32):
    _need_pos(pos)
    pos = pos.contiguous()
    N = pos.shape[0]
    W = max_num_neighbors + (0 if loop else 1)
    tab = torch.empty((N, W), dtype=_i32, device=pos.device)
    cnt = torch.empty(N, dtype=_i32, device=pos.device)
    if _use_grid(N, batch, ptr, W):
        nb = _abi.lib().dc_knn_grid_workspace_bytes(N)
        ws = _workspace(nb, pos.device)
        order = torch.empty(N, dtype=_i32, device=pos.device) if REORDER and N >= REORDER_MIN_NODES else None
        _abi.call("dc_radius_grid", _ptr(pos), N, float(r), max_num_neighbors, int(bool(loop)), _ptr(tab), _ptr(cnt), _ptr(order),
                  _ptr(ws), nb, _stream())
        tab._cell_order = order
        return tab, cnt
    p = _ptr_tensor(N, batch, ptr, pos.device)
    B = p.numel() - 1
    if _use_grid_batched(N, B, W, RADIUS_GRID_BATCH_MIN):
        nb = _abi.lib().dc_knn_grid_batched_workspace_bytes(N, B)
        ws = _workspace(nb, pos.device)
        _abi.call("dc_radius_grid_batched", _ptr(pos), _ptr(p), B, N, float(r), max_num_neighbors, int(bool(loop)), _ptr(tab), _ptr(cnt),
                  _ptr(ws), nb, _stream())
        tab._grid_ws = ws
        return tab, cnt
    _abi.call("dc_radius", _ptr(pos), _ptr(p), B, N, float(r), max_num_neighbors, int(bool(loop)), _ptr(tab), _ptr(cnt), _stream())
    return tab, cnt


def grid_took_it(tab):
    """True if the uniform-grid kernel produced this table, False if the library's device-side dispatch handed the cloud to
    the brute-force kernel (a grid cannot split it: outliers, few dense clusters).  Reads one int back (host sync)."""
    ws = getattr(tab, "_grid_ws", None)
    if ws is None:
        return False
    return bool(ws[40:44].view(torch.int32).item())   # GridParams::use_grid at byte 40 (static_assert in csrc/knn_grid.cu)


def table_to_edge_index(tab):
    """Padded neighbour table -> int64 [2, E] (row 0 = neighbour, row 1 = query).  Reads E back
    (one host sync) because the output shape is data dependent, like torch_cluster."""
    N, W = tab.shape
    cap = N * W
    ei = torch.empty((2, max(cap, 1)), dtype=_i64, device=tab.device)
    num = torch.zeros(1, dtype=_i64, device=tab.device)
    nb = _abi.lib().dc_nbr_to_edge_index_workspace_bytes(N)
    ws = _workspace(nb, tab.device)
    _abi.call("dc_nbr_to_edge_index", _ptr(tab), N, W, _ptr(ei), max(cap, 1), _ptr(num), _ptr(ws), nb, _stream())
    E = int(num.item())
    return ei[:, :E].contiguous() if E != cap else ei


# ----------------------------------------------------------------------------- A6
def mesh_edges(triangles, offset=0, out=None, start=0):
    _need(triangles, _i64, "triangles")
    tri = triangles.contiguous()
    T = tri.shape[0]
    if out is None:
        out = torch.empty((2, 3 * T), dtype=_i64, device=tri.device)
    _abi.call("dc_mesh_edges", _ptr(tri), T, int(offset), _ptr(out), out.shape[1], int(start), _stream())
    return out


def posenc(pos, out=None, col0=0):
    _need_pos(pos)
    pos = pos.contiguous()
    N = pos.shape[0]
    if out is None:
        out = torch.empty((N, 21), dtype=_f32, device=pos.device)
    _abi.call("dc_posenc", _ptr(pos), N, _ptr(out), _rows(out, "out"), int(col0), _stream())
    return out


# ----------------------------------------------------------------------------- N3: batch assembly
def _index_bytes(t, name):
    if t.dtype == _i32:
        return 4
    if t.dtype == _i64:
        return 8
    raise _abi.DcError(f"{name}: expected int32 or int64 indices, got {t.dtype}")


def batch_vector(node_ptr, num_nodes):
    """Batch.batch: int64 [N] graph id per node from ``ptr`` (int64 [B+1], device)."""
    _need(node_ptr, _i64, "node_ptr")
    out = torch.empty(int(num_nodes), dtype=_i64, device=node_ptr.device)
    _abi.call("dc_batch_vector", _ptr(node_ptr), node_ptr.numel() - 1, int(num_nodes), _ptr(out), _stream())
    return out


def edges_offset(local, edge_ptr, node_ptr, out=None):
    """``local`` [2, E] graph-local indices (int32 / int64), graphs back to back -> int64 [2, E] with each graph's
    cumulative node offset added (the ``edge_index`` increment of PyG's collate)."""
    _need(edge_ptr, _i64, "edge_ptr"); _need(node_ptr, _i64, "node_ptr")
    if not local.is_cuda:
        raise _abi.DcError("local: expected a CUDA tensor (libdcb200 has no CPU path)")
    ib = _index_bytes(local, "local")
    E = local.shape[1]
    if out is None:
        out = torch.empty((2, E), dtype=_i64, device=local.device)
    _abi.call("dc_edges_offset", _ptr(local), ib, _rows(local, "local"), _ptr(edge_ptr), _ptr(node_ptr), node_ptr.numel() - 1, E,
              _ptr(out), _rows(out, "out"), _stream())
    return out


def mesh_edges_batched(triangles, tri_ptr=None, node_ptr=None, num_graphs=None, nodes_per_graph=0, out=None):
    """mesh_to_graph edges of a whole batch in one launch.  Ragged: ``triangles`` [sum T, 3] local indices with
    ``tri_ptr`` / ``node_ptr``.  Instanced (``tri_ptr`` None): ``triangles`` [T, 3] is a template shared by
    ``num_graphs`` graphs of ``nodes_per_graph`` nodes each."""
    if not triangles.is_cuda:
        raise _abi.DcError("triangles: expected a CUDA tensor (libdcb200 has no CPU path)")
    ib = _index_bytes(triangles, "triangles")
    tri = triangles.contiguous()
    if tri_ptr is not None:
        _need(tri_ptr, _i64, "tri_ptr"); _need(node_ptr, _i64, "node_ptr")
        B, T, tpg = node_ptr.numel() - 1, tri.shape[0], 0
    else:
        B, tpg = int(num_graphs), tri.shape[0]
        T = B * tpg
    if out is None:
        out = torch.empty((2, 3 * T), dtype=_i64, device=tri.device)
    _abi.call("dc_mesh_edges_batched", _ptr(tri), ib, _ptr(tri_ptr), _ptr(node_ptr), B, T, tpg, int(nodes_per_graph), _ptr(out),
              _rows(out, "out"), _stream())
    return out


def node_features(pos, head=None, node_ptr=None, out=None):
    """[head[graph(n)] | to_log_freq(pos[n], 3, 1)]: the 21-d soft features (``head`` None) or the collider's
    25-d ``_feature_rigid`` (``head`` fp32 [B, 4] = force_vector | force)."""
    _need_pos(pos); _need(head, _f32, "head"); _need(node_ptr, _i64, "node_ptr")
    pos = pos.contiguous()
    N = pos.shape[0]
    H = 0 if head is None else head.shape[1]
    if out is None:
        out = torch.empty((N, H + 21), dtype=_f32, device=pos.device)
    _abi.call("dc_node_features", _ptr(pos), _ptr(None if head is None else head.contiguous()), H, _ptr(node_ptr),
              0 if node_ptr is None else node_ptr.numel() - 1, N, _ptr(out), _rows(out, "out"), _stream())
    return out


def instance_points(template, centers):
    """fp64 template [V, 3] + fp64 centers [B, 3] -> fp32 [B*V, 3] (fp64 add, then round: Open3D translate)."""
    _need(template, torch.float64, "template"); _need(centers, torch.float64, "centers")
    B, V = centers.shape[0], template.shape[0]
    out = torch.empty((B * V, 3), dtype=_f32, device=template.device)
    _abi.call("dc_instance_points", _ptr(template.contiguous()), _ptr(centers.contiguous()), B, V, _ptr(out), _stream())
    return out


# ----------------------------------------------------------------------------- K6
def gat_scores(xs, att_src, att_dst, heads, C_):
    N = xs.shape[0]
    a_src = torch.empty((N, heads), dtype=_f32, device=xs.device)
    a_dst = torch.empty((N, heads), dtype=_f32, device=xs.device)
    _abi.call("dc_gat_scores", _ptr(xs), _rows(xs, "xs"), N, heads, C_, _ptr(att_src.contiguous()), _ptr(att_dst.contiguous()),
              _ptr(a_src), _ptr(a_dst), _stream())
    return a_src, a_dst


def gat_softmax(g, a_src, a_dst, slope):
    alpha_e = torch.zeros(max(g.E, 1), dtype=_f32, device=a_src.device)
    alpha_s = torch.empty(g.N, dtype=_f32, device=a_src.device)
    _abi.call("dc_gat_softmax", _ptr(g.rowptr), _ptr(g.nbr), _ptr(g.eid), _ptr(a_src), _ptr(a_dst), float(slope), g.N,
              _ptr(alpha_e), _ptr(alpha_s), _stream())
    return alpha_e, alpha_s


def gat_bwd_edge(g, a_src, a_dst, slope, alpha_e, alpha_s, xs, dout):
    dz_e = torch.zeros(max(g.E, 1), dtype=_f32, device=xs.device)
    dz_s = torch.empty(g.N, dtype=_f32, device=xs.device)
    da_dst = torch.empty(g.N, dtype=_f32, device=xs.device)
    _abi.call("dc_gat_bwd_edge", _ptr(g.rowptr), _ptr(g.nbr), _ptr(g.eid), _ptr(a_src), _ptr(a_dst), float(slope),
              _ptr(alpha_e), _ptr(alpha_s), _ptr(xs), _rows(xs, "xs"), _ptr(dout), _rows(dout, "dout"), xs.shape[1], g.N,
              _ptr(dz_e), _ptr(dz_s), _ptr(da_dst), _stream())
    return dz_e, dz_s, da_dst


def segment_sum(rowptr, eid, val, init, N):
    out = torch.empty(N, dtype=_f32, device=val.device)
    _abi.call("dc_segment_sum", _ptr(rowptr), _ptr(eid), _ptr(val), _ptr(init), N, _ptr(out), _stream())
    return out


# ----------------------------------------------------------------------------- K6 multi-head (csrc/gat.cu)
def _dout_heads(heads, C_, concat):
    """(head stride, scale) of the per-head output gradient: concat reads head h's column slice, mean reads dout / H
    (stride 0) without materialising it."""
    return (C_, 1.0) if concat else (0, 1.0 / heads)


def gat_aggregate(g, xs, a_src, a_dst, slope, heads, C_, concat, bias=None, relu=False):
    """Per-head softmax + aggregation + concat / mean + bias (+ReLU) -> (out, alpha_e [max(E,1), H], alpha_s [N, H]);
    see dc_gat_aggregate."""
    _need(xs, _f32, "xs"), _need(bias, _f32, "bias")
    out = torch.empty((g.N, heads * C_ if concat else C_), dtype=_f32, device=xs.device)
    alpha_e = torch.zeros((max(g.E, 1), heads), dtype=_f32, device=xs.device)
    alpha_s = torch.empty((g.N, heads), dtype=_f32, device=xs.device)
    _abi.call("dc_gat_aggregate", _ptr(g.rowptr), _ptr(g.nbr), _ptr(g.eid), _ptr(xs), _rows(xs, "xs"), _ptr(a_src), _ptr(a_dst),
              float(slope), int(heads), int(C_), int(bool(concat)), _ptr(bias), int(bool(relu)), g.N, _ptr(out), _rows(out, "out"),
              _ptr(alpha_e), _ptr(alpha_s), _stream())
    return out, alpha_e, alpha_s


def gat_bwd_edge_heads(g, a_src, a_dst, slope, alpha_e, alpha_s, xs, dout, heads, C_, concat, dalpha_e=None, dalpha_s=None):
    """-> (dz_e [max(E,1), H], dz_s [N, H], da_dst [N, H]); see dc_gat_bwd_edge_heads.  ``dalpha_e`` [max(E,1), H] (by edge id)
    / ``dalpha_s`` [N, H]: the gradient that reaches alpha itself, added to the one through the aggregation
    (dc_gat_bwd_edge_heads_ext); without either the call is dc_gat_bwd_edge_heads."""
    hs, scale = _dout_heads(heads, C_, concat)
    dz_e = torch.zeros((max(g.E, 1), heads), dtype=_f32, device=xs.device)
    dz_s = torch.empty((g.N, heads), dtype=_f32, device=xs.device)
    da_dst = torch.empty((g.N, heads), dtype=_f32, device=xs.device)
    args = (_ptr(g.rowptr), _ptr(g.nbr), _ptr(g.eid), _ptr(a_src), _ptr(a_dst), float(slope), _ptr(alpha_e), _ptr(alpha_s), _ptr(xs),
            _rows(xs, "xs"), _ptr(dout), _rows(dout, "dout"), hs, scale, int(heads), int(C_), g.N)
    if dalpha_e is None and dalpha_s is None:
        _abi.call("dc_gat_bwd_edge_heads", *args, _ptr(dz_e), _ptr(dz_s), _ptr(da_dst), _stream())
        return dz_e, dz_s, da_dst
    for t, rows, name in ((dalpha_e, max(g.E, 1), "dalpha_e"), (dalpha_s, g.N, "dalpha_s")):
        if t is not None:
            _need(t, _f32, name)
            if tuple(t.shape) != (rows, heads) or not t.is_contiguous():
                raise _abi.DcError(f"{name}: expected a contiguous [{rows}, {heads}] tensor, got {tuple(t.shape)}")
    _abi.call("dc_gat_bwd_edge_heads_ext", *args, _ptr(dalpha_e), _ptr(dalpha_s), _ptr(dz_e), _ptr(dz_s), _ptr(da_dst), _stream())
    return dz_e, dz_s, da_dst


def gat_scatter_heads(g, alpha_e, alpha_s, dz_e, dz_s, da_dst, att_src, att_dst, dout, heads, C_, concat):
    """-> (dxs [N, H*C], da_src [N, H]) over the by-source structure; see dc_gat_scatter_heads."""
    hs, scale = _dout_heads(heads, C_, concat)
    rpt, nbt, eidt = g.t
    att_src, att_dst = att_src.contiguous(), att_dst.contiguous()
    dxs = torch.empty((g.N, heads * C_), dtype=_f32, device=dout.device)
    da_src = torch.empty((g.N, heads), dtype=_f32, device=dout.device)
    _abi.call("dc_gat_scatter_heads", _ptr(rpt), _ptr(nbt), _ptr(eidt), _ptr(alpha_e), _ptr(alpha_s), _ptr(dz_e), _ptr(dz_s),
              _ptr(da_dst), _ptr(att_src), _ptr(att_dst), _ptr(dout), _rows(dout, "dout"), hs, scale, int(heads), int(C_), g.N,
              _ptr(dxs), _rows(dxs, "dxs"), _ptr(da_src), _stream())
    return dxs, da_src


def gat_att_grad(xs, da_src, da_dst, heads, C_):
    """-> (datt_src [H*C], datt_dst [H*C]); see dc_gat_att_grad."""
    N = xs.shape[0]
    datt_src = torch.empty(heads * C_, dtype=_f32, device=xs.device)
    datt_dst = torch.empty(heads * C_, dtype=_f32, device=xs.device)
    nb = _abi.lib().dc_gat_att_grad_workspace_bytes(N, heads, C_)
    ws = _workspace(nb, xs.device)
    _abi.call("dc_gat_att_grad", _ptr(xs), _rows(xs, "xs"), _ptr(da_src), _ptr(da_dst), N, int(heads), int(C_), _ptr(datt_src),
              _ptr(datt_dst), _ptr(ws), nb, _stream())
    return datt_src, datt_dst
