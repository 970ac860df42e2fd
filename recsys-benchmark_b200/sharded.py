"""Row-sharded embedding tables over the GPUs of one box (SURVEY.md section 8e).

The reference is single-device; this is the scale-out of its ONE concatenated table
(`src/models/embeddings/base.py:53-57`, addressed by global row id, `src/models/deepfm.py:88`):
rank g owns rows r with r % G == g at local row r // G (block-cyclic: balances the very
uneven field sizes).  The batch is data parallel, dense parameters are replicated.

No index / row all-to-all is issued: shards live in CUDA-IPC-exported buffers and
  * the forward gather kernel reads peer rows directly over NVLink (rsb_lookup_fwd_sharded),
  * the backward sorts + pre-reduces this rank's lookups and adds each unique row's sum into
    the OWNER's dense shard gradient with 128-bit atomics over NVLink
    (rsb_segment_scatter_shards),
so the exchange is fused into the gather / scatter kernels.  Two stream-ordered NCCL
collectives per step provide the cross-rank ordering: the dense-gradient allreduce (all
pushes are complete once it returns) and a 1-element allreduce after the optimizer step
(shards updated and gradient buffers re-zeroed before anyone gathers again).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, List, Optional

import torch
import torch.distributed as dist
from torch import nn

from . import _lib as L
from . import functional as RF
from .dcn import DCN_Mix
from .deepfm import DeepFM
from .embeddings import IEmbedding, OptEmbed, RetrainOptEmbed
from .linalg import run_sequential


# ------------------------------------------------------------------ host-side shard math ---
def shard_rows(num_rows: int, world: int) -> int:
    """Rows per shard (uniform; the last rows of some shards may be padding)."""
    return (num_rows + world - 1) // world


def owner_of(row, world: int):
    return row % world


def local_row(row, world: int):
    return row // world


def shard_of_full(full: torch.Tensor, rank: int, world: int) -> torch.Tensor:
    """Rows of `full` owned by `rank`, padded with zeros to shard_rows()."""
    n = shard_rows(full.shape[0], world)
    out = torch.zeros((n,) + tuple(full.shape[1:]), dtype=full.dtype, device=full.device)
    mine = full[rank::world]
    out[: mine.shape[0]] = mine
    return out


def full_from_shards(shards: List[torch.Tensor], num_rows: int) -> torch.Tensor:
    world = len(shards)
    out = torch.empty((num_rows,) + tuple(shards[0].shape[1:]), dtype=shards[0].dtype, device=shards[0].device)
    for g, s in enumerate(shards):
        cnt = len(range(g, num_rows, world))
        out[g::world] = s[:cnt]
    return out


# Fields with at most this many ids are replicated on every rank instead of sharded (world > 1).  Criteo shape: 31 of
# the 39 fields (42 644 of 1 086 810 rows, 2.7 MB) - they serve 31 of a sample's 39 lookups, so the rows crossing NVLink
# drop from 39 * (G-1)/G to 8 * (G-1)/G per sample; their [H, D] gradient rides the replicated-gradient allreduce.
HOT_FIELD_ROWS = int(os.environ.get("RSB_HOT_FIELD_ROWS", "16384"))


def hot_field_map(field_dims, hot_field_rows: int):
    """-> (int64 [F, 3] rows (lo, hi, delta), H).  lo = the field's offset in the concatenated table; a replicated
    ("hot") field has hi = lo + dim and lives at rows [lo + delta, hi + delta) of the [H, D] replica; hi == lo marks
    a sharded field.  The layout rsb_lookup_fwd_sharded / rsb_segment_scatter_shards take."""
    rows, off, base = [], 0, 0
    for d in field_dims:
        d = int(d)
        hot = d <= hot_field_rows
        rows.append((off, off + d if hot else off, base - off if hot else 0))
        base += d if hot else 0
        off += d
    return torch.tensor(rows, dtype=torch.int64).reshape(-1, 3), base


def hot_global_rows(hot_map: torch.Tensor) -> torch.Tensor:
    """Global row ids of the replica's rows, in replica order."""
    parts = [torch.arange(int(lo), int(hi), dtype=torch.int64) for lo, hi, _ in hot_map.tolist() if hi > lo]
    return torch.cat(parts) if parts else torch.empty(0, dtype=torch.int64)


def allreduce_mean_(grads: List[torch.Tensor], group=None) -> None:
    """Average a list of gradient tensors over the ranks with ONE flat allreduce (in place)."""
    if not grads or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    world = dist.get_world_size(group)
    flat = torch.cat([g.reshape(-1) for g in grads])
    if dist.get_backend(group) == "nccl":
        dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=group)      # the mean inside the collective: one launch fewer
    else:
        dist.all_reduce(flat, group=group)
        flat.div_(world)
    views, off = [], 0
    for g in grads:
        views.append(flat[off:off + g.numel()].view_as(g))
        off += g.numel()
    torch._foreach_copy_(grads, views)


# ------------------------------------------------------------------ IPC buffers ---
class SharedBuffer:
    """cudaMalloc'ed, zero-filled, CUDA-IPC-exportable fp32 buffer viewed as a torch tensor."""

    def __init__(self, shape, device: torch.device):
        lib = L.load()
        self.shape = tuple(int(s) for s in shape)
        self.device = device
        nbytes = 4 * max(1, math.prod(self.shape))
        p = C.c_void_p()
        with torch.cuda.device(device):
            L.check(lib.rsb_shared_alloc(nbytes, C.byref(p)), "shared_alloc")
        self.ptr = int(p.value)
        self.__cuda_array_interface__ = {"shape": self.shape, "typestr": "<f4", "data": (self.ptr, False),
                                         "version": 3, "strides": None}
        self.tensor = torch.as_tensor(self, device=device)

    def handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        with torch.cuda.device(self.device):
            L.check(L.load().rsb_ipc_get_handle(self.ptr, buf), "ipc_get_handle")
        return buf.raw

    def free(self):
        """cudaFree the buffer.  `self.tensor` (and every view of it) dangles afterwards: drop them first."""
        if self.ptr:
            with torch.cuda.device(self.device):
                L.check(L.load().rsb_shared_free(self.ptr), "shared_free")
            self.ptr = 0
            self.tensor = None


def _open(handle: bytes, device) -> int:
    p = C.c_void_p()
    with torch.cuda.device(device):
        L.check(L.load().rsb_ipc_open_handle(handle, C.byref(p)), "ipc_open_handle")
    return int(p.value)


class ShardGroup:
    """The per-rank buffers (table shard and its gradient accumulator; optionally a per-row aux array - PEP thresholds
    or a retrain mask - and its gradient accumulator; optionally an `eval` shard [n_local, dim] - OptEmbed's cached
    masked table) and the device-resident pointer tables to every rank's copy."""

    def __init__(self, num_rows: int, dim: int, device: torch.device, group=None, aux_cols: int = 0,
                 aux_is_mask: bool = False, aux_grad: bool = False, eval_table: bool = False):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.num_rows, self.dim, self.device = num_rows, dim, device
        self.n_local = shard_rows(num_rows, self.world)
        self.buf: Dict[str, SharedBuffer] = {
            "table": SharedBuffer((self.n_local, dim), device),
            "table_grad": SharedBuffer((self.n_local, dim), device)}
        self.aux_cols, self.aux_is_mask = int(aux_cols), bool(aux_is_mask)
        if aux_cols:
            # a bool mask [n_local, cols] is stored in a float-typed IPC buffer and viewed as bytes
            shape = ((self.n_local * aux_cols + 3) // 4,) if aux_is_mask else (self.n_local, aux_cols)
            self.buf["aux"] = SharedBuffer(shape, device)
            if aux_grad:
                self.buf["aux_grad"] = SharedBuffer((self.n_local, aux_cols), device)
        if eval_table:
            self.buf["eval"] = SharedBuffer((self.n_local, dim), device)
        names = tuple(self.buf)
        handles = {k: self.buf[k].handle() for k in names}
        if self.world > 1:
            gathered: List[Optional[dict]] = [None] * self.world
            dist.all_gather_object(gathered, handles, group=group)
        else:
            gathered = [handles]
        self.ptrs: Dict[str, torch.Tensor] = {}
        self._peer_maps: List[int] = []          # peer buffers mapped into this process (closed by close())
        for k in names:
            addr = [self.buf[k].ptr if g == self.rank else _open(gathered[g][k], device) for g in range(self.world)]
            self._peer_maps += [a for g, a in enumerate(addr) if g != self.rank]
            self.ptrs[k] = torch.tensor(addr, dtype=torch.int64, device=device)
        self._tick = torch.zeros(1, device=device)
        self.err_flag = torch.zeros(1, dtype=torch.int32, device=device)   # set by the gather on an out-of-range id

    def aux_tensor(self) -> Optional[torch.Tensor]:
        """This rank's shard of the per-row aux array: fp32 [n_local, cols], or bool [n_local, cols] for a mask."""
        if "aux" not in self.buf:
            return None
        t = self.buf["aux"].tensor
        if self.aux_is_mask:
            return t.view(torch.uint8)[: self.n_local * self.aux_cols].view(self.n_local, self.aux_cols).view(torch.bool)
        return t

    def barrier(self):
        """Stream-ordered cross-rank ordering point (a 1-element allreduce, no host sync)."""
        if self.world > 1:
            dist.all_reduce(self._tick, group=self.group)

    def close(self):
        """Release the shards: every rank first unmaps its peers' buffers, then (after a barrier: nobody may still
        have a buffer mapped when its owner frees it) frees its own.  Collective; the module that owned the shards
        must not be used afterwards (its parameters pointed into the freed buffers).  Not called implicitly - the
        buffers live as long as the process otherwise, like the reference's parameters."""
        torch.cuda.synchronize(self.device)
        lib = L.load()
        with torch.cuda.device(self.device):
            for a in self._peer_maps:
                L.check(lib.rsb_ipc_close_handle(a), "ipc_close_handle")
        self._peer_maps = []
        if self.world > 1:
            dist.barrier(group=self.group)
        for b in self.buf.values():
            b.free()
        self.ptrs = {}

    def zero_grads(self):
        self.buf["table_grad"].tensor.zero_()
        if "aux_grad" in self.buf:
            self.buf["aux_grad"].tensor.zero_()


# ------------------------------------------------------------------ differentiable op ---
class _ShardedLookup(torch.autograd.Function):
    """(x, offsets, fc, bias; shard group) -> emb [B,F,D], y_fm [B].  The table-shard gradients are not
    returned to autograd: they are accumulated (pre-scaled by 1/G) in the owners' buffers.  The first-order
    weights `fc` [N,1] are REPLICATED (4 B per row: peer reads / NVLink atomics of that size cost as many
    transactions as the 64-byte rows - at N=8 the sharded first-order gradient alone took 0.76 ms of a 5.0 ms
    step); their dense gradient goes back to autograd and is averaged with the other replicated gradients."""

    @staticmethod
    def forward(ctx, sg: ShardGroup, x, offsets, fc, bias, use_fm: bool, presort: bool = False, hot=None,
                hot_map=None, amax_slots=None, table=None):
        # `table` (this rank's shard parameter) is an input only so that autograd runs the backward when nothing else
        # requires a gradient (DCN-Mix: no first-order weights, world 1: no replica); its gradient is never returned
        lib = L.load()
        dev = L.require_cuda(x, offsets, bias)
        x = x.contiguous()
        b, f = x.shape
        d = sg.dim
        emb = torch.empty(b, f, d, dtype=torch.float32, device=dev)
        y = torch.empty(b, dtype=torch.float32, device=dev) if use_fm else None
        s = torch.empty(b, d, dtype=torch.float32, device=dev) if use_fm else None
        rows = torch.empty(b, f, dtype=torch.int64, device=dev)
        if hot is not None and hot_map.shape[0] != f:
            raise ValueError(f"replicated small fields need one id column per field: x has {f} columns, the table "
                             f"{hot_map.shape[0]} fields")
        nbytes = b * (f * x.element_size() + 2 * f * d * 4 + f * 8 + (f * 4 + 4 + d * 4 if use_fm else 0))
        if sg.world == 1 and hot is None:
            # one shard IS the table: the single-table entry point (no owner arithmetic, no pointer-table load in front
            # of every row load: 0.69 -> 0.77 of the copy peak on the headline gather)
            RF._call("lookup_fwd_sharded", lib.rsb_lookup_fwd, L.KIND_VANILLA, L.ptr(x), int(x.dtype == torch.int32),
                     L.ptr(offsets), b, f, d, L.ptr(sg.buf["table"].tensor), sg.num_rows, sg.num_rows, None, 0, None, 0,
                     None, L.ptr(fc) if use_fm else None, L.ptr(bias) if use_fm else None, L.ptr(emb), L.ptr(y), L.ptr(s),
                     L.ptr(rows), L.ptr(sg.err_flag), L.ptr(amax_slots), L.stream_ptr(dev), nbytes=nbytes)
        else:
            RF._call("lookup_fwd_sharded", lib.rsb_lookup_fwd_sharded, L.ptr(x), int(x.dtype == torch.int32),
                     L.ptr(offsets), b, f, d, L.ptr(sg.ptrs["table"]), L.ptr(fc) if use_fm else None,
                     sg.world, sg.num_rows, L.ptr(bias) if use_fm else None, L.ptr(hot) if hot is not None else None,
                     L.ptr(hot_map) if hot is not None else None, L.ptr(emb), L.ptr(y), L.ptr(s), L.ptr(rows),
                     L.ptr(sg.err_flag), L.ptr(amax_slots), L.stream_ptr(dev), nbytes=nbytes)
        ctx.sg, ctx.use_fm, ctx.shape = sg, use_fm, (b, f)
        ctx.hot_map = hot_map if hot is not None else None
        ctx.hot_shape = tuple(hot.shape) if hot is not None else None
        ctx.fc_shape = tuple(fc.shape) if fc is not None else None
        ctx.fc_param = fc
        # the backward's row sort needs only `rows`: queued on the side stream now, consumed at the end of backward
        ctx.presorted = RF.early_sort(rows, sg.num_rows) if presort else None
        ctx.save_for_backward(rows, emb, s)
        ctx.mark_non_differentiable(rows)
        return emb, (y if use_fm else emb.new_empty(0)), rows

    @staticmethod
    def backward(ctx, g_emb, g_y, _g_rows):
        lib = L.load()
        sg: ShardGroup = ctx.sg
        rows, emb, s = ctx.saved_tensors
        b, f = ctx.shape
        d = sg.dim
        n = b * f
        dev = rows.device
        use_gy = ctx.use_fm and g_y is not None and g_y.numel() == b
        g_emb = g_emb.contiguous() if g_emb is not None else None
        if use_gy:
            g_y = g_y.contiguous()
            rg = torch.empty(n, d, dtype=torch.float32, device=dev)
            RF._call("lookup_bwd_rows", lib.rsb_lookup_bwd_rows, L.KIND_VANILLA, L.ptr(rows), b, f, d, L.ptr(emb),
                     sg.num_rows, None, 0, None, 0, None, L.ptr(emb), L.ptr(s), L.ptr(g_y), L.ptr(g_emb), L.ptr(rg),
                     None, None, L.stream_ptr(dev), nbytes=b * (f * 8 + 3 * f * d * 4 + d * 4 + 4))
        else:
            rg = g_emb.view(n, d)
        pre, ctx.presorted = ctx.presorted, None
        skeys, perm = pre.get() if pre is not None else RF.sort_rows(rows, sg.num_rows)
        scale = 1.0 / sg.world
        g_bias = g_fc = None
        if use_gy and ctx.needs_input_grad[3]:
            # beside the pushes, on its own stream (same sorted lookups, independent output)
            g_fc = RF.fc_grad_beside(ctx.fc_param, rows, g_y, b, f, ctx.fc_shape, sg.num_rows, (skeys, perm))
        ws = RF._ws(lib.rsb_segment_workspace_bytes(n, d), dev)
        g_hot = None
        if ctx.hot_map is not None:
            # dense local gradient of the replicated rows (averaged over the ranks with the other replicated grads)
            g_hot = torch.zeros(ctx.hot_shape, dtype=torch.float32, device=dev)
        RF._call("segment_scatter_shards", lib.rsb_segment_scatter_shards, L.ptr(skeys), L.ptr(perm), n, L.ptr(rg), d,
                 L.ptr(sg.ptrs["table_grad"]), sg.world, scale,
                 L.ptr(ctx.hot_map) if g_hot is not None else None, f, L.ptr(g_hot) if g_hot is not None else None,
                 L.ptr(ws), ws.numel(), L.stream_ptr(dev), nbytes=n * (8 + 4 * d))
        if use_gy:
            g_bias = g_y.sum().reshape(1)
        return None, None, None, g_fc, g_bias, None, None, g_hot, None, None, None


# ------------------------------------------------------------------ modules ---
class ShardedVanillaEmbedding(IEmbedding):
    """VanillaEmbedding (base.py:23-75) whose table is row-sharded over the process group.
    `_emb_module.weight` is THIS rank's shard [ceil(N/G), D]; use `load_full_weight` /
    `gather_full_weight` to convert from / to the reference's full-table state dict."""

    def __init__(self, field_dims, hidden_size: int, mode=None, initializer="xavier", device=None, group=None,
                 hot_field_rows: Optional[int] = None, **kwargs):
        """hot_field_rows: fields of at most this many ids are replicated (`_emb_module.hot` [H, D], a plain
        replicated parameter) instead of sharded; default HOT_FIELD_ROWS when world > 1, nothing at world 1."""
        super().__init__()
        assert mode is None, "sharded tables serve the [B,F,D] lookup only"
        field_dims = [field_dims] if isinstance(field_dims, int) else [int(v) for v in field_dims]
        self._num_item = sum(field_dims)
        self._hidden_size = hidden_size
        device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.shards = ShardGroup(self._num_item, hidden_size, device, group)
        self._emb_module = nn.Module()
        self._emb_module.weight = nn.Parameter(self.shards.buf["table"].tensor)
        if hot_field_rows is None:
            hot_field_rows = HOT_FIELD_ROWS if self.shards.world > 1 else 0
        hot_map, n_hot = hot_field_map(field_dims, int(hot_field_rows))
        self.hot_map = hot_map.to(device) if n_hot > 0 else None
        self._hot_rows = hot_global_rows(hot_map).to(device) if n_hot > 0 else None
        if n_hot > 0:
            self._emb_module.hot = nn.Parameter(torch.zeros(n_hot, hidden_size, dtype=torch.float32, device=device))
        self._init_shard(initializer)

    INIT_CHUNK_ROWS = 1 << 20

    @torch.no_grad()
    def _init_shard(self, initializer: str):
        """i.i.d. init of the FULL table (base.py:62-67: xavier_uniform_ / normal_(std=0.1)), of which this rank keeps
        its rows: every rank draws the same global row blocks from the device generator (same seed on every rank, as
        the replicated parameters already require) and copies out rows r with r % G == rank.  The gathered table is
        the same for every world size, and no two global rows share values (drawing the local shard directly from
        the same seed would give rows kG..kG+G-1 identical vectors)."""
        sg = self.shards
        n, d, g = self._num_item, self._hidden_size, sg.world
        a = math.sqrt(6.0 / (n + d))            # xavier_uniform_ bound of the FULL [N, D] table
        w = self._emb_module.weight
        w.zero_()
        for lo in range(0, n, self.INIT_CHUNK_ROWS):
            hi = min(n, lo + self.INIT_CHUNK_ROWS)
            blk = torch.empty(hi - lo, d, dtype=torch.float32, device=sg.device)
            if initializer == "xavier":
                blk.uniform_(-a, a)
            else:
                blk.normal_(std=0.1)
            first = lo + ((sg.rank - lo) % g)   # first global row >= lo owned by this rank
            if first < hi:
                mine = blk[first - lo::g]
                w[first // g: first // g + mine.shape[0]].copy_(mine)
            if self._hot_rows is not None:
                sel = (self._hot_rows >= lo) & (self._hot_rows < hi)
                if bool(sel.any()):
                    self._emb_module.hot[sel] = blk[self._hot_rows[sel] - lo]

    def get_weight(self):
        return self.gather_full_weight()

    def load_full_weight(self, full: torch.Tensor):
        sg = self.shards
        with torch.no_grad():
            full = full.to(sg.device)
            self._emb_module.weight.copy_(shard_of_full(full, sg.rank, sg.world))
            if self._hot_rows is not None:
                self._emb_module.hot.copy_(full[self._hot_rows])

    def gather_full_weight(self) -> torch.Tensor:
        sg = self.shards
        local = self._emb_module.weight.detach()
        if sg.world == 1:
            full = local[: self._num_item].clone()
        else:
            parts = [torch.empty_like(local) for _ in range(sg.world)]
            dist.all_gather(parts, local.contiguous(), group=sg.group)
            full = full_from_shards(parts, self._num_item)
        if self._hot_rows is not None:
            full[self._hot_rows] = self._emb_module.hot.detach()   # the owners' copies of replicated rows are stale
        return full

    def lookup(self, x, offsets=None, fc=None, bias=None):
        if offsets is not None:
            offsets = offsets.reshape(-1).long()
        use_fm = fc is not None
        self._rsb_err_flag = self.shards.err_flag     # read by IEmbedding.train() / validate=True like the others
        presort = RF.EARLY_SORT and torch.is_grad_enabled()
        hot = getattr(self._emb_module, "hot", None)
        slots = RF.amax_slots_for(x.device)
        emb, y, _ = _ShardedLookup.apply(self.shards, x, offsets, fc, bias, use_fm, presort, hot, self.hot_map, slots,
                                         self._emb_module.weight)
        if slots is not None:
            emb._rsb_amax_slots = slots
        if self.validate:
            RF.check_index_errors(self)
        return emb, (y if use_fm else None)


# ------------------------------------------------------------------ any variant, sharded ---
_PER_ROW_PEP = (L.PEP_FEATURE, L.PEP_FEATURE_DIM)


class _ShardedKindLookup(torch.autograd.Function):
    """_ShardedLookup for the lightweight variants (SURVEY 8e): the MAIN table (PEP / masked weight, QR emb2) and the
    per-row aux array (PEP `s` of the feature / feature_dim kinds, retrain masks) are read from the owners' shards inside
    the gather and inside the backward's chain-rule kernel; their gradients are pre-reduced per unique row and pushed
    into the owners' accumulators.  Small parameters (QR emb1, PEP global / dimension thresholds, OptEmbed's per-field
    thresholds `t`, fc, bias) are replicated: their gradients go back to autograd and are averaged with the other
    replicated gradients.  `mask_d` (OptEmbed) is the [B, F] int64 mask-D draw of this rank's lookups.
    `table` (this rank's shard) is an input only so that autograd runs the backward; its gradient is never returned."""

    @staticmethod
    def forward(ctx, sg: ShardGroup, spec, x, offsets, table, table1, aux_rep, fc, bias, presort, amax_slots,
                mask_d=None):
        lib = L.load()
        dev = L.require_cuda(x, offsets, table, table1, aux_rep, fc, bias, mask_d)
        x = x.contiguous()
        b, f = x.shape
        e = spec.row_width
        use_fm = fc is not None
        emb = torch.empty(b, f, e, dtype=torch.float32, device=dev)
        y = torch.empty(b, dtype=torch.float32, device=dev) if use_fm else None
        s = torch.empty(b, e, dtype=torch.float32, device=dev) if use_fm else None
        rows = torch.empty(b, f, dtype=torch.int64, device=dev)
        aux_sh = sg.ptrs.get("aux")
        md_bytes = RF._aux_row_bytes(spec, f, mask_d) if mask_d is not None else 0
        nbytes = b * (f * x.element_size() + 2 * f * e * 4 + f * 8 + md_bytes + (f * 4 + 4 + e * 4 if use_fm else 0))
        RF._call("lookup_fwd_sharded", lib.rsb_lookup_fwd_sharded_kind, spec.kind, L.ptr(x), int(x.dtype == torch.int32),
                 L.ptr(offsets), b, f, spec.dim, L.ptr(sg.ptrs["table"]), sg.world, sg.num_rows, spec.num_global,
                 L.ptr(table1), spec.divider, L.ptr(aux_rep), L.ptr(aux_sh), spec.aux_mode, L.ptr(mask_d),
                 L.ptr(fc) if use_fm else None, L.ptr(bias) if use_fm else None, L.ptr(emb), L.ptr(y), L.ptr(s),
                 L.ptr(rows), L.ptr(sg.err_flag), L.ptr(amax_slots), L.stream_ptr(dev), nbytes=nbytes)
        ctx.sg, ctx.spec, ctx.use_fm, ctx.shape = sg, spec, use_fm, (b, f)
        ctx.fc_shape = tuple(fc.shape) if fc is not None else None
        ctx.presorted = RF.early_sort(rows, sg.num_rows, key_div=spec.divider if spec.is_qr else 0) if presort else None
        ctx.save_for_backward(rows, emb, s, table1, aux_rep, mask_d)
        ctx.mark_non_differentiable(rows)
        return emb, (y if use_fm else emb.new_empty(0)), rows

    @staticmethod
    def backward(ctx, g_emb, g_y, _g_rows):
        lib = L.load()
        sg: ShardGroup = ctx.sg
        spec = ctx.spec
        rows, emb, s, table1, aux_rep, mask_d = ctx.saved_tensors
        b, f = ctx.shape
        e = spec.row_width
        n = b * f
        dev = rows.device
        kind = spec.kind
        # (sg, spec, x, offsets, table, table1, aux_rep, fc, bias, presort, amax_slots, mask_d)
        need = ctx.needs_input_grad
        use_gy = ctx.use_fm and g_y is not None and g_y.numel() == b
        g_emb = g_emb.contiguous() if g_emb is not None else None
        g_y = g_y.contiguous() if use_gy else None
        aux_sh = sg.ptrs.get("aux")
        per_row_s = kind == L.KIND_PEP and spec.aux_mode in _PER_ROW_PEP and "aux_grad" in sg.buf
        # ---- stage 1: per-lookup row gradients (the chain rule re-reads the rows from their owners) ----
        rg_aux = None
        if kind == L.KIND_VANILLA and not use_gy:
            rg_main = g_emb.view(n, e)
        else:
            rg_main = torch.empty(n, e, dtype=torch.float32, device=dev)
            if kind == L.KIND_QR_MULT or (kind == L.KIND_PEP and (per_row_s or need[6])):
                rg_aux = torch.empty(n, e, dtype=torch.float32, device=dev)
            elif kind == L.KIND_OPTEMBED and aux_rep is not None and need[6]:
                rg_aux = torch.empty(b, f, dtype=torch.float32, device=dev)     # one g_z per lookup
            n_out = 2 if (rg_aux is not None and kind != L.KIND_OPTEMBED) else 1
            md_bytes = RF._aux_row_bytes(spec, f, mask_d) if mask_d is not None else 0
            nbytes = b * (f * 8 + f * e * 4 * (1 + int(use_gy)) + n_out * f * e * 4 + md_bytes
                          + (e * 4 + 4 if use_gy else 0))
            RF._call("lookup_bwd_rows", lib.rsb_lookup_bwd_rows_sharded, kind, L.ptr(rows), b, f, spec.dim,
                     L.ptr(sg.ptrs["table"]), sg.world, sg.num_rows, L.ptr(table1), spec.divider, L.ptr(aux_rep),
                     L.ptr(aux_sh), spec.aux_mode, L.ptr(mask_d), L.ptr(emb), L.ptr(s), L.ptr(g_y), L.ptr(g_emb),
                     L.ptr(rg_main), L.ptr(rg_aux), L.stream_ptr(dev), nbytes=nbytes)
            if kind == L.KIND_QR_ADD:
                rg_aux = rg_main
        # ---- stage 2: sorted, pre-reduced per unique row, pushed to the owner ----
        pre, ctx.presorted = ctx.presorted, None
        skeys, perm = pre.get() if pre is not None else RF.sort_rows(rows, sg.num_rows,
                                                                     key_div=spec.divider if spec.is_qr else 0)
        scale = 1.0 / sg.world

        def push(rg, width, target):
            ws = RF._ws(lib.rsb_segment_workspace_bytes(n, width), dev)
            RF._call("segment_scatter_shards", lib.rsb_segment_scatter_shards, L.ptr(skeys), L.ptr(perm), n, L.ptr(rg),
                     width, L.ptr(sg.ptrs[target]), sg.world, scale, None, f, None, L.ptr(ws), ws.numel(),
                     L.stream_ptr(dev), nbytes=n * (8 + 4 * width))

        push(rg_main, e, "table_grad")
        g_table1 = g_aux = g_fc = g_bias = None
        if per_row_s:
            if spec.aux_mode == L.PEP_FEATURE_DIM:
                push(rg_aux, e, "aux_grad")
            else:
                push(rg_aux.sum(dim=1, keepdim=True).contiguous(), 1, "aux_grad")
        elif kind == L.KIND_PEP and need[6]:
            g_aux = rg_aux.sum(dim=0) if spec.aux_mode == L.PEP_DIMENSION else rg_aux.sum().reshape(1)
        elif kind == L.KIND_OPTEMBED and rg_aux is not None:
            g_aux = -rg_aux.sum(dim=0)               # as the single-device backward: g_t[f] = -sum_b g_z[b, f]
        if spec.is_qr and need[5]:
            g_table1 = (RF.small_table_grad(rows, rg_aux, table1.shape[0], key_mod=spec.divider)
                        if (not RF.DETERMINISTIC or table1.shape[0] <= 32) else None)
            if g_table1 is None:
                g_table1 = RF.dense_row_grad(rows, rg_aux, table1.shape[0], key_mod=spec.divider)
        if use_gy:
            if need[7]:
                g_fc = RF.fc_grad(rows, g_y, b, f, ctx.fc_shape, spec.num_global, None if spec.is_qr else (skeys, perm))
            g_bias = g_y.sum().reshape(1)
        return None, None, None, None, None, g_table1, g_aux, g_fc, g_bias, None, None, None


def _kernel_tensors(inner: IEmbedding):
    """(main table, QR emb1, aux) as the module holds them.  The OptEmbed kinds' own _tensors() returns other things:
    the supernet its eval cache outside training, the retrain module a uint8 copy of its mask (or an AssertionError
    before init_mask); here they are the weight and `t` Parameters, resp. the weight and the `_mask` Parameter (None
    before init_mask)."""
    if isinstance(inner, OptEmbed):
        return inner._weight, None, inner._t_param()
    if isinstance(inner, RetrainOptEmbed):
        return inner._weight, None, inner._mask
    return inner._tensors()


class ShardedEmbedding(IEmbedding):
    """Any of the per-row variants with its big arrays row-sharded over the process group (SURVEY 8e):
    QRHashingEmbedding mult / add (emb2 sharded, the <= divider-row emb1 replicated), PepEmbeeding (emb.weight sharded;
    `s` sharded for the feature / feature_dim threshold types, replicated for global / dimension), the OptEmbed
    supernet (`_weight` sharded, the per-field thresholds `t` replicated, mask-D drawn per lookup), RetrainPepEmbedding
    and RetrainOptEmbed (weight and bool mask sharded).

    Built FROM the single-device module (`inner`, constructed the usual way - same seed on every rank - so its
    initialisation, kwargs and methods are the reference's): its big tensors are copied into this rank's IPC shard
    buffers and the module's own Parameters are re-pointed at them, so parameter names stay the reference's while
    their leading dimension becomes ceil(rows / G).  `load_full_state_dict` / `full_state_dict` convert from / to the
    reference's single-device state dict.

    OptEmbed in eval mode gathers, like the reference, from a cached masked table: here one `eval` shard per rank,
    rebuilt by every rank at the same point (a collective, between two barriers: nobody overwrites its shard while a
    peer still reads it, and nobody gathers before every shard is rebuilt).  A training forward invalidates it."""

    KINDS = (L.KIND_QR_MULT, L.KIND_QR_ADD, L.KIND_PEP, L.KIND_MASK, L.KIND_OPTEMBED)

    def __init__(self, inner: IEmbedding, group=None, device=None):
        super().__init__()
        spec = inner._spec()
        if spec.kind not in self.KINDS:
            raise NotImplementedError("row sharding covers vanilla (ShardedVanillaEmbedding), QR mult / add, PEP, "
                                      "OptEmbed and masked-retrain tables")
        if inner._mode is not None or spec.sparse_grad or spec.modulus:
            raise NotImplementedError("sharded tables serve the dense-gradient [B,F,D] lookup only")
        if isinstance(inner, OptEmbed) and inner._t_param() is not None and inner._mask_e_module.mode_threshold_e != "field":
            raise NotImplementedError("sharded OptEmbed takes its mask-E thresholds per field (mode_threshold_e='field')")
        device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        inner = inner.to(device)
        table, _table1, aux = _kernel_tensors(inner)
        per_row = spec.kind == L.KIND_MASK or (spec.kind == L.KIND_PEP and spec.aux_mode in _PER_ROW_PEP)
        aux_cols = (int(table.shape[1]) if spec.kind == L.KIND_MASK else int(aux.shape[1])) if per_row else 0
        self.shards = ShardGroup(table.shape[0], table.shape[1], device, group, aux_cols=aux_cols,
                                 aux_is_mask=spec.kind == L.KIND_MASK, aux_grad=per_row and spec.kind == L.KIND_PEP,
                                 eval_table=spec.kind == L.KIND_OPTEMBED)
        self._per_row_aux = per_row
        self._full_rows = int(table.shape[0])
        self.inner = inner
        sg = self.shards
        with torch.no_grad():
            sg.buf["table"].tensor.copy_(shard_of_full(table.detach(), sg.rank, sg.world))
            table.data = sg.buf["table"].tensor
            if isinstance(inner, RetrainOptEmbed):
                if aux is not None:
                    self._install_mask(aux.detach())
            elif per_row:
                sg.aux_tensor().copy_(shard_of_full(aux.detach(), sg.rank, sg.world))
                aux.data = sg.aux_tensor()
        if hasattr(inner, "_nnz") and torch.is_tensor(inner._nnz):
            inner._nnz = inner._nnz.to(device)
        if isinstance(inner, OptEmbed):
            # the reference's eval cache: "fresh" (an empty table: eval() before any training or get_weight raises,
            # as F.embedding does), "stale" (rebuilt on the next eval lookup) or "ready"
            cur = inner._cur_weight
            self._eval_state = "fresh" if cur is not None and cur.numel() == 0 else "stale"
            inner._cur_weight = None if self._eval_state == "stale" else cur

    # -- what the step protocol of the sharded models needs -------------------------------
    def shard_params(self) -> List[torch.nn.Parameter]:
        table, _t1, aux = _kernel_tensors(self.inner)
        out = [table]
        if self._per_row_aux and aux is not None and aux.requires_grad:
            out.append(aux)
        return out

    def expose_shard_grads(self, on: bool):
        table, _t1, aux = _kernel_tensors(self.inner)
        table.grad = self.shards.buf["table_grad"].tensor if on else None
        if "aux_grad" in self.shards.buf:
            aux.grad = self.shards.buf["aux_grad"].tensor if on else None

    # -- conversion from / to the reference's single-device tensors --------------------------
    def _names(self):
        """{state-dict key: sharded?} over the module's persistent state (the reference's keys; OptEmbed's
        non-persistent `_cur_weight` is not part of it)."""
        table, _t1, aux = _kernel_tensors(self.inner)
        big = {id(table)}
        if self._per_row_aux and aux is not None:
            big.add(id(aux))
        return {n: id(t) in big for n, t in self.inner.state_dict(keep_vars=True).items()}

    def _gather_full(self, local: torch.Tensor, num_rows: int) -> torch.Tensor:
        """The full array of which every rank holds `local` (its rows, padded): an all-gather at world > 1."""
        sg = self.shards
        as_bytes = local.dtype == torch.bool
        local = (local.view(torch.uint8) if as_bytes else local).contiguous()
        if sg.world == 1:
            parts = [local]
        else:
            parts = [torch.empty_like(local) for _ in range(sg.world)]
            dist.all_gather(parts, local, group=sg.group)
        full = full_from_shards(parts, num_rows)
        return full.view(torch.bool) if as_bytes else full

    def _all_sum(self, count: torch.Tensor) -> int:
        """A device int64 count summed over the ranks."""
        sg = self.shards
        if sg.world > 1:
            dist.all_reduce(count, group=sg.group)
        return int(count.item())

    @torch.no_grad()
    def _install_mask(self, full: torch.Tensor):
        """Keep this rank's rows of a full [N, D] retrain mask (any dtype, non-zero = kept) in the aux shard and point
        the module's `_mask` at that shard; no full copy stays alive.  full_state_dict gives the mask back in `full`'s
        dtype (RetrainOptEmbed.init_mask makes an int64 mask)."""
        sg, inner = self.shards, self.inner
        self._mask_dtype = full.dtype
        m = sg.aux_tensor()
        mine = full.to(sg.device)[sg.rank::sg.world]
        m[: mine.shape[0]].copy_(mine != 0)
        m[mine.shape[0]:] = False
        inner._mask = nn.Parameter(m, requires_grad=False)
        inner._cur_weight = None

    def init_mask(self, mask_e: torch.Tensor, mask_d: torch.Tensor):
        """RetrainOptEmbed.init_mask (deepfm_opt_embed.py:660-672) over the shards: the module builds the reference
        mask, this rank keeps its rows.  Returns this rank's shard of the mask ([ceil(N / G), D] bool)."""
        inner = self.inner
        if not isinstance(inner, RetrainOptEmbed):
            raise AttributeError(f"'{type(inner).__name__}' has no init_mask")
        full = inner.init_mask(mask_e, mask_d)
        self._install_mask(full.detach())
        del full
        return inner._mask

    @torch.no_grad()
    def load_full_state_dict(self, state: Dict[str, torch.Tensor]):
        sg, inner = self.shards, self.inner
        if isinstance(inner, RetrainOptEmbed) and inner._mask is None and "_mask" in state:
            self._install_mask(state["_mask"])
        mine = dict(list(inner.named_parameters()) + list(inner.named_buffers()))
        for name, sharded in self._names().items():
            src = state[name].to(sg.device)
            mine[name].copy_(shard_of_full(src, sg.rank, sg.world) if sharded else src)
        if isinstance(inner, OptEmbed) and self._eval_state == "ready":
            self._eval_state = "stale"

    @torch.no_grad()
    def full_state_dict(self) -> Dict[str, torch.Tensor]:
        inner = self.inner
        out = {}
        mine = dict(list(inner.named_parameters()) + list(inner.named_buffers()))
        for name, sharded in self._names().items():
            t = mine[name].detach()
            if not sharded:
                out[name] = t.clone()
            else:
                full = self._gather_full(t, self._full_rows)
                out[name] = full.to(self._mask_dtype) if isinstance(inner, RetrainOptEmbed) and name == "_mask" else full
        return out

    # -- OptEmbed: the eval cache over the shards ----------------------------------------------
    def _shard_rows(self, full_rows: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        """This rank's rows of a global per-row array (zero padding: a zero weight row yields a zero masked row)."""
        if full_rows is None:
            return None
        return shard_of_full(full_rows.to(self.shards.device), self.shards.rank, self.shards.world).contiguous()

    @torch.no_grad()
    def _rebuild_eval(self, mask_d: Optional[torch.Tensor]):
        """OptEmbed.get_weight(mask_d) into this rank's `eval` shard: every row through rsb_optembed_eval_weight, the
        kernel of the single-device cache, with the global per-row `t` and mask-D arrays sliced to this rank's rows.
        Collective: all ranks rebuild at the same point (as validate_epoch does)."""
        inner, sg = self.inner, self.shards
        rows_idx, bool_mask = inner._mask_d_rows(mask_d)
        t_sh = self._shard_rows(inner._t_rows())
        md_sh = self._shard_rows(rows_idx)
        out = sg.buf["eval"].tensor
        dev = sg.device
        sg.barrier()        # no peer still gathers from the shard about to be overwritten
        RF._call("optembed_eval_weight", L.load().rsb_optembed_eval_weight, L.ptr(inner._weight), L.ptr(t_sh),
                 L.ptr(md_sh), inner._norm, sg.n_local, sg.dim, L.ptr(out), None, L.stream_ptr(dev))
        if bool_mask is not None:
            out.mul_(self._shard_rows(bool_mask).to(out.dtype))
        sg.barrier()        # every shard rebuilt before any peer gathers from it
        self._eval_state = "ready"

    def _eval_lookup(self, x, offsets, fc, bias, mask_d):
        """OptEmbed.lookup outside training: the plain gather over the `eval` shards (rebuilt first when stale or when a
        mask_d is given).  Not differentiable: the reference evaluates under no_grad."""
        if self._eval_state != "ready" or mask_d is not None:
            if self._eval_state == "fresh" and mask_d is None:
                # reference behaviour on a fresh module in eval(): F.embedding on an empty weight
                raise RuntimeError("'weight' must be 2-D")
            self._rebuild_eval(mask_d)
        sg = self.shards
        lib = L.load()
        dev = L.require_cuda(x, offsets, fc, bias)
        if x.dtype not in (torch.int32, torch.int64):
            raise RuntimeError(f"rsb: ids must be int32 or int64, got {x.dtype}")
        x = x.contiguous()
        b, f = x.shape
        d = sg.dim
        use_fm = fc is not None
        emb = torch.empty(b, f, d, dtype=torch.float32, device=dev)
        y = torch.empty(b, dtype=torch.float32, device=dev) if use_fm else None
        s = torch.empty(b, d, dtype=torch.float32, device=dev) if use_fm else None
        rows = torch.empty(b, f, dtype=torch.int64, device=dev)
        slots = RF.amax_slots_for(dev)
        nbytes = b * (f * x.element_size() + 2 * f * d * 4 + f * 8 + (f * 4 + 4 + d * 4 if use_fm else 0))
        RF._call("lookup_fwd_sharded", lib.rsb_lookup_fwd_sharded_kind, L.KIND_VANILLA, L.ptr(x),
                 int(x.dtype == torch.int32), L.ptr(offsets), b, f, d, L.ptr(sg.ptrs["eval"]), sg.world, sg.num_rows,
                 sg.num_rows, None, 0, None, None, 0, None, L.ptr(fc) if use_fm else None,
                 L.ptr(bias) if use_fm else None, L.ptr(emb), L.ptr(y), L.ptr(s), L.ptr(rows), L.ptr(sg.err_flag),
                 L.ptr(slots), L.stream_ptr(dev), nbytes=nbytes)
        if slots is not None:
            emb._rsb_amax_slots = slots
        return emb, y

    @torch.no_grad()
    def get_weight(self, mask_d: Optional[torch.Tensor] = None):
        """The effective [N, D] table the reference's get_weight returns (QR: emb1 (x) emb2, PEP: soft-thresholded,
        retrain: weight * mask) = the lookup of every id; peer rows are read in place, no collective.  OptEmbed: the
        masked table for `mask_d` (deepfm_opt_embed.py:148-202), rebuilt into the eval shards (which it leaves as the
        eval cache, like the reference) and all-gathered - a collective.  The other kinds ignore mask_d, as
        RetrainOptEmbed does."""
        if isinstance(self.inner, OptEmbed):
            self._rebuild_eval(mask_d)
            return self._gather_full(self.shards.buf["eval"].tensor, self._full_rows)
        ids = torch.arange(self.inner._num_item, device=self.shards.device)
        return self(ids)

    def forward(self, x, mask_d=None):
        """IEmbedding.forward; OptEmbed outside training rebuilds its eval cache with `mask_d` first (a collective), as
        OptEmbed.forward does."""
        if isinstance(self.inner, OptEmbed) and not self.training and mask_d is not None:
            self._rebuild_eval(mask_d)
        return self._plugin_forward(x)

    # -- the plugin's bookkeeping methods, global over the shards (the scripts call them: train_deepfm_pep.py:63,71,
    #    train_deepfm_optembed.py, SURVEY 8b) ------
    def __getattr__(self, name):
        """Attributes of the wrapped module (`sparsity`, `checkpoint_weight_dir`, `threshold_type`, `get_l_s`, ...)
        read through."""
        try:
            return super().__getattr__(name)
        except AttributeError:
            inner = self.__dict__.get("_modules", {}).get("inner")
            if inner is None or name == "inner":
                raise
            return getattr(inner, name)

    def _optembed_count(self) -> int:
        """Surviving weights of the mask-E-only table (OptEmbed.get_sparsity): the eval kernel's count on every shard,
        all-reduced (padding rows are zero and count nothing)."""
        inner = self.inner
        _, cnt = RF.optembed_eval_weight(inner._weight.detach(), self._shard_rows(inner._t_rows()), None, inner._norm,
                                         want_out=False, want_count=True)
        return self._all_sum(cnt)

    def get_num_params(self) -> int:
        inner, sg = self.inner, self.shards
        kind = inner._spec().kind
        if kind == L.KIND_PEP:
            n = int(inner.get_num_params())              # surviving weights of THIS shard (padding rows are zero)
            if sg.world > 1:
                t = torch.tensor([n], dtype=torch.int64, device=sg.device)
                dist.all_reduce(t, group=sg.group)
                n = int(t.item())
            return n
        if kind == L.KIND_OPTEMBED:
            if self._eval_state == "ready" and not self.training:
                return self._all_sum(torch.count_nonzero(sg.buf["eval"].tensor).reshape(1))
            return self._optembed_count()
        if isinstance(inner, RetrainOptEmbed):
            return self._all_sum(torch.count_nonzero(inner._mask).reshape(1))
        if kind == L.KIND_MASK:
            return inner.get_num_params()                # counted on the full mask when the module was built
        sharded = self._names()
        total = 0
        for name, p in inner.named_parameters():
            total += self._full_rows * (p.numel() // max(p.shape[0], 1)) if sharded[name] else p.numel()
        return total

    def get_sparsity(self, get_n_params=False):
        inner = self.inner
        kind = inner._spec().kind
        if kind == L.KIND_PEP:
            total = self._full_rows * inner._hidden_size
            n = self.get_num_params()
            return ((1 - n / total), n) if get_n_params else 1 - n / total
        if kind == L.KIND_OPTEMBED or isinstance(inner, RetrainOptEmbed):
            n = self._optembed_count() if kind == L.KIND_OPTEMBED else self.get_num_params()
            sparsity = 1 - n / (inner._num_item * inner._hidden_size)
            return (sparsity, n) if get_n_params else sparsity
        return inner.get_sparsity(get_n_params)

    @torch.no_grad()
    def get_mask_e(self) -> torch.Tensor:
        """OptEmbed.get_mask_e: [N] int64 on the CPU, 1 where a row survives mask-E; per shard, then all-gathered."""
        inner = self.inner
        if isinstance(inner._mask_e_module, nn.Identity):
            return torch.ones(inner._num_item, dtype=torch.int64)
        emb, _ = RF.optembed_eval_weight(inner._weight.detach(), self._shard_rows(inner._t_rows()), None, inner._norm)
        local = (emb.abs().sum(1) > 0).to(torch.int64)
        return self._gather_full(local, self._full_rows).cpu()

    def get_submask(self) -> torch.Tensor:
        """OptEmbed.get_submask from the global mask-E, cached on the wrapped module until the next training forward."""
        inner = self.inner
        if inner._submask_cache is None:
            inner._submask_cache = inner._submask(self.get_mask_e)
        return inner._submask_cache

    def train_callback(self):
        """PepEmbeeding.train_callback (pep_embedding.py:132-147) on the global sparsity: when a target is crossed every
        rank takes part in gathering the full state (a collective) and rank 0 writes `{sparsity}.pth`."""
        inner, sg = self.inner, self.shards
        if inner._spec().kind != L.KIND_PEP:
            return inner.train_callback()
        with torch.no_grad():
            cur = self.get_sparsity()
        while inner._cur_min_spar_idx < len(inner.sparsity) and inner.sparsity[inner._cur_min_spar_idx] < cur:
            target = inner.sparsity[inner._cur_min_spar_idx]
            state = self.full_state_dict()
            if sg.rank == 0:
                torch.save(state, os.path.join(inner.checkpoint_weight_dir, f"{target}.pth"))
            inner._cur_min_spar_idx += 1

    def lookup(self, x, offsets=None, fc=None, bias=None, mask_d=None):
        """The fused lookup over the shards.  `mask_d` is OptEmbed's: used outside training only (see forward)."""
        inner = self.inner
        spec = inner._spec()
        if offsets is not None:
            offsets = offsets.reshape(-1).long()
        self._rsb_err_flag = self.shards.err_flag
        mask_d_idx = None
        if spec.kind == L.KIND_OPTEMBED:
            if not self.training:
                emb, y = self._eval_lookup(x, offsets, fc, bias, mask_d)
                if self.validate:
                    RF.check_index_errors(self)
                return emb, y
            if x.dim() != 2 or x.shape[1] != inner._num_field:
                raise RuntimeError("OptEmbed training forward expects x of shape [B, num_field]")
            # weights are about to change: drop the eval cache (the module's own backward hook never runs here)
            self._eval_state = "stale"
            inner._submask_cache = None
            # the same draw as the single-device forward (one torch.randint over this rank's [B, F] lookups)
            mask_d_idx = inner._mask_d_for(x.shape[0], x.shape[1], x.device)
        table, table1, aux = _kernel_tensors(inner)
        if isinstance(inner, RetrainOptEmbed):
            assert aux is not None, "Mask is not initialized"
        presort = RF.EARLY_SORT and torch.is_grad_enabled() and table.requires_grad
        slots = RF.amax_slots_for(x.device)
        aux_rep = None if self._per_row_aux else aux
        emb, y, _ = _ShardedKindLookup.apply(self.shards, spec, x, offsets, table, table1, aux_rep, fc, bias, presort,
                                             slots, mask_d_idx)
        if slots is not None:
            emb._rsb_amax_slots = slots
        if self.validate:
            RF.check_index_errors(self)
        return emb, (y if fc is not None else None)


class _ShardedStepMixin:
    """The two calls a training step adds around the optimizers (see the module docstring)."""

    def shard_params(self):
        emb = self.embedding
        return emb.shard_params() if isinstance(emb, ShardedEmbedding) else [emb._emb_module.weight]

    def replicated_params(self):
        ids = {id(p) for p in self.shard_params()}
        return [p for p in self.parameters() if id(p) not in ids and p.requires_grad]

    def sync_gradients(self):
        """Call after backward(): averages the replicated gradients over the ranks (this
        allreduce is also the point after which every rank's pushes into our shard gradient
        are complete) and exposes the accumulated shard gradients as `.grad`."""
        emb = self.embedding
        sg = emb.shards
        allreduce_mean_([p.grad for p in self.replicated_params() if p.grad is not None], sg.group)
        if isinstance(emb, ShardedEmbedding):
            emb.expose_shard_grads(True)
        else:
            emb._emb_module.weight.grad = sg.buf["table_grad"].tensor

    def finish_step(self):
        """Call after optimizer.step(): re-zero the shard gradient accumulators and order the
        next step's peer gathers / pushes after every rank's update."""
        emb = self.embedding
        sg = emb.shards
        if isinstance(emb, ShardedEmbedding):
            emb.expose_shard_grads(False)
        else:
            emb._emb_module.weight.grad = None
        sg.zero_grads()
        sg.barrier()


def _sharded_embedding(embedding_config, field_dims, num_factor, field_name, group):
    from . import get_embedding

    cfg = dict(embedding_config or {"name": "vanilla"})
    if cfg.get("name", "vanilla") == "vanilla":
        cfg.pop("name", None)
        cfg.pop("sparse", None)
        return ShardedVanillaEmbedding(field_dims, num_factor, group=group, **cfg)
    return ShardedEmbedding(get_embedding(cfg, field_dims, num_factor, mode=None, field_name=field_name), group=group)


class ShardedDeepFM(_ShardedStepMixin, DeepFM):
    """DeepFM (src/models/deepfm.py:11-105) with the embedding's big arrays row-sharded (vanilla table, QR emb2, PEP
    weight + thresholds, OptEmbed weight, retrain weight + mask); the first-order weights `fc` (4 B per row), the MLP, `_bias` and
    BatchNorm are replicated (BatchNorm statistics stay per-rank).  Build it after `dist.init_process_group` with the
    device current and the same seed on every rank."""

    def __init__(self, field_dims, num_factor, hidden_sizes, p_dropout=0.1, use_batchnorm=False,
                 embedding_config=None, group=None):
        super().__init__(field_dims, num_factor, hidden_sizes, p_dropout, use_batchnorm, {"name": "vanilla"},
                         empty_embedding=True)
        self.embedding = _sharded_embedding(embedding_config, field_dims, num_factor, "deepfm", group)

    def forward(self, x):
        emb, y_fm = self.embedding.lookup(x, self.offsets, self.fc.weight, self._bias)
        b = emb.shape[0]
        scores = y_fm.unsqueeze(1) + run_sequential(self._deep_branch, emb.reshape(b, emb.shape[1] * emb.shape[2]),
                                                    overlap_first_dw=True, x_amax_slots=RF.amax_slots_of(emb))
        return scores.squeeze(-1)


class ShardedDCNMix(_ShardedStepMixin, DCN_Mix):
    """DCN_Mix (src/models/dcn.py:11-96) over a row-sharded embedding; cross layers and the MLP tail replicated."""

    def __init__(self, field_dims, num_factor, hidden_sizes, num_layers=3, num_experts=4, rank=64, activation=None,
                 embedding_config=None, p_dropout=0.5, group=None):
        super().__init__(field_dims, num_factor, hidden_sizes, num_layers, num_experts, rank, activation,
                         {"name": "vanilla"}, p_dropout, empty_embedding=True)
        self.embedding = _sharded_embedding(embedding_config, field_dims, num_factor, "dcn", group)


class ShardedStepOptimizers:
    """Facade with the `zero_grad()` / `step()` interface the reference trainer drives
    (src/trainer/deepfm.py:52-60): step() = sync_gradients -> inner optimizers -> finish_step."""

    def __init__(self, model, optimizers: List[torch.optim.Optimizer]):
        self.model, self.optimizers = model, optimizers

    def zero_grad(self, set_to_none: bool = True):
        for p in self.model.replicated_params():
            p.grad = None

    def step(self):
        self.model.sync_gradients()
        for o in self.optimizers:
            o.step()
        self.model.finish_step()
