"""B200-native embedding plugins behind the reference's IEmbedding API.

Same class roles, constructor kwargs, parameter names / shapes / dtypes / requires_grad
flags and extra methods as the reference classes they replace, so existing yaml configs
and checkpoints load unchanged (SURVEY.md section 8b):

    VanillaEmbedding        src/models/embeddings/base.py:23-75
    QRHashingEmbedding      src/models/embeddings/qr_embedding.py:10-113
    PepEmbeeding            src/models/embeddings/pep_embedding.py:12-147
    RetrainPepEmbedding     src/models/embeddings/pep_embedding.py:150-229
    OptEmbed                src/models/embeddings/deepfm_opt_embed.py:40-307
    RetrainOptEmbed         src/models/embeddings/deepfm_opt_embed.py:633-718

Every forward is ONE launch of the fused gather kernel with the variant applied inside
it.  `forward(x)` keeps the plugin contract (x already offset -> [B,F,D]);
`lookup(x, offsets, fc, bias)` is the fused entry our DeepFM / DCN_Mix call (offset add,
gather, first order and FM second order in the same launch).
"""
from __future__ import annotations

import math
import os
from typing import Iterable, List, Optional, Union

import torch
from torch import nn

from . import _lib as L
from . import functional as RF


class IEmbedding(nn.Module):
    """Reference interface (src/models/embeddings/base.py:8-20)."""

    def get_weight(self) -> torch.Tensor:
        raise NotImplementedError

    def get_num_params(self) -> int:
        return sum(p.numel() for p in self.parameters())

    # ---- shared machinery ---------------------------------------------------
    _mode: Optional[str] = None
    validate: bool = False  # True: synchronise and raise IndexError on out-of-range ids

    def _spec(self) -> RF.LookupSpec:
        raise NotImplementedError

    def _tensors(self):
        """(table, table1, aux) handed to the kernel."""
        raise NotImplementedError

    def _mask_d_for(self, b: int, f: int, device) -> Optional[torch.Tensor]:
        return None

    def train(self, mode: bool = True):
        """Out-of-range ids do not fault inside the gather (they are clamped to row 0 and an error flag is set; the
        reference's F.embedding raises IndexError / a device assert).  Reading the flag needs a host sync, so it is
        read where the reference trainer synchronises anyway: on every train() / eval() switch (epoch boundaries,
        src/trainer/deepfm.py:27,113) - and on every call with `validate = True`."""
        RF.check_index_errors(self)
        return super().train(mode)

    def lookup(self, x: torch.Tensor, offsets: Optional[torch.Tensor] = None, fc: Optional[torch.Tensor] = None,
               bias: Optional[torch.Tensor] = None):
        """Fused lookup on raw [B,F] ids. Returns (emb [B,VF,E], y_fm [B] or None)."""
        table, table1, aux = self._tensors()
        if offsets is not None:
            offsets = offsets.reshape(-1)
            if offsets.dtype != torch.int64:
                offsets = offsets.long()
        mask_d = self._mask_d_for(x.shape[0], x.shape[1], x.device)
        emb, y = RF.fused_lookup(self._spec(), x, offsets, table, table1, aux, mask_d, fc, bias)
        if self.validate:
            RF.check_index_errors(self)
        return emb, y

    def _plugin_forward(self, x: torch.Tensor) -> torch.Tensor:
        """IEmbedding.forward contract: ids already offset; any leading shape; bag modes."""
        one_d = x.dim() == 1
        x2 = x.reshape(-1, 1) if one_d else x.reshape(-1, x.shape[-1])
        emb, _ = self.lookup(x2, None)
        if one_d:
            return emb.reshape(x.shape[0], -1)
        if x.dim() > 2:
            emb = emb.reshape(*x.shape[:-1], *emb.shape[1:])
        mode = self._mode
        if mode is None:
            return emb
        if mode == "sum":
            return emb.sum(-2)
        if mode == "mean":
            return emb.mean(-2)
        return emb.max(-2).values

    def forward(self, x):
        return self._plugin_forward(x)


def _as_list(field_dims) -> List[int]:
    if isinstance(field_dims, int):
        return [field_dims]
    return [int(v) for v in field_dims]


# ------------------------------------------------------------------------------
class VanillaEmbedding(IEmbedding):
    """One concatenated table (base.py:23-75).  kwargs (e.g. sparse=True) go to nn.Embedding
    exactly like the reference; `sparse=True` makes backward emit the same uncoalesced COO grad."""

    def __init__(self, field_dims: Union[Iterable[int], int], hidden_size: int, mode: Optional[str] = None,
                 initializer="xavier", **kwargs):
        super().__init__()
        field_dims = _as_list(field_dims)
        assert mode in [None, "sum", "mean", "max"]
        self._mode = mode
        if mode is None:
            self._emb_module = nn.Embedding(sum(field_dims), hidden_size, **kwargs)
        else:
            self._emb_module = nn.EmbeddingBag(sum(field_dims), hidden_size, mode=mode, **kwargs)
        if initializer == "xavier":
            nn.init.xavier_uniform_(self._emb_module.weight)
        else:
            nn.init.normal_(self._emb_module.weight, std=0.1)
        self._num_item = sum(field_dims)
        self._hidden_size = hidden_size

    def get_weight(self):
        return self._emb_module.weight

    def _spec(self):
        return RF.LookupSpec(L.KIND_VANILLA, self._num_item, self._hidden_size,
                             sparse_grad=bool(getattr(self._emb_module, "sparse", False)), module=self)

    def _tensors(self):
        return self._emb_module.weight, None, None


# ------------------------------------------------------------------------------
class QRHashingEmbedding(IEmbedding):
    """Quotient-remainder hashing (qr_embedding.py:10-113); index math inside the gather."""

    def __init__(self, field_dims: Union[int, List[int]], hidden_size: int, mode: Optional[str] = None,
                 divider: Optional[int] = None, operation: str = "mult", initializer="uniform"):
        super().__init__()
        assert operation in ["cat", "add", "mult"]
        if operation == "cat":
            assert hidden_size % 2 == 0
        field_dims = _as_list(field_dims)
        num_item = sum(field_dims)
        if divider is None:
            divider = int(math.sqrt(num_item))
        emb_size = hidden_size // 2 if operation == "cat" else hidden_size
        self._operation = operation
        size = (num_item - 1) // divider + 1
        if mode is None:
            self.emb1 = nn.Embedding(divider, emb_size)
            self.emb2 = nn.Embedding(size, emb_size)
        else:
            self.emb1 = nn.EmbeddingBag(divider, emb_size, mode=mode)
            self.emb2 = nn.EmbeddingBag(size, emb_size, mode=mode)
        self._mode = mode
        self._hidden_size = hidden_size
        self._divider = divider
        self._num_item = num_item
        if initializer == "normal":
            self._init_normal_weight()
        elif initializer == "uniform":
            self._init_uniform_weight()

    def _init_uniform_weight(self):
        alpha = math.sqrt(1 / self._num_item)
        nn.init.uniform_(self.emb1.weight, alpha, 1)
        nn.init.uniform_(self.emb2.weight, alpha, 1)

    def _init_normal_weight(self):
        std = 0.1
        if self._operation == "add":
            std = std / 2
        elif self._operation == "mult":
            std = math.sqrt(std)
        nn.init.normal_(self.emb1.weight, std=std)
        nn.init.normal_(self.emb2.weight, std=std)

    def _spec(self):
        return RF.LookupSpec(L.QR_KINDS[self._operation], self._num_item, self._hidden_size,
                             divider=self._divider, module=self)

    def _tensors(self):
        return self.emb2.weight, self.emb1.weight, None

    def get_weight(self):
        arr = torch.arange(self._num_item, device=self.emb1.weight.device)
        return self(arr)


# ------------------------------------------------------------------------------
class PepEmbeeding(IEmbedding):
    """PEP learnable soft-threshold pruning (pep_embedding.py:12-147).  The reference
    thresholds the WHOLE table every forward; here the threshold is applied to the gathered
    rows only, inside the gather, and the dense gradients autograd expects are rebuilt from
    the touched rows."""

    def __init__(self, field_dims: Union[List[int], int], hidden_size: int, mode: Optional[str] = None,
                 ori_weight_dir: str = "", checkpoint_weight_dir: str = "checkpoints", field_name: str = "",
                 init_threshold: float = -150, threshold_type: str = "feature_dim",
                 sparsity: Optional[List[float]] = None):
        super().__init__()
        field_dims = _as_list(field_dims)
        num_item = sum(field_dims)
        if sparsity is None:
            sparsity = [0.8, 0.9, 0.99]
        assert isinstance(sparsity, list) and isinstance(sparsity[0], float)
        self.sparsity = list(sorted(sparsity))
        self._cur_min_spar_idx = 0
        self.emb = nn.Embedding(num_item, hidden_size)
        nn.init.xavier_uniform_(self.emb.weight)
        if ori_weight_dir:
            os.makedirs(ori_weight_dir, exist_ok=True)
            torch.save({"state_dict": self.emb.state_dict()}, os.path.join(ori_weight_dir, field_name + ".pth"))
        self.threshold_type = threshold_type
        self.s = self.init_threshold(init_threshold, num_item, hidden_size)
        self.field_name = field_name
        if field_name:
            checkpoint_weight_dir = os.path.join(checkpoint_weight_dir, field_name)
        os.makedirs(checkpoint_weight_dir, exist_ok=True)
        self.checkpoint_weight_dir = checkpoint_weight_dir
        self._mode = mode
        self._num_item = num_item
        self._hidden_size = hidden_size

    def init_threshold(self, init, num_item, hidden_size) -> nn.Parameter:
        if self.threshold_type == "global":
            return nn.Parameter(init * torch.ones(1))
        if self.threshold_type == "dimension":
            return nn.Parameter(init * torch.ones([hidden_size]))
        if self.threshold_type == "feature":
            return nn.Parameter(init * torch.ones([num_item, 1]))
        if self.threshold_type == "feature_dim":
            return nn.Parameter(init * torch.ones([num_item, hidden_size]))
        if self.threshold_type in ("field", "field_dim"):
            raise NotImplementedError()
        raise ValueError("Invalid threshold_type: {}".format(self.threshold_type))

    def soft_threshold(self, v, s):
        """Full-table soft threshold (used by get_weight / callers that want the tensor)."""
        out, _ = RF.pep_threshold_table(v.detach(), s.detach(), L.PEP_TYPES[self.threshold_type])
        return out

    def get_weight(self):
        return self.soft_threshold(self.emb.weight, self.s)

    def _spec(self):
        return RF.LookupSpec(L.KIND_PEP, self._num_item, self._hidden_size,
                             aux_mode=L.PEP_TYPES[self.threshold_type], module=self)

    def _tensors(self):
        return self.emb.weight, None, self.s

    def get_num_params(self) -> int:
        _, cnt = RF.pep_threshold_table(self.emb.weight.detach(), self.s.detach(),
                                        L.PEP_TYPES[self.threshold_type], want_out=False, want_count=True)
        return int(cnt.item())

    def get_sparsity(self, get_n_params=False):
        total_params = self.emb.weight.numel()
        n_params = self.get_num_params()
        if get_n_params:
            return (1 - n_params / total_params), n_params
        return 1 - n_params / total_params

    def train_callback(self):
        with torch.no_grad():
            cur_sparsity = self.get_sparsity()
        while self._cur_min_spar_idx < len(self.sparsity) and self.sparsity[self._cur_min_spar_idx] < cur_sparsity:
            sparsity = self.sparsity[self._cur_min_spar_idx]
            torch.save(self.state_dict(), os.path.join(self.checkpoint_weight_dir, f"{sparsity}.pth"))
            self._cur_min_spar_idx += 1


class RetrainPepEmbedding(IEmbedding):
    """PEP retrain: weight * fixed bool mask (pep_embedding.py:150-229); the mask row is read
    inside the gather instead of multiplying the whole table every forward."""

    def __init__(self, field_dims: Union[List[int], int], hidden_size, mode: Optional[str], checkpoint_weight_dir,
                 sparsity: Union[float, str] = 0.8, ori_weight_dir: Optional[str] = None, field_name: str = "",
                 sparse=False):
        super().__init__()
        field_dims = _as_list(field_dims)
        num_item = sum(field_dims)
        self.emb = nn.Embedding(num_item, hidden_size)
        if ori_weight_dir:
            ori = torch.load(os.path.join(ori_weight_dir, field_name + ".pth"), map_location="cpu")["state_dict"]
            self.emb.load_state_dict(ori)
        finish = torch.load(os.path.join(checkpoint_weight_dir, field_name, f"{sparsity}.pth"), map_location="cpu")
        weight, s = finish["emb.weight"], finish["s"]
        self.mask = nn.Parameter((torch.abs(weight) - torch.sigmoid(s)) > 0, False)
        nnz = self.mask.sum()
        self._nnz = nnz
        self.sparsity = 1 - (nnz / torch.prod(torch.tensor(self.mask.size()))).item()
        self._mode = mode
        self._sparse = sparse
        self._num_item = num_item
        self._hidden_size = hidden_size

    def get_weight(self):
        return RF.mask_table(self.emb.weight.detach(), self.mask)

    def _spec(self):
        return RF.LookupSpec(L.KIND_MASK, self._num_item, self._hidden_size, sparse_grad=bool(self._sparse),
                             module=self)

    def _tensors(self):
        return self.emb.weight, None, self.mask

    def get_sparsity(self, get_n_params=False):
        if get_n_params:
            return self.sparsity, self._nnz
        return self.sparsity

    def get_num_params(self):
        return self._nnz


# ------------------------------------------------------------------------------
def get_mask(hidden_size: int) -> torch.Tensor:
    """matrix[i][j] = 1 if i >= j (optembed_utils.py:10-22)."""
    return torch.tril(torch.ones((hidden_size, hidden_size), dtype=torch.bool))


class _MaskEmbeddingModule(nn.Module):
    """Holder of the mask-E threshold `_t_param` (optembed_utils.py:47-106); the mask itself
    is computed inside the gather (training) or by the eval-weight kernel."""

    def __init__(self, field_dims: torch.Tensor, t_init: float = 0, mode_threshold_e="field", norm=1):
        super().__init__()
        assert mode_threshold_e in ["feature", "field"]
        self.mode_threshold_e = mode_threshold_e
        self.register_buffer("_field_dims", field_dims)
        self._num_item = int(field_dims.sum())
        self._num_field = len(field_dims)
        t_size = self._num_item if mode_threshold_e == "feature" else self._num_field
        self._t_param = nn.Parameter(torch.empty(t_size))
        nn.init.constant_(self._t_param, t_init)
        self._norm = norm

    def _transform_t_to_feat(self):
        if self.mode_threshold_e == "feature":
            return self._t_param
        return torch.repeat_interleave(self._t_param, self._field_dims, dim=0, output_size=self._num_item)


def _delete_cache(module, grad_input, grad_output):
    module._cur_weight = None
    if hasattr(module, "_submask_cache"):
        module._submask_cache = None


class IOptEmbed(IEmbedding):
    def get_l_s(self):
        return 0


class OptEmbed(IOptEmbed):
    """OptEmbed supernet for DeepFM (deepfm_opt_embed.py:40-307): per-field threshold mask-E
    (BinaryStep STE on the row norm) x random lower-triangular mask-D, both applied inside
    the gather in training; eval gathers from a cached masked table like the reference.
    The evolutionary search (deepfm_opt_embed.py:310-622) is host-side bookkeeping and out
    of scope; the methods it calls (get_weight(mask_d), get_submask, get_mask_e) are here."""

    def __init__(self, field_dims: Union[List[int], int], hidden_size: int, mode: Optional[str] = None,
                 t_init: Optional[float] = 0, mode_threshold_e="field", mode_threshold_d="field", norm=1,
                 target_sparsity: Optional[float] = None):
        super().__init__()
        field_dims = _as_list(field_dims)
        assert mode in ["sum", "mean", "max", None]
        assert mode_threshold_e in ["field", "feature"]
        assert mode_threshold_d in ["field", "feature"]
        self._field_dims = torch.tensor(field_dims, dtype=torch.int64)
        self._num_item = int(self._field_dims.sum())
        self._num_field = len(field_dims)
        self._hidden_size = hidden_size
        self._weight = nn.Parameter(torch.empty((self._num_item, hidden_size)))
        self.register_buffer("_cur_weight", torch.empty(0), persistent=False)
        nn.init.xavier_uniform_(self._weight)
        self._handle = self.register_full_backward_hook(_delete_cache)
        self._mode = mode
        self._t_init = t_init
        if t_init is None:
            self._mask_e_module = nn.Identity()
        else:
            self._mask_e_module = _MaskEmbeddingModule(self._field_dims, t_init, mode_threshold_e, norm)
        self.register_buffer("_full_mask_d", get_mask(hidden_size))
        self._target_sparsity = target_sparsity
        self._naive = False
        self._mode_d = mode_threshold_d
        self._norm = norm
        self._submask_cache = None

    # -- helpers ---------------------------------------------------------------
    def _t_param(self) -> Optional[torch.Tensor]:
        if isinstance(self._mask_e_module, nn.Identity):
            return None
        return self._mask_e_module._t_param

    def _t_rows(self) -> Optional[torch.Tensor]:
        if isinstance(self._mask_e_module, nn.Identity):
            return None
        return self._mask_e_module._transform_t_to_feat().detach().contiguous()

    def get_l_s(self):
        if self._t_init is None:
            return 0
        return torch.exp(-self._mask_e_module._t_param).sum()

    def _masked_table(self, mask_d_rows: Optional[torch.Tensor], want_count=False):
        out, cnt = RF.optembed_eval_weight(self._weight.detach(), self._t_rows(), mask_d_rows, self._norm,
                                           want_out=True, want_count=want_count)
        return out, cnt

    def get_weight(self, mask_d: Optional[torch.Tensor] = None):
        """Masked full table (deepfm_opt_embed.py:148-202).  mask_d: int indices per field /
        per feature (dims 0..k kept) or a [N,D] bool mask."""
        rows_idx, bool_mask = self._mask_d_rows(mask_d)
        out, _ = self._masked_table(rows_idx)
        if bool_mask is not None:
            out = out * bool_mask.to(out.dtype)
        self._cur_weight = out
        return self._cur_weight

    def _mask_d_rows(self, mask_d: Optional[torch.Tensor]):
        """get_weight's mask-D as (per-row int64 [N] indices or None, [N, D] bool mask or None); in training without
        a mask_d, the reference's random draw."""
        device = self._weight.device
        rows_idx = None
        bool_mask = None
        if self.training and mask_d is None:
            if self._mode_d == "feature":
                rows_idx = torch.randint(0, self._hidden_size, (self._num_item,), device=device)
            else:
                idx = torch.randint(0, self._hidden_size, (self._num_field,))
                rows_idx = torch.repeat_interleave(idx, self._field_dims, dim=0, output_size=self._num_item).to(device)
        elif mask_d is not None:
            if mask_d.dtype in (torch.int32, torch.int64):
                rows_idx = mask_d.to(device).long()
                if self._mode_d == "field" and rows_idx.numel() == self._num_field:
                    rows_idx = torch.repeat_interleave(rows_idx, self._field_dims.to(device), dim=0,
                                                       output_size=self._num_item)
            else:
                bool_mask = mask_d.to(device)
        return (rows_idx.contiguous() if rows_idx is not None else None), bool_mask

    def _spec(self):
        return RF.LookupSpec(L.KIND_OPTEMBED, self._num_item, self._hidden_size, aux_mode=self._norm, module=self)

    def _tensors(self):
        if self.training:
            return self._weight, None, self._t_param()
        return self._cur_weight, None, None

    def _mask_d_for(self, b, f, device):
        if not self.training:
            return None
        # the SAME torch call the reference makes (deepfm_opt_embed.py:222-224), so that a
        # seeded run draws the identical mask
        return torch.randint(0, self._hidden_size, size=(b, self._num_field), device=device)

    def lookup(self, x, offsets=None, fc=None, bias=None, mask_d=None):
        if self.training:
            t = self._t_param()
            if t is not None and self._mask_e_module.mode_threshold_e != "field":
                raise AssertionError("Cannot apply field mask to input")
            if x.dim() != 2 or x.shape[1] != self._num_field:
                raise RuntimeError("OptEmbed training forward expects x of shape [B, num_field]")
            # weights are about to change: drop the eval cache (the reference does it in a backward hook)
            self._cur_weight = None
            self._submask_cache = None
            return super().lookup(x, offsets, fc, bias)
        # evaluation: gather from the cached masked table (built on demand)
        if self._cur_weight is None or self._cur_weight.numel() == 0 or mask_d is not None:
            if self._cur_weight is not None and self._cur_weight.numel() == 0 and mask_d is None:
                # reference behaviour on a fresh module in eval(): F.embedding on an empty weight
                raise RuntimeError("'weight' must be 2-D")
            self.get_weight(mask_d)
        spec = RF.LookupSpec(L.KIND_VANILLA, self._num_item, self._hidden_size, module=self)
        if offsets is not None:
            offsets = offsets.reshape(-1).long()
        emb, y = RF.fused_lookup(spec, x, offsets, self._cur_weight, None, None, None, fc, bias)
        return emb, y

    def forward(self, x, mask_d=None):
        if not self.training and mask_d is not None:
            self.get_weight(mask_d)
        return self._plugin_forward(x)

    def get_sparsity(self, get_n_params=False):
        _, cnt = RF.optembed_eval_weight(self._weight.detach(), self._t_rows(), None, self._norm, want_out=False,
                                         want_count=True)
        nnz = int(cnt.item())
        sparsity = 1 - nnz / (self._num_item * self._hidden_size)
        if get_n_params:
            return sparsity, nnz
        return sparsity

    def get_num_params(self):
        if self._cur_weight is not None and self._cur_weight.numel() > 0 and not self.training:
            return int(torch.count_nonzero(self._cur_weight).item())
        return self.get_sparsity(True)[1]

    def get_mask_e(self):
        if isinstance(self._mask_e_module, nn.Identity):
            return torch.ones(self._num_item, dtype=torch.int64)
        emb, _ = self._masked_table(None)
        return (emb.abs().sum(1) > 0).to(torch.int64).cpu()

    def get_submask(self) -> torch.Tensor:
        if self._submask_cache is None:
            self._submask_cache = self._submask(self.get_mask_e)
        return self._submask_cache

    def _submask(self, get_mask_e) -> torch.Tensor:
        """get_submask without the cache, from the mask-E that `get_mask_e()` returns."""
        if isinstance(self._mask_e_module, nn.Identity):
            return self._field_dims if self._mode_d == "field" else torch.ones(self._num_item, dtype=torch.int64)
        mask_e = get_mask_e()
        if self._mode_d == "feature":
            return mask_e
        num_e = torch.cat([torch.zeros(1, dtype=torch.int64), mask_e.cumsum(0)])
        offsets = torch.cat([torch.zeros(1, dtype=torch.int64), self._field_dims]).cumsum(0)
        return num_e[offsets[1:]] - num_e[offsets[:-1]]


class RetrainOptEmbed(IOptEmbed):
    """OptEmbed retrain: weight * fixed mask (deepfm_opt_embed.py:633-718); mask row read
    inside the gather (the reference re-multiplies the whole table after every backward)."""

    def __init__(self, field_dims: Union[List[int], int], hidden_size, mode: Optional[str] = None,
                 t_init: Optional[float] = 0, mode_threshold_e="field", mode_threshold_d="field", norm=1,
                 target_sparsity: Optional[float] = None):
        super().__init__()
        field_dims = _as_list(field_dims)
        self._num_item = sum(field_dims)
        self._field_dims = torch.tensor(field_dims, dtype=torch.int64)
        self._mode_d = mode_threshold_d
        self._mode = mode
        self._hidden_size = hidden_size
        self._weight = nn.Parameter(torch.empty((self._num_item, hidden_size)))
        self.register_buffer("_full_mask_d", get_mask(hidden_size))
        self._mask_d = None
        self._mask_e = None
        self._mask = None
        self._sparsity = 0
        self._cur_weight = None

    def init_mask(self, mask_e, mask_d):
        mask_e = mask_e.unsqueeze(-1)
        if self._mode_d == "field":
            mask_d = torch.repeat_interleave(mask_d, self._field_dims.to(mask_d.device), dim=0,
                                             output_size=self._num_item)
        mask_d = torch.nn.functional.embedding(mask_d, self._full_mask_d.to(mask_d.device))
        self._mask = nn.Parameter((mask_d * mask_e).to(self._weight.device), False)
        self._cur_weight = None
        return self._mask

    def _mask_u8(self) -> torch.Tensor:
        m = self._mask
        cache = getattr(self, "_mask_u8_cache", None)
        if cache is None or cache[0] is not m or cache[1].device != self._weight.device:
            u8 = (m.detach() != 0).to(device=self._weight.device, dtype=torch.uint8).contiguous()
            self._mask_u8_cache = (m, u8)
            return u8
        return cache[1]

    def get_weight(self, mask_d: Optional[torch.Tensor] = None):
        assert self._mask is not None, "Mask is not initialized"
        self._cur_weight = RF.mask_table(self._weight.detach(), self._mask_u8())
        return self._cur_weight

    def _spec(self):
        return RF.LookupSpec(L.KIND_MASK, self._num_item, self._hidden_size, module=self)

    def _tensors(self):
        assert self._mask is not None, "Mask is not initialized"
        return self._weight, None, self._mask_u8()

    def forward(self, x, mask_d=None):
        return self._plugin_forward(x)

    def get_sparsity(self, get_n_params=False):
        nnz = torch.count_nonzero(self._mask).item()
        sparsity = 1 - nnz / (self._hidden_size * self._num_item)
        if not get_n_params:
            return sparsity
        return sparsity, nnz

    def get_num_params(self):
        return torch.count_nonzero(self._mask).item()


# ------------------------------------------------------------------------------
class CerpEmbedding(IEmbedding):
    """CERP (src/models/embeddings/cerp_embedding.py:14-207): two bucket tables P, Q, each PEP
    soft-thresholded with element-wise thresholds, composed by QR-style index math
    (q = x // q_entity_per_row, p = x % bucket_size) and summed.  The two small tables are
    thresholded in one pass each (differentiable), the index math + both gathers + the add run
    inside the fused gather kernel (QR "add" with a separate modulus)."""

    def __init__(self, field_dims: Union[List[int], int], hidden_size: int, mode: Optional[str] = None,
                 bucket_size: int = 8000, threshold_init: float = -100.0, threshold_init_method="all-ones",
                 field_name: str = ""):
        super().__init__()
        field_dims = _as_list(field_dims)
        assert mode in [None, "sum", "mean", "max"]
        num_item = sum(field_dims)
        self._field_dims = torch.tensor(field_dims)
        self._mode = mode
        self.field_name: str = field_name
        self.p_weight = nn.Parameter(torch.zeros(bucket_size, hidden_size))
        self.q_weight = nn.Parameter(torch.zeros(bucket_size, hidden_size))
        nn.init.xavier_uniform_(self.p_weight)
        nn.init.xavier_uniform_(self.q_weight)
        self.q_threshold = self.init_threshold("element-wise", threshold_init, bucket_size, hidden_size,
                                               threshold_init_method)
        self.p_threshold = self.init_threshold("element-wise", threshold_init, bucket_size, hidden_size,
                                               threshold_init_method)
        self._num_item = num_item
        self._hidden_size = hidden_size
        self._bucket_size = bucket_size
        self.q_entity_per_row = int(math.ceil(self._num_item / self._bucket_size))
        self.sparse_q_weight = None
        self.sparse_p_weight = None

    @staticmethod
    def init_threshold(threshold_type, init: float, row_size: int, col_size: int,
                       threshold_init_method="all_ones") -> nn.Parameter:
        """Same initialisers as the reference (cerp_embedding.py:76-140)."""
        requires_scaling = True
        if threshold_type == "global":
            mat = torch.ones(1)
            if threshold_init_method == "uniform":
                mat = mat * torch.rand(1)
                requires_scaling = False
            elif threshold_init_method == "normal":
                mat = mat * torch.normal(mean=0.0, std=1.0, size=(1,))
            elif threshold_init_method == "xavier_uniform":
                raise NotImplementedError
            else:
                requires_scaling = False
            if requires_scaling:
                mat = torch.sigmoid(mat)
            return nn.Parameter(mat * init)
        if threshold_type == "element-wise":
            mat = torch.ones([row_size, col_size])
            if threshold_init_method == "uniform":
                mat = mat * torch.nn.init.uniform_(torch.zeros((row_size, col_size)))
            elif threshold_init_method == "normal":
                mat = mat * torch.normal(mean=0.0, std=1.0, size=mat.shape)
            elif threshold_init_method == "xavier_uniform":
                mat = mat * nn.init.xavier_uniform_(torch.zeros(size=mat.shape))
            else:
                requires_scaling = False
            if requires_scaling:
                mat_min, _ = mat.min(dim=1, keepdim=True)
                mat_max, _ = mat.max(dim=1, keepdim=True)
                mat = (mat - mat_min) / (mat_max - mat_min)
            assert (0 <= mat).all() and (1 >= mat).all()
            return nn.Parameter(init * mat)
        raise ValueError("Invalid threshold_type: {}".format(threshold_type))

    def apply_pruning(self):
        self.sparse_q_weight = RF.soft_threshold_table(self.q_weight, self.q_threshold)
        self.sparse_p_weight = RF.soft_threshold_table(self.p_weight, self.p_threshold)

    def _spec(self):
        return RF.LookupSpec(L.KIND_QR_ADD, self._num_item, self._hidden_size, divider=self.q_entity_per_row,
                             modulus=self._bucket_size, module=self)

    def _tensors(self):
        self.apply_pruning()
        return self.sparse_q_weight, self.sparse_p_weight, None

    def _count(self) -> int:
        n = 0
        for w, t in ((self.p_weight, self.p_threshold), (self.q_weight, self.q_threshold)):
            _, cnt = RF.pep_threshold_table(w.detach(), t.detach(), L.PEP_FEATURE_DIM, want_out=False, want_count=True)
            n += int(cnt.item())
        return n

    def get_sparsity(self, get_n_params=False):
        total_params = self._num_item * self._hidden_size
        n_params = self._count()
        if get_n_params:
            return (1 - n_params / total_params), n_params
        return 1 - n_params / total_params

    def get_num_params(self):
        return self._count()

    def get_weight(self):
        return self(torch.arange(self._num_item, device=self.p_weight.device))

    def get_prune_loss(self, K=100):
        emb = self.sparse_p_weight + self.sparse_q_weight
        return -torch.tanh(emb * K).norm(2) ** 2


class RetrainCerpEmbedding(IEmbedding):
    """CERP retrain (cerp_embedding.py:210-378): P, Q re-initialised from `initial.pth`, fixed bool masks
    from the searched checkpoint; the masked tables feed the same fused gather."""

    def __init__(self, field_dims: Union[List[int], int], hidden_size: int, mode: Optional[str],
                 checkpoint_weight_dir: str, field_name: str = "", weight_name: str = "target",
                 bucket_size: int = 8000, sparse: bool = False):
        super().__init__()
        field_dims = _as_list(field_dims)
        mask_weight_path = os.path.join(checkpoint_weight_dir, field_name, f"{weight_name}.pth")
        init_weight_path = os.path.join(checkpoint_weight_dir, field_name, "initial.pth")
        assert os.path.exists(mask_weight_path), f"Weight not found at {mask_weight_path} to re-init mask"
        assert os.path.exists(init_weight_path), f"Weight not found at {init_weight_path} to re-init original weight"
        num_item = sum(field_dims)
        self._field_dims = torch.tensor(field_dims)
        self._mode = mode
        self.field_name: str = field_name
        self._bucket_size = bucket_size
        self._hidden_size = hidden_size
        self.p_weight = nn.Parameter(torch.zeros(bucket_size, hidden_size))
        self.q_weight = nn.Parameter(torch.zeros(bucket_size, hidden_size))
        init_weight = torch.load(init_weight_path)
        self.q_mask, self.p_mask = None, None
        assert init_weight["q_weight"].shape == (bucket_size, hidden_size)
        assert init_weight["p_weight"].shape == (bucket_size, hidden_size)
        self.q_weight.data = init_weight["q_weight"]
        self.p_weight.data = init_weight["p_weight"]
        self.q_mask, self.p_mask = self.load_mask(mask_weight_path)
        self.sparse_q_weight, self.sparse_p_weight = None, None
        self._num_item = num_item
        self.q_entity_per_row = int(math.ceil(self._num_item / self._bucket_size))
        self._sparse = sparse

    def load_mask(self, weight_path: str):
        checkpoint = torch.load(weight_path, map_location="cpu")
        masks = []
        for weight_name, threshold_name in (("q_weight", "q_threshold"), ("p_weight", "p_threshold")):
            mask = (checkpoint[weight_name].abs() - torch.sigmoid(checkpoint[threshold_name])) > 0
            assert mask.shape == (self._bucket_size, self._hidden_size)
            masks.append(nn.Parameter(mask, False))
        return masks

    def _spec(self):
        return RF.LookupSpec(L.KIND_QR_ADD, self._num_item, self._hidden_size, divider=self.q_entity_per_row,
                             modulus=self._bucket_size, module=self)

    def _tensors(self):
        if self.sparse_q_weight is None or self.training:
            self.sparse_q_weight = self.q_weight * self.q_mask
            self.sparse_p_weight = self.p_weight * self.p_mask
        return self.sparse_q_weight, self.sparse_p_weight, None

    def get_weight(self):
        return self(torch.arange(self._num_item, device=self.p_weight.device))

    def get_num_params(self):
        if self.sparse_p_weight is None:
            return (torch.count_nonzero(self.q_mask) + torch.count_nonzero(self.p_mask)).item()
        return (torch.count_nonzero(self.sparse_p_weight) + torch.count_nonzero(self.sparse_q_weight)).item()
