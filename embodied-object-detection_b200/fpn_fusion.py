"""Memory read + projection + weighted fusion behind the reference's backbone call surface.

Mirrors the memory block of ``CustomRecurrentFPN`` (detic/modeling/backbone/timm.py:54-213):
  * parameters ``map_merge_projection{1,2,3}`` = Conv2d(512, 256, 1, bias=True) (timm.py:78-86) - same
    state-dict names, so reference checkpoints load and the 'map_merge' LR/un-freeze rules keep matching;
  * ``forward(x, map_memory, proj_indices, observations, sequence_name=None) -> (features dict, map_memory[0])``
    (timm.py:91,213);
  * MODEL.MEMORY_TYPE image_only | implicit_memory, MODEL.MAP_FEAT_FUSION sum | mem_only | image_only,
    MODEL.MAP_FEATURE_WEIGHT (timm.py:142,177-186).

The gather -> avg-pool 4 -> (avg-pool 2 -> half) x3 chain runs as ONE kernel (eod_read_pool).  In inference the
1x1 projection, the ``* weight`` and the ``+ res`` run as ONE tensor-core kernel per level (eod_project_fuse: fp16
levels x hi/lo-split fp32 weights on tcgen05, fp32-GEMM accuracy).  When gradients are needed (training un-freezes the
``map_merge`` parameters, custom_rcnn.py:609-613) the projection is the tcgen05 row GEMM eod_linear_rows (3xTF32, fp32 accuracy) under
autograd - its forward and both gradient GEMMs - and the epilogue is eod_fuse with a hand-written backward.  The dense backbone itself is out of scope and supplied by the caller.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import torch
import torch.nn as nn

from . import ops
from ._lib import FUSE_IMAGE_ONLY, FUSE_MEM_ONLY, FUSE_SUM

_FUSE_MODES = {"sum": FUSE_SUM, "mem_only": FUSE_MEM_ONLY, "image_only": FUSE_IMAGE_ONLY}


class _LinearFn(torch.autograd.Function):
    """y = x @ W^T + b on the tensor cores with fp32 accuracy (eod_linear_rows, 3xTF32) and its backward: the forward and both gradient
    GEMMs are the same kernel fed with transposed VIEWS (the kernel takes any strides), the bias gradient is a column sum."""

    @staticmethod
    def forward(ctx, x2d, weight, bias):
        ctx.save_for_backward(x2d, weight)
        ctx.has_bias = bias is not None
        return ops.linear_rows(x2d, weight, bias)

    @staticmethod
    def backward(ctx, g):
        x2d, weight = ctx.saved_tensors
        g = g.contiguous()
        g_x = ops.linear_rows(g, weight.t()) if ctx.needs_input_grad[0] else None                    # (M,N) @ (N,K)
        g_w = ops.linear_rows(g.t(), x2d.t()) if ctx.needs_input_grad[1] else None                    # (N,M) @ (M,K)
        g_b = g.sum(0) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return g_x, g_w, g_b


class _FuseFn(torch.autograd.Function):
    """eod_fuse with its backward: out = res + w * mem | w * mem  =>  d res = g (sum only), d mem = w * g."""

    @staticmethod
    def forward(ctx, res, mem, weight: float, mode: int):
        ctx.weight, ctx.mode = weight, mode
        return ops.fuse(res, mem, weight, mode)

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        g_res = g if (ctx.mode == FUSE_SUM and ctx.needs_input_grad[0]) else None
        g_mem = ops.fuse(None, g, ctx.weight, FUSE_MEM_ONLY) if ctx.needs_input_grad[1] else None
        return g_res, g_mem, None, None


class MemoryFusion(nn.Module):
    def __init__(self, memory_type: str = "implicit_memory", fusion: str = "sum", map_feature_weight: float = 500.0,
                 memory_feature_weight: float = 100.0, merge_type: str = "", mem_feat_dim: int = 512,
                 ego_feat_dim: int = 256, tensor_core: bool = True):
        super().__init__()
        self.tensor_core = tensor_core      # False: the row GEMM (eod_linear_rows, 3xTF32) + eod_fuse also in inference, instead of the fused fp16-split launch
        self.validate_indices = True        # range-check proj_indices against the memory table before the gather
        self._w_split = {}                  # level -> ((weight ptr, version), (2N,K) f16 hi/lo split)
        self.memory_type, self.feat_fusion, self.merge_type = memory_type, fusion, merge_type
        self.map_feature_weight, self.memory_feature_weight = map_feature_weight, memory_feature_weight
        self.memory_dim = mem_feat_dim
        if memory_type == "implicit_memory":
            self.map_merge_projection1 = nn.Conv2d(mem_feat_dim, ego_feat_dim, kernel_size=1, bias=True)
            self.map_merge_projection2 = nn.Conv2d(mem_feat_dim, ego_feat_dim, kernel_size=1, bias=True)
            self.map_merge_projection3 = nn.Conv2d(mem_feat_dim, ego_feat_dim, kernel_size=1, bias=True)

    @property
    def merge_map_projections(self) -> List[nn.Conv2d]:
        return [self.map_merge_projection1, self.map_merge_projection2, self.map_merge_projection3]

    def read(self, map_memory: Sequence[torch.Tensor], proj_indices: Sequence[torch.Tensor],
             observations: Optional[Sequence[Optional[torch.Tensor]]] = None) -> List[torch.Tensor]:
        """timm.py:144-168 -> three (B, C, h_l, w_l) fp16 tensors.  map_memory[i]: (cells, C) fp16 normalised table
        (reference API) or fp32 sums with observations[i] (normalisation fused into the kernel)."""
        per_image = []
        for i, mem in enumerate(map_memory):
            counts = None
            if mem.dtype == torch.float32 and observations is not None and observations[i] is not None:
                counts = observations[i].to(torch.float32).unsqueeze(0).contiguous()
            idx = proj_indices[i]
            if idx.dim() == 3 and idx.shape[-1] == 1:
                idx = idx.squeeze(2)
            idx = idx.unsqueeze(0).contiguous()
            if self.validate_indices:                     # the reference's gather raises on a bad id (timm.py:147)
                ops.check_indices(idx, mem.shape[0])
            per_image.append(ops.read_pool(mem.unsqueeze(0).contiguous(), counts, idx))
        if len(per_image) == 1:
            return per_image[0]
        return [torch.cat([lv[k] for lv in per_image], dim=0) for k in range(3)]

    def read_roi(self, map_memory, proj_indices, boxes: Sequence[torch.Tensor], observations=None, pooled: int = 7,
                 project: bool = False) -> torch.Tensor:
        """Optional per-proposal path (BASELINE north star, subsystem 3): the map feature of every proposal box =
        ROIAlign(7x7, aligned, FPN level assignment: detic_roi_heads.py:331-334) of the pooled memory levels.  boxes: one (n_i,4)
        XYXY tensor per image, as ``[x.proposal_boxes.tensor for x in proposals]``.  -> (sum n_i, C_mem, 7, 7) fp32.
        project=True applies ``map_merge_projection_l`` of each box's level and ``* MAP_FEATURE_WEIGHT`` per bin, i.e. returns
        exactly the memory term of ``box_pooler(fused levels)``: by linearity box_pooler(p_l) = box_pooler(res_l) + this.
        Cheaper than pooling the fused levels only while 49 * (number of proposals) stays below the 6 300 level pixels."""
        levels = self.read(map_memory, proj_indices, observations)
        dev = levels[0].device
        bx = torch.cat([b.to(dev, torch.float32) for b in boxes], 0).contiguous()
        bi = torch.cat([torch.full((b.shape[0],), i, dtype=torch.int32, device=dev) for i, b in enumerate(boxes)], 0)
        roi, lvl, valid = ops.read_roi(levels, bx, bi, pooled, want_levels=True, want_valid=True)
        if not project:
            return roi
        # a box without a level (lvl -1) pools nothing from the fused levels either: its memory term is zero
        out = torch.zeros((roi.shape[0], self.merge_map_projections[0].weight.shape[0], pooled, pooled), dtype=torch.float32, device=dev)
        for k, conv in enumerate(self.merge_map_projections):
            sel = (lvl == k).nonzero().squeeze(1)
            if sel.numel():
                x = roi[sel].permute(0, 2, 3, 1)                                              # (n, 7, 7, C)
                w2 = conv.weight.detach().to(torch.float32).reshape(conv.weight.shape[0], -1)
                b2 = None if conv.bias is None else conv.bias.detach().to(torch.float32).contiguous()
                y = ops.linear_rows(x.reshape(-1, x.shape[-1]), w2, None, float(self.map_feature_weight))   # x.W * MAP_FEATURE_WEIGHT
                if b2 is not None:
                    # the reference adds the bias per level pixel BEFORE the pooling, so it survives with the bin's share of sample points
                    # that lie on the level (1 for boxes inside the image, 0 for an empty box - whose pooled features are all zero)
                    y.addcmul_(valid[sel].reshape(-1, 1), b2.view(1, -1), value=float(self.map_feature_weight))
                out[sel] = y.view(x.shape[0], pooled, pooled, -1).permute(0, 3, 1, 2)
        return out

    def fuse_roi(self, box_features: torch.Tensor, map_memory, proj_indices, boxes: Sequence[torch.Tensor], observations=None) -> torch.Tensor:
        """North-star subsystem (4) at the ROI level: the ROI box-head input with the memory fused in.  box_features (sum n_i, C_ego, P, P)
        = ``box_pooler(image-only levels, boxes)`` (detic_roi_heads.py:331-334 on the un-fused FPN output); returns what the reference's
        ``box_pooler(fused levels, boxes)`` holds: by linearity of ROIAlign, box_features + MAP_FEATURE_WEIGHT * (conv1x1_l(pool(L_l)) + b_l)
        ('sum'), the memory term alone ('mem_only'), or box_features unchanged ('image_only' / no memory)."""
        if self.memory_type != "implicit_memory" or self.feat_fusion == "image_only":
            return box_features
        if self.feat_fusion not in _FUSE_MODES:
            raise UnboundLocalError("new_res")
        P = box_features.shape[-1]
        mem = self.read_roi(map_memory, proj_indices, boxes, observations, pooled=P, project=True)         # already times MAP_FEATURE_WEIGHT
        if self.feat_fusion == "mem_only":
            return mem.to(box_features.dtype)
        res = box_features.to(mem.device, torch.float32).contiguous()
        return ops.fuse(res, mem.contiguous(), 1.0, FUSE_SUM).to(box_features.dtype)

    def forward(self, results: Sequence[torch.Tensor], map_memory, proj_indices, observations=None) -> List[torch.Tensor]:
        """results = [p3, p4, p5] -> fused [p3, p4, p5] (timm.py:142-192)."""
        if self.memory_type != "implicit_memory":
            return list(results)
        if self.feat_fusion not in _FUSE_MODES:
            raise UnboundLocalError("new_res")        # the reference leaves new_res unbound here (timm.py:181-189)
        mode = _FUSE_MODES[self.feat_fusion]
        if self.feat_fusion == "image_only":
            return list(results)
        levels = self.read(map_memory, proj_indices, observations)
        convs = self.merge_map_projections
        N, K = convs[0].weight.shape[0], convs[0].weight.shape[1]
        needs_grad = torch.is_grad_enabled() and (any(r.requires_grad for r in results) or any(p.requires_grad for p in self.parameters()))
        if self.tensor_core and not needs_grad and N % 128 == 0 and K % 64 == 0:
            # inference: projection, scaling and sum of all three levels in ONE persistent tcgen05 launch
            for k, conv in enumerate(convs):
                key = (conv.weight.data_ptr(), conv.weight._version)
                if self._w_split.get(k, (None,))[0] != key:
                    self._w_split[k] = (key, ops.project_split_weights(conv.weight.detach().to(torch.float32).contiguous()))
            biases = [None if c.bias is None else c.bias.detach().to(torch.float32).contiguous() for c in convs]
            res32 = [r.detach().to(torch.float32).contiguous() for r in results[:3]] if mode == FUSE_SUM else None
            fused = ops.project_fuse_levels(levels, [self._w_split[k][1] for k in range(3)], biases, res32, float(self.map_feature_weight), mode)
            return [f.to(r.dtype) for f, r in zip(fused, results)]
        out = []
        for k, (lvl, res, conv) in enumerate(zip(levels, results, convs)):
            # timm.py:174: 1x1 conv in fp32 (eval, no autocast) == per-pixel GEMM on the channels-last level
            x = lvl.permute(0, 2, 3, 1).to(torch.float32)                             # (B, h, w, C) contiguous
            w2 = conv.weight.to(torch.float32).reshape(conv.weight.shape[0], -1)
            b2 = None if conv.bias is None else conv.bias.to(torch.float32)
            mem = _LinearFn.apply(x.reshape(-1, x.shape[-1]), w2, b2).view(x.shape[0], x.shape[1], x.shape[2], -1)
            mem = mem.permute(0, 3, 1, 2).contiguous()                               # NCHW like res
            res32 = res.to(torch.float32).contiguous()
            fused = _FuseFn.apply(res32, mem, float(self.map_feature_weight), mode)
            out.append(fused.to(res.dtype))
        return out


class CustomRecurrentFPN(nn.Module):
    """Backbone wrapper with the reference's forward signature (timm.py:91-213).  ``fpn_body(x)`` is the
    caller's stock bottom-up + FPN returning ([p3, p4, p5], aux) ; ``top_block(p5)`` returns [p6, p7]."""

    def __init__(self, fpn_body: Callable, top_block: Optional[Callable], fusion: MemoryFusion,
                 out_features=("p3", "p4", "p5", "p6", "p7")):
        super().__init__()
        self.fpn_body, self.top_block = fpn_body, top_block
        # ``fusion`` is held OUTSIDE the module tree: its three 1x1 convs are registered once, directly on the backbone under
        # the reference's state-dict names (timm.py:78-86), so state_dict() carries exactly `map_merge_projection{1,2,3}.*`
        # and a reference checkpoint loads with strict=True (no duplicate `fusion.*` keys)
        object.__setattr__(self, "fusion", fusion)
        self._out_features = list(out_features)
        if fusion.memory_type == "implicit_memory":
            self.map_merge_projection1 = fusion.map_merge_projection1
            self.map_merge_projection2 = fusion.map_merge_projection2
            self.map_merge_projection3 = fusion.map_merge_projection3

    def forward(self, x, map_memory, proj_indices, observations, sequence_name=None):
        results = self.fpn_body(x)
        results = self.fusion(results, map_memory, proj_indices, observations)
        if self.top_block is not None:
            results = list(results) + list(self.top_block(results[-1]))
        return {f: r for f, r in zip(self._out_features, results)}, map_memory[0]
