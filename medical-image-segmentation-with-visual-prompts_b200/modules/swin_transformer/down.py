"""PatchMerging (reference swin_transformer/down.py:5-59): 2x2x2 (or 2x2x1) strided gather ->
LayerNorm(8C / 4C) -> Linear(no bias).  Adjacent to the hot path (SURVEY §8f-2); kept API- and
state-dict-compatible so ConsecutiveSwinBlocks(down=True) chains stages.  Gather order of the
neighbourhood offsets (dh,dw,dd): 000,100,010,001,110,101,011,111 (:31-39); 00,10,01,11 when the last
axis is not merged (:41-45).  Odd axes get one zero plane on the LOW side (the reference reverses the
flat padding list before F.pad, :26-28, which swaps each (lo,hi) pair)."""
import torch
import torch.nn as nn
import torch.nn.functional as F

_OFFS3 = ((0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, 1, 1))
_OFFS2 = ((0, 0), (1, 0), (0, 1), (1, 1))


class PatchMerging(nn.Module):
    def __init__(self, in_channels, out_channels, merge_last_dim=True):
        super().__init__()
        k = 8 if merge_last_dim else 4
        self.norm = nn.LayerNorm(k * in_channels, eps=1e-6)
        self.reduction = nn.Linear(k * in_channels, out_channels, bias=False)
        self.merge_last_dim = merge_last_dim

    def _norm_reduce(self, t):
        from ... import functional as PF
        t = PF.layer_norm(t, self.norm.weight, self.norm.bias, self.norm.eps)
        return PF.multi_linear(t, None, self.reduction.weight)

    def forward_tokens(self, y, m, geom):
        """Block output tokens y + m in window order `geom` -> merged feature map.  The window reverse, the 2x2x2
        strided slices + cat (:21-47) and the block's last residual add are ONE row gather (csrc/gather.cu)."""
        from ... import functional as PF
        from ...geometry import rowmap_merge
        rm, (h2, w2, d2) = rowmap_merge(geom, bool(self.merge_last_dim))
        b, c = y.shape[0], y.shape[-1]
        k = 8 if self.merge_last_dim else 4
        t = PF.gather_rows(y, m, rm).view(b, h2 * w2 * d2, k * c)
        t = self._norm_reduce(t)
        # same strides as the reference's final rearrange (a permuted view, :48-53)
        return t.view(b, h2, w2, d2, -1).permute(0, 4, 1, 2, 3)

    def forward(self, x):
        from ... import functional as PF
        k = 8 if self.merge_last_dim else 4
        if x.is_cuda and x.dim() == 5 and x.shape[1] > 1 and x.permute(0, 2, 3, 4, 1).is_contiguous() \
                and PF.layer_norm_supported(k * x.shape[1]) and x.dtype in (torch.float32, torch.bfloat16, torch.float16):
            from ...geometry import rowmap_merge_from_voxels
            b, c = x.shape[:2]
            rm, (h2, w2, d2) = rowmap_merge_from_voxels(tuple(int(v) for v in x.shape[2:]), bool(self.merge_last_dim))
            t = PF.gather_rows(x.permute(0, 2, 3, 4, 1).reshape(b, -1, c), None, rm).view(b, h2 * w2 * d2, k * c)
            return self._norm_reduce(t).view(b, h2, w2, d2, -1).permute(0, 4, 1, 2, 3)
        h, w, d = x.shape[2:]
        if h % 2 or w % 2 or d % 2:
            x = F.pad(x, (d % 2, 0, w % 2, 0, h % 2, 0))
        if self.merge_last_dim:
            parts = [x[:, :, a::2, b::2, c::2] for a, b, c in _OFFS3]
        else:
            parts = [x[:, :, a::2, b::2, :] for a, b in _OFFS2]
        t = torch.cat(parts, dim=1).permute(0, 2, 3, 4, 1)             # [B,h/2,w/2,d',kC] channels last
        from ... import functional as PF
        if not t.is_cuda:
            raise RuntimeError("pwa_b200.PatchMerging runs on CUDA (sm_100a) only; there is no CPU path")
        if not PF.layer_norm_supported(t.shape[-1]):
            raise NotImplementedError(f"PatchMerging: {t.shape[-1]} merged channels (need a multiple of 4, at most 2048)")
        t = PF.layer_norm(t.contiguous(), self.norm.weight, self.norm.bias, self.norm.eps)
        t = PF.multi_linear(t, None, self.reduction.weight)
        return t.permute(0, 4, 1, 2, 3)

    def named_parameters_body(self):
        return [*self.reduction.named_parameters(), *self.norm.named_parameters()]
