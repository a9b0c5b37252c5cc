"""Drop-in replacement of the reference attention module for ATTN_TYPE='longformerhand'.

`B200Long2DSCSelfAttention` mirrors `Long2DSCSelfAttention`
(src/models/layers/longformer2d.py:12-229): identical constructor signature,
`forward(x, nx, ny)` contract, public attributes (`mode`, `Nglo`, `num_heads`,
`head_dim`, `attention_window`, `only_glo`, `query`, `kv`, `proj`, ...) and
parameter / buffer names, so checkpoints (utils/checkpoint.py:32-41,98-108),
`MsViT.reset_vil_mode` (msvit.py:532-541) and the MAC-counting hook keep working.

The q / kv / proj Linears stay stock PyTorch (north star); everything between
them is ONE fused CUDA operator (`ops.vil_attention`).  There is no CPU path:
calling forward on CPU tensors raises.
"""
from __future__ import annotations

import random

import torch
import torch.nn.functional as F
from torch import nn

from .ops import vil_attention


def relative_position_index(w: int) -> torch.Tensor:
    """(w^2, 9 w^2) int64 index into the ((4w-1)^2, H) bias table - the buffer the reference registers
    (longformer2d.py:68-100), here in closed form.  Column block order: chunk offsets
    (-1,-1),(-1,0),(-1,1),(0,-1),(0,0),(0,1),(1,-1),(1,0),(1,1)."""
    ar = torch.arange(w * w)
    lr, lc = ar // w, ar % w
    cols = []
    for dR in (-1, 0, 1):
        for dC in (-1, 0, 1):
            dr = lr[:, None] - (dR * w + lr[None, :]) + 2 * w - 1
            dc = lc[:, None] - (dC * w + lc[None, :]) + 2 * w - 1
            cols.append(dr * (4 * w - 1) + dc)
    return torch.cat(cols, dim=-1)


class B200Long2DSCSelfAttention(nn.Module):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0., proj_drop=0., w=7, d=1,
                 autoregressive=False, sharew=False, nglo=1, only_glo=False, exact=0, autograd=False, rpe=False,
                 mode=0):
        # NOT super().__init__(): in the drop-in class of `make_dropin_class` the MRO continues into the reference's
        # Long2DSCSelfAttention.__init__(dim, ...), which must not run (it would build a second set of parameters)
        nn.Module.__init__(self)
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = qk_scale or self.head_dim ** -0.5
        self.Nglo = nglo
        self.only_glo = only_glo
        if self.only_glo:
            assert self.Nglo >= 1, "Nglo == 0 in the only global mode!"

        self.query = nn.Linear(dim, dim, bias=qkv_bias)
        self.kv = nn.Linear(dim, dim * 2, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)
        self.sharew = bool(sharew)
        if nglo >= 1:
            if sharew:
                self.query_global, self.kv_global, self.proj_global = self.query, self.kv, self.proj
            else:
                self.query_global = nn.Linear(dim, dim, bias=qkv_bias)
                self.kv_global = nn.Linear(dim, dim * 2, bias=qkv_bias)
                self.proj_global = nn.Linear(dim, dim)

        self.attn_drop = nn.Dropout(attn_drop)
        self.proj_drop = nn.Dropout(proj_drop)
        self.attention_window = w
        self.attention_dilation = d
        self.autoregressive = autoregressive
        assert self.attention_dilation == 1, "Dilation is not supported!"
        assert not self.autoregressive, "Autoregressive is not supported yet!"
        if exact not in (0, 1, -1):
            raise ValueError("longsc exact should be in [0,1,-1]!")
        self.exact = exact
        self.autograd = autograd        # accepted for signature parity; the fused op has one hand-written backward
        self.impl = "auto"              # "auto" | "simt" | "tcgen05" (kernel family; see include/vil_attn.h)

        self.rpe = rpe
        if rpe:
            self.local_relative_position_bias_table = nn.Parameter(torch.zeros((4 * w - 1) * (4 * w - 1), num_heads))
            nn.init.trunc_normal_(self.local_relative_position_bias_table, std=.02)
            if nglo >= 1:
                self.g2l_relative_position_bias = nn.Parameter(torch.zeros(2, num_heads, nglo))
                self.g2g_relative_position_bias = nn.Parameter(torch.zeros(num_heads, nglo, nglo))
                nn.init.trunc_normal_(self.g2l_relative_position_bias, std=.02)
                nn.init.trunc_normal_(self.g2g_relative_position_bias, std=.02)
            # kept only for state_dict compatibility: the kernel derives the index arithmetically
            self.register_buffer("relative_position_index", relative_position_index(w))
        # 0: all 8 neighbour chunks; -1: own chunk only; >0: one random neighbour per training step
        self.mode = mode

    # -- mode selection exactly as longformer2d.py:113-123
    def _pick_mode(self) -> int:
        mode = self.mode
        if self.mode > 0:
            mode = random.randrange(1, 9) if self.training else 0
        return mode

    supports_deferred_bias = True       # forward(..., defer_proj_bias=True) -> (projection without bias, bias)

    @staticmethod
    def _lin(layer, x):
        """`layer(x)` for the q / kv Linears: stock GEMMs, bias gradient by one column-sum kernel (epilogue.py)."""
        from .epilogue import linear_colsum_bias
        return linear_colsum_bias(x, layer.weight, layer.bias)

    def forward(self, x, nx, ny, defer_proj_bias: bool = False):
        """`defer_proj_bias=True` (used by the fused residual epilogue of the harness, SURVEY.md section 8 (f) row 4) returns
        `(out, bias)`: the output projection WITHOUT its bias plus the bias that the caller's residual-add kernel applies
        (`bias` is None when nothing was deferred and `out` is complete).  The default is the reference's contract."""
        if defer_proj_bias:
            can = (not self.only_glo) and (self.Nglo == 0 or self.sharew) and not (self.training and self.proj_drop.p > 0)
            if not can:
                return self.forward(x, nx, ny), None
        B, N, C = x.shape
        Nloc = nx * ny
        g, H = self.Nglo, self.num_heads
        assert g + Nloc == N, "Global dimension does not match!"
        if not x.is_cuda:
            raise RuntimeError("B200Long2DSCSelfAttention only runs on a CUDA (sm_100a) device; there is no CPU "
                               "fallback (use the reference module / oracle for CPU parity checks)")
        if self.attn_drop.p > 0 and self.training:
            raise NotImplementedError("attention dropout > 0 is not supported by the fused kernel "
                                      "(the reference never enables it: build_model does not set attn_drop_rate)")
        if self.only_glo:
            return self._forward_only_glo(x, nx, ny)
        mode = self._pick_mode()
        table = self.local_relative_position_bias_table if self.rpe else None
        g2l = self.g2l_relative_position_bias if (self.rpe and g >= 1) else None
        g2g = self.g2g_relative_position_bias if (self.rpe and g >= 1) else None
        kw = dict(num_heads=H, nx=nx, ny=ny, w=self.attention_window, nglo=g, exact=self.exact, mode=mode,
                  scale=self.scale, impl=self.impl)
        if g >= 1 and self.sharew:
            # one GEMM for local + global queries, the kv GEMM is not recomputed (cf. longformer2d.py:211)
            out = vil_attention(self._lin(self.query, x), self._lin(self.kv, x), None, None, table, g2l, g2g, **kw)
            if defer_proj_bias:
                return F.linear(out, self.proj.weight), self.proj.bias
            return self.proj_drop(self.proj(out))
        if g >= 1:
            out = vil_attention(self._lin(self.query, x[:, g:]), self._lin(self.kv, x), self._lin(self.query_global, x[:, :g]),
                                self._lin(self.kv_global, x), table, g2l, g2g, **kw)
            x0 = self.proj_global(out[:, :g])
            x1 = self.proj(out[:, g:])
            return self.proj_drop(torch.cat((x0, x1), dim=1))
        out = vil_attention(self._lin(self.query, x), self._lin(self.kv, x), None, None, table, None, None, **kw)
        if defer_proj_bias:
            return F.linear(out, self.proj.weight), self.proj.bias
        return self.proj_drop(self.proj(out))

    def _forward_only_glo(self, x, nx, ny):
        """ONLY_GLOBAL ablation (longformer2d.py:130-132,189-192): local queries attend to the global tokens
        only.  Not on the north-star path; plain PyTorch, kept for API completeness."""
        B, N, C = x.shape
        g, H, M = self.Nglo, self.num_heads, self.head_dim
        q = self.scale * self.query(x[:, g:]).reshape(B, N - g, H, M).transpose(1, 2)
        kv = self.kv(x).reshape(B, N, 2, H, M).permute(2, 0, 3, 1, 4)
        k, v = kv[0], kv[1]
        a1 = (q @ k[:, :, :g].transpose(-2, -1)).softmax(dim=-1)
        x1 = self.proj((a1 @ v[:, :, :g]).transpose(1, 2).reshape(B, N - g, C))
        qg = self.scale * self.query_global(x[:, :g]).reshape(B, g, H, M).transpose(1, 2)
        kvg = self.kv_global(x).reshape(B, N, 2, H, M).permute(2, 0, 3, 1, 4)
        a0 = qg @ kvg[0].transpose(-2, -1)
        if self.rpe:
            a0 = a0 + torch.cat([self.g2g_relative_position_bias,
                                 self.g2l_relative_position_bias[0].unsqueeze(-1).expand(-1, -1, N - g)], dim=-1)
        x0 = self.proj_global((a0.softmax(dim=-1) @ kvg[1]).transpose(1, 2).reshape(B, g, C))
        return self.proj_drop(torch.cat((x0, x1), dim=1))

    @staticmethod
    def compute_macs(module, input, output):
        """MAC counter hook with the reference's accounting (longformer2d.py:231-280)."""
        _, T, C = input[0].shape
        g, W = module.Nglo, module.attention_window
        if module.only_glo:
            kq = (C - g) * g * C
        else:
            kq = (C - g) * (9 * W ** 2) * C + (C - g) * g * C
        kq += g * T * C
        macs = 2 * kq
        qkv = sum(p.numel() for p in module.query.parameters()) + sum(p.numel() for p in module.kv.parameters())
        macs += qkv * T + sum(p.numel() for p in module.proj.parameters()) * T
        module.__flops__ += macs


def make_dropin_class(reference_cls):
    """Build a subclass of BOTH the B200 module and the reference `Long2DSCSelfAttention`, so that
    `isinstance(m, Long2DSCSelfAttention)` checks (msvit.py:532-541 `reset_vil_mode`) keep finding it.
    Used by INTEGRATION.md's `elif attn_type == 'longformer_b200'` stub.

    MRO = (B200DropIn, B200Long2DSCSelfAttention, reference_cls, nn.Module): constructor, `forward`, `compute_macs`
    resolve to the B200 module (whose __init__ calls nn.Module.__init__ directly, so the reference constructor never
    runs); the reference class only contributes its identity.  Pinned by tests/test_dropin_reference.py against what
    the unmodified reference MsViT exposes (tests/golden/dropin_reference.pt)."""
    class B200DropIn(B200Long2DSCSelfAttention, reference_cls):
        pass
    B200DropIn.__name__ = B200DropIn.__qualname__ = "B200" + reference_cls.__name__
    return B200DropIn
