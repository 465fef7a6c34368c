"""Tensor-level wrappers over the C ABI (include/vitk.h).  Each function takes CUDA tensors,
launches the kernel on torch's current stream and returns/fills tensors; nothing here computes
on the CPU or through ATen — if libvitk is missing these raise.

The operators replaced are the ATen ops HF ViT dispatches (SURVEY.md §2.2); citations are in
include/vitk.h next to each entry point.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import (EPI_ACCUM_F32, EPI_BIAS_BF16, EPI_BIAS_GELU_BF16, EPI_BIAS_GELUG_BF16, EPI_BIAS_RESID_F32,  # noqa: F401
                   EPI_DGELU_BF16, EPI_MUL_BF16, EPI_PATCH_F32, EPI_STORE_BF16, EPI_STORE_F32, GemmArgs)

bf16, f32 = torch.bfloat16, torch.float32


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


_replayed_launches = 0


def launch_count() -> int:
    """Kernels of libvitk launched so far by this process: the library's own counter (one per kernel launch call)
    plus the kernel nodes executed by CUDA-graph replays (counted when the graph was captured)."""
    return int(_lib.lib().vitk_launch_count()) + _replayed_launches


def direct_launch_count() -> int:
    return int(_lib.lib().vitk_launch_count())


def note_graph_replay(kernel_nodes: int) -> None:
    global _replayed_launches
    _replayed_launches += kernel_nodes


def check_device(dev: int = 0) -> None:
    _lib.check(_lib.lib().vitk_check_device(dev), "check_device")


# ----------------------------------------------------------------------------- input
def patchify_u8(gray: torch.Tensor, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5), out: Optional[torch.Tensor] = None):
    """uint8 gray [B,H,W] → bf16 im2col [B·(H/16)·(W/16), 768] (ViT-Training.py:60-66 + HF:166)."""
    assert gray.dtype == torch.uint8 and gray.is_cuda and gray.is_contiguous() and gray.dim() == 3
    B, H, W = gray.shape
    if out is None:
        out = torch.empty((B * (H // 16) * (W // 16), 768), dtype=bf16, device=gray.device)
    m = (C.c_float * 3)(*mean)
    s = (C.c_float * 3)(*std)
    _lib.check(_lib.lib().vitk_patchify_u8(gray.data_ptr(), B, H, W, 16, m, s, out.data_ptr(), _stream()), "patchify_u8")
    return out


def hflip_u8(gray: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """RandomHorizontalFlip on the device (ViT-Training.py:61): uint8 gray [B,H,W] mirrored IN PLACE along W where the
    uint8 / bool mask [B] is non-zero.  Returns ``gray``."""
    assert gray.dtype == torch.uint8 and gray.is_cuda and gray.is_contiguous() and gray.dim() == 3
    assert mask.is_cuda and mask.is_contiguous() and mask.numel() == gray.shape[0] and mask.dtype in (torch.uint8, torch.bool)
    B, H, W = gray.shape
    _lib.check(_lib.lib().vitk_hflip_u8(gray.data_ptr(), mask.data_ptr(), B, H, W, _stream()), "hflip_u8")
    return gray


def patchify_f32(pix: torch.Tensor, out: Optional[torch.Tensor] = None):
    """fp32 NCHW [B,3,H,W] → bf16 im2col [B·P, 768] (collate_fn contract, ViT-Training.py:77-80)."""
    assert pix.dtype == f32 and pix.is_cuda and pix.is_contiguous() and pix.dim() == 4 and pix.shape[1] == 3
    B, _, H, W = pix.shape
    if out is None:
        out = torch.empty((B * (H // 16) * (W // 16), 768), dtype=bf16, device=pix.device)
    _lib.check(_lib.lib().vitk_patchify_f32(pix.data_ptr(), B, H, W, 16, out.data_ptr(), _stream()), "patchify_f32")
    return out


# ----------------------------------------------------------------------------- LayerNorm
def _check_rows(what: str, t: torch.Tensor, M: int, row_stride: int, width: int) -> None:
    # logical row r of a row_stride buffer is physical row r·row_stride of a contiguous [·, width] tensor
    assert t.is_contiguous() and t.numel() >= ((M - 1) * row_stride + 1) * width, \
        f"{what}: needs a contiguous buffer of at least {(M - 1) * row_stride + 1} rows of {width}"


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float,
                  y: Optional[torch.Tensor] = None, mean: Optional[torch.Tensor] = None,
                  rstd: Optional[torch.Tensor] = None, *, row_stride: int = 1) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """LayerNorm of the M rows of ``x`` (fp32, own row stride) into y (bf16) and mean / rstd (fp32).  With
    ``row_stride`` > 1, logical row r goes to physical row r·row_stride of y / mean / rstd — the CLS rows of a
    [B, T, D] buffer stay in place with row_stride = T — and the caller passes all three, sized for the physical rows."""
    M, D = x.shape
    assert x.dtype == f32 and x.stride(1) == 1
    if row_stride != 1:
        assert y is not None and mean is not None and rstd is not None, "layernorm_fwd: row_stride > 1 needs y, mean and rstd"
        _check_rows("layernorm_fwd y", y, M, row_stride, D)
        _check_rows("layernorm_fwd mean", mean, M, row_stride, 1)
        _check_rows("layernorm_fwd rstd", rstd, M, row_stride, 1)
    if y is None:
        y = torch.empty((M, D), dtype=bf16, device=x.device)
    if mean is None:
        mean = torch.empty((M,), dtype=f32, device=x.device)
    if rstd is None:
        rstd = torch.empty((M,), dtype=f32, device=x.device)
    _lib.check(_lib.lib().vitk_layernorm_fwd_rows(x.data_ptr(), x.stride(0), gamma.data_ptr(), beta.data_ptr(), eps, M, D,
                                                   row_stride, y.data_ptr(), mean.data_ptr(), rstd.data_ptr(), _stream()),
               "layernorm_fwd")
    return y, mean, rstd


def layernorm_bwd(dy, x, mean, rstd, gamma, dres, dgamma, dbeta, dx=None, dxsum=None, *, row_stride: int = 1):
    """dx = dres + LNbwd(dy) (bf16); dgamma/dbeta (fp32) are accumulated; dxsum (optional) += Σ_rows dx.
    With ``row_stride`` > 1, logical row r of dy / dres / dx / mean / rstd is physical row r·row_stride (x keeps its
    own row stride), and the caller passes ``dx`` sized for the physical rows."""
    M, D = x.shape
    if row_stride != 1:
        assert dx is not None, "layernorm_bwd: row_stride > 1 needs dx"
        for what, t, width in (("dy", dy, D), ("dres", dres, D), ("dx", dx, D), ("mean", mean, 1), ("rstd", rstd, 1)):
            if t is not None:
                _check_rows(f"layernorm_bwd {what}", t, M, row_stride, width)
    if dx is None:
        dx = torch.empty((M, D), dtype=bf16, device=x.device)
    _lib.check(_lib.lib().vitk_layernorm_bwd_rows(dy.data_ptr(), x.data_ptr(), x.stride(0), mean.data_ptr(), rstd.data_ptr(),
                                                   gamma.data_ptr(), _ptr(dres), M, D, row_stride, dx.data_ptr(),
                                                   dgamma.data_ptr(), dbeta.data_ptr(), _ptr(dxsum), _stream()),
               "layernorm_bwd")
    return dx


# ----------------------------------------------------------------------------- GEMM
def gemm(a: torch.Tensor, b: torch.Tensor, M: int, N: int, K: int, d: torch.Tensor, *, epilogue: int,
         a_mn_major: bool = False, b_mn_major: bool = False, lda: Optional[int] = None, ldb: Optional[int] = None,
         ldd: Optional[int] = None, d2: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
         aux: Optional[torch.Tensor] = None, ld_aux: int = 0, rows_in: int = 0, rows_out: int = 0, row_off: int = 0,
         split_k: int = 0, tile_n: int = 0, max_ctas: int = 0, variant: int = 0) -> torch.Tensor:
    """D[M,N] = A·Bᵀ (logical A [M,K], B [N,K]) on tcgen05 with a fused epilogue; see vitk.h."""
    g = GemmArgs()
    g.a, g.b = a.data_ptr(), b.data_ptr()
    g.M, g.N, g.K = M, N, K
    g.lda = lda if lda is not None else a.stride(0)
    g.ldb = ldb if ldb is not None else b.stride(0)
    g.a_mn_major, g.b_mn_major = int(a_mn_major), int(b_mn_major)
    g.epilogue, g.split_k = epilogue, split_k
    g.d, g.ldd = d.data_ptr(), (ldd if ldd is not None else d.stride(0))
    g.d2 = _ptr(d2)
    g.bias = _ptr(bias)
    g.aux = _ptr(aux)
    g.ld_aux = ld_aux if ld_aux else (aux.stride(0) if aux is not None else 0)
    g.rows_in, g.rows_out, g.row_off = rows_in, rows_out, row_off
    g.tile_n, g.max_ctas, g.variant = tile_n, max_ctas, variant
    _lib.check(_lib.lib().vitk_gemm_bf16(C.byref(g), _stream()), "gemm_bf16")
    return d


def gemm_plan(M: int, N: int, K: int, *, epilogue: int, b_mn_major: bool = False, a_mn_major: bool = False,
              split_k: int = 0, tile_n: int = 0, max_ctas: int = 0, sms: int = 148) -> dict:
    """Host-only: the tiling vitk_gemm_bf16 would pick for this problem on a GPU with ``sms`` SMs (no device needed)."""
    g = GemmArgs()
    g.M, g.N, g.K = M, N, K
    g.a_mn_major, g.b_mn_major = int(a_mn_major), int(b_mn_major)
    g.epilogue, g.split_k, g.tile_n, g.max_ctas = epilogue, split_k, tile_n, max_ctas
    tn, sk, nh, items = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    _lib.check(_lib.lib().vitk_gemm_plan(C.byref(g), sms, C.byref(tn), C.byref(sk), C.byref(nh), C.byref(items)), "gemm_plan")
    return {"tile_n": tn.value, "split_k": sk.value, "n_half": nh.value, "work_items": items.value}


def colsum(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[n] += Σ_m x[m,n]  (bias gradients)."""
    M, N = x.shape
    _lib.check(_lib.lib().vitk_colsum_bf16(x.data_ptr(), M, N, x.stride(0), out.data_ptr(), _stream()), "colsum_bf16")
    return out


# ----------------------------------------------------------------------------- attention
def attn_fwd(qkv: torch.Tensor, B: int, T: int, H: int, scale: float, o: Optional[torch.Tensor] = None,
             lse: Optional[torch.Tensor] = None):
    """qkv bf16 [B,T,3,H,64] → o bf16 [B,T,H·64], lse fp32 [B,H,T]."""
    if o is None:
        o = torch.empty((B * T, H * 64), dtype=bf16, device=qkv.device)
    if lse is None:
        lse = torch.empty((B, H, T), dtype=f32, device=qkv.device)
    _lib.check(_lib.lib().vitk_attn_fwd(qkv.data_ptr(), B, T, H, scale, o.data_ptr(), lse.data_ptr(), _stream()), "attn_fwd")
    return o, lse


def attn_bwd_workspace_bytes(B: int, T: int, H: int) -> int:
    return int(_lib.lib().vitk_attn_bwd_workspace_bytes(B, T, H))


def attn_bwd(qkv, o, do, lse, B: int, T: int, H: int, scale: float, dqkv: Optional[torch.Tensor] = None,
             workspace: Optional[torch.Tensor] = None):
    if dqkv is None:
        dqkv = torch.empty((B * T, 3 * H * 64), dtype=bf16, device=qkv.device)
    if workspace is None:
        workspace = torch.empty((attn_bwd_workspace_bytes(B, T, H),), dtype=torch.uint8, device=qkv.device)
    _lib.check(_lib.lib().vitk_attn_bwd(qkv.data_ptr(), o.data_ptr(), do.data_ptr(), lse.data_ptr(), B, T, H, scale,
                                         dqkv.data_ptr(), workspace.data_ptr(), _stream()), "attn_bwd")
    return dqkv


def attn_cls_fwd(qkv: torch.Tensor, B: int, T: int, H: int, scale: float, o: torch.Tensor, lse: torch.Tensor):
    """Attention of the CLS query only (top encoder layer): writes o[b,0,:] and lse[b,:,0]."""
    _lib.check(_lib.lib().vitk_attn_cls_fwd(qkv.data_ptr(), B, T, H, scale, o.data_ptr(), lse.data_ptr(), _stream()), "attn_cls_fwd")
    return o, lse


def attn_cls_bwd(qkv, o, do, lse, B: int, T: int, H: int, scale: float, dqkv: Optional[torch.Tensor] = None):
    """Backward of attn_cls_fwd: reads do / o at token 0 only; dqkv dense (dQ zero except token 0)."""
    if dqkv is None:
        dqkv = torch.empty((B * T, 3 * H * 64), dtype=bf16, device=qkv.device)
    _lib.check(_lib.lib().vitk_attn_cls_bwd(qkv.data_ptr(), o.data_ptr(), do.data_ptr(), lse.data_ptr(), B, T, H, scale,
                                             dqkv.data_ptr(), _stream()), "attn_cls_bwd")
    return dqkv


# ----------------------------------------------------------------------------- embeddings glue
def embed_cls(cls: torch.Tensor, pos: torch.Tensor, B: int, T: int, D: int, h: torch.Tensor):
    _lib.check(_lib.lib().vitk_embed_cls(cls.data_ptr(), pos.data_ptr(), B, T, D, h.data_ptr(), _stream()), "embed_cls")
    return h


def embed_bwd(dh, B: int, T: int, D: int, dpos, dcls, dbias, dpatch):
    _lib.check(_lib.lib().vitk_embed_bwd(dh.data_ptr(), B, T, D, dpos.data_ptr(), dcls.data_ptr(), dbias.data_ptr(),
                                          dpatch.data_ptr(), _stream()), "embed_bwd")
    return dpatch


# ----------------------------------------------------------------------------- head + loss
def head_fwd(h, B: int, T: int, D: int, Cn: int, gamma, beta, eps: float, Wc, bc, labels, logits, loss, dlogits,
             mean, rstd):
    _lib.check(_lib.lib().vitk_head_fwd(h.data_ptr(), B, T, D, Cn, gamma.data_ptr(), beta.data_ptr(), eps, Wc.data_ptr(),
                                         bc.data_ptr(), _ptr(labels), logits.data_ptr(), _ptr(loss), _ptr(dlogits),
                                         _ptr(mean), _ptr(rstd), _stream()), "head_fwd")


def head_bwd(h, mean, rstd, gamma, beta, Wc, B: int, T: int, D: int, Cn: int, dlogits, dloss, dh, dWc, dbc, dgamma, dbeta):
    _lib.check(_lib.lib().vitk_head_bwd(h.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                         Wc.data_ptr(), B, T, D, Cn, dlogits.data_ptr(), _ptr(dloss), dh.data_ptr(),
                                         dWc.data_ptr(), dbc.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), _stream()),
               "head_bwd")


def multilabel_counts(logits: torch.Tensor, labels: torch.Tensor, counts: torch.Tensor, threshold: float = 0.5):
    """counts[c] += (TP, FP, FN, TN) of sigmoid(logits) >= threshold against {0,1} labels (ViT-Training.py:112-118)."""
    B, Cn = logits.shape
    assert logits.dtype == f32 and labels.dtype == f32 and labels.shape == logits.shape and logits.is_contiguous() and \
        labels.is_contiguous() and counts.dtype == torch.int64 and counts.shape == (Cn, 4) and counts.is_contiguous()
    _lib.check(_lib.lib().vitk_multilabel_counts(logits.data_ptr(), labels.data_ptr(), B, Cn, threshold, counts.data_ptr(),
                                                  _stream()), "multilabel_counts")
    return counts


# ----------------------------------------------------------------------------- misc / optimizer
def cast_f32_bf16(src: torch.Tensor, dst: torch.Tensor):
    _lib.check(_lib.lib().vitk_cast_f32_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()), "cast_f32_bf16")
    return dst


def fill_zero(t: torch.Tensor):
    _lib.check(_lib.lib().vitk_fill_zero(t.data_ptr(), t.numel() * t.element_size(), _stream()), "fill_zero")
    return t


def adamw(p, g, m, v, p16, n: int, lr: float, beta1: float, beta2: float, eps: float, wd: float, bc1: float, bc2: float,
          grad_scale: Optional[torch.Tensor] = None, zero_grad: bool = False, bias_corr_dev: Optional[torch.Tensor] = None):
    _lib.check(_lib.lib().vitk_adamw(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), _ptr(p16), n, lr, beta1, beta2,
                                      eps, wd, bc1, bc2, _ptr(grad_scale), int(zero_grad), _ptr(bias_corr_dev), _stream()), "adamw")


def adamw_tick(step_dev: torch.Tensor, increment: bool, beta1: float, beta2: float, bias_corr_dev: torch.Tensor):
    """Device-side AdamW step counter (int64 [1]) → bias corrections (fp32 [2]) for graph replay."""
    assert step_dev.dtype == torch.int64 and bias_corr_dev.dtype == f32 and bias_corr_dev.numel() >= 2
    _lib.check(_lib.lib().vitk_adamw_tick(step_dev.data_ptr(), int(increment), beta1, beta2, bias_corr_dev.data_ptr(), _stream()),
               "adamw_tick")


_sumsq_scratch = {}


def sumsq(x: torch.Tensor, out: torch.Tensor, scratch: Optional[torch.Tensor] = None):
    """out[0] += Σ x², in a fixed summation order (bit-reproducible).  ``scratch``: zero-initialised fp32 buffer of
    ``vitk_sumsq_scratch_floats()`` elements; one per device is kept here when none is given."""
    if scratch is None:
        scratch = _sumsq_scratch.get(x.device)
        if scratch is None:
            scratch = _sumsq_scratch[x.device] = torch.zeros(int(_lib.lib().vitk_sumsq_scratch_floats()), dtype=f32, device=x.device)
    _lib.check(_lib.lib().vitk_sumsq_f32(x.data_ptr(), x.numel(), out.data_ptr(), scratch.data_ptr(), _stream()), "sumsq_f32")


def shard_mean(own: torch.Tensor, peers: Optional[torch.Tensor], peer_stride: int, n_peers: int, inv_world: float, max_ctas: int = 0):
    """own[i] = (own[i] + Σ_p peers[p·peer_stride + i]) · inv_world  (owner's step of the peer-memory gradient all-reduce)."""
    _lib.check(_lib.lib().vitk_shard_mean(own.data_ptr(), _ptr(peers), own.numel(), peer_stride, n_peers, inv_world, max_ctas,
                                           _stream()), "shard_mean")


def clip_scale(sumsq_t: torch.Tensor, max_norm: float, scale: torch.Tensor):
    _lib.check(_lib.lib().vitk_clip_scale(sumsq_t.data_ptr(), max_norm, scale.data_ptr(), _stream()), "clip_scale")
