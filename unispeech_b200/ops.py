"""Tensor-level wrappers over the C ABI (one Python function per `b200s_*` entry point).

All tensors are CUDA tensors owned by the caller; outputs are passed in (the library never allocates).  A "rows view"
is described by (tensor, batch_stride, row_stride) in elements so padded / strided / overlapping activations can be
addressed without copies.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L

i32 = int      # (argtypes are declared once in _lib: plain Python numbers go straight to the C call)
f32 = float


def _s():
    return L.stream_ptr()


class Profiler:
    """Per-op CUDA-event timing of one step (bench.py): every C-ABI call is bracketed by events on the launch stream."""

    def __init__(self):
        self.records = []

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, flops, nbytes, e0, e1 in self.records:
            d = out.setdefault(name, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "calls": 0})
            d["ms"] += e0.elapsed_time(e1)
            d["flops"] += flops
            d["bytes"] += nbytes
            d["calls"] += 1
        return out


_profiler: Optional[Profiler] = None


def set_profiler(p: Optional[Profiler]):
    global _profiler
    _profiler = p


def _call(name, *args, flops=0.0, nbytes=0.0):
    """`flops` / `nbytes`: ALGORITHMIC work of the call (logical tensors read / written once), recorded by the step profiler."""
    if _profiler is None:
        return L.call(name, *args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    L.call(name, *args)
    e1.record()
    _profiler.records.append((name[len("b200s_"):], flops, nbytes, e0, e1))


# ------------------------------------------------------------------------------------------------- GEMM family
def gemm_rows(a, a_bs, a_rs, rows, batches, K, w, N, out, out_bs, out_ld, epi: Optional[L.Epilogue] = None, valid=None):
    """`valid` (int32 [batches] on the device): ragged batch -- M tiles beyond an utterance's valid frames are zero-filled."""
    if valid is not None:
        return _call("b200s_gemm_rows_ragged", L.ptr(a), L.ll(a_bs), L.ll(a_rs), i32(rows), i32(batches), i32(K), L.ptr(w), i32(N),
                     L.ptr(out), L.ll(out_bs), L.ll(out_ld), C.addressof(epi) if epi is not None else None, L.ptr(valid), _s(),
                     flops=2.0 * rows * batches * K * N)
    _call("b200s_gemm_rows", L.ptr(a), L.ll(a_bs), L.ll(a_rs), i32(rows), i32(batches), i32(K), L.ptr(w), i32(N),
           L.ptr(out), L.ll(out_bs), L.ll(out_ld), C.addressof(epi) if epi is not None else None, _s(),
          flops=2.0 * rows * batches * K * N)


def gemm_wgrad(y, y_bs, y_rs, x, x_bs, x_rs, rows, batches, N, K, dw, dw_ld, valid=None):
    """`valid` (int32 [batches] on the device): ragged batch -- row blocks beyond an utterance's valid frames are skipped."""
    if valid is not None:
        return _call("b200s_gemm_wgrad_ragged", L.ptr(y), L.ll(y_bs), L.ll(y_rs), L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(rows),
                     i32(batches), i32(N), i32(K), L.ptr(dw), L.ll(dw_ld), L.ptr(valid), _s(), flops=2.0 * rows * batches * K * N)
    _call("b200s_gemm_wgrad", L.ptr(y), L.ll(y_bs), L.ll(y_rs), L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(rows),
           i32(batches), i32(N), i32(K), L.ptr(dw), L.ll(dw_ld), _s(), flops=2.0 * rows * batches * K * N)


def posconv_gemm(xpad, xpad_bs, T, B, D, G, taps, wp, out, out_bs, out_ld, epi=None):
    _call("b200s_posconv_gemm", L.ptr(xpad), L.ll(xpad_bs), i32(T), i32(B), i32(D), i32(G), i32(taps), L.ptr(wp),
           L.ptr(out), L.ll(out_bs), L.ll(out_ld), C.addressof(epi) if epi is not None else None, _s(),
          flops=2.0 * T * B * D * (D // G) * taps)


def posconv_wgrad(dy, dy_bs, dy_rs, xpad, xpad_bs, T, B, D, G, taps, dwp):
    _call("b200s_posconv_wgrad", L.ptr(dy), L.ll(dy_bs), L.ll(dy_rs), L.ptr(xpad), L.ll(xpad_bs), i32(T), i32(B),
           i32(D), i32(G), i32(taps), L.ptr(dwp), _s(), flops=2.0 * T * B * D * (D // G) * taps)


# ------------------------------------------------------------------------------------------------- row kernels
def reserve_sms(n: int):
    """SMs the persistent GEMM kernels leave free for a concurrent collective (see parallel.configure_overlap)."""
    _call("b200s_reserve_sms", i32(n))


def layer_norm_fwd(x, x_bs, x_rs, gamma, beta, y, y_bs, y_rs, mean, rstd, rows_per_batch, batches, D, gelu=False, valid=None):
    """`valid` (int32 [batches], device): ragged batch, rows at or beyond valid[b] are padding (written as zeros, not read)."""
    nb = 2.0 * 2 * rows_per_batch * batches * D
    if valid is None:
        _call("b200s_layer_norm_fwd", L.ptr(x), L.ll(x_bs), L.ll(x_rs), L.ptr(gamma), L.ptr(beta), L.ptr(y), L.ll(y_bs),
              L.ll(y_rs), L.ptr(mean), L.ptr(rstd), i32(rows_per_batch), i32(batches), i32(D), i32(1 if gelu else 0), _s(),
              nbytes=nb)
    else:
        _call("b200s_layer_norm_fwd_ragged", L.ptr(x), L.ll(x_bs), L.ll(x_rs), L.ptr(gamma), L.ptr(beta), L.ptr(y), L.ll(y_bs),
              L.ll(y_rs), L.ptr(mean), L.ptr(rstd), i32(rows_per_batch), i32(batches), i32(D), i32(1 if gelu else 0),
              L.ptr(valid), _s(), nbytes=nb)


def layer_norm_gate_fwd(x, x_bs, x_rs, gamma, beta, y, y_bs, y_rs, mean, rstd, T, B, D, grep_w, grep_b, grep_a, H, gate,
                        valid=None):
    nb = 2.0 * 2 * T * B * D
    if valid is None:
        _call("b200s_layer_norm_gate_fwd", L.ptr(x), L.ll(x_bs), L.ll(x_rs), L.ptr(gamma), L.ptr(beta), L.ptr(y), L.ll(y_bs),
              L.ll(y_rs), L.ptr(mean), L.ptr(rstd), i32(T), i32(B), i32(D), L.ptr(grep_w), L.ptr(grep_b), L.ptr(grep_a), i32(H),
              L.ptr(gate), _s(), nbytes=nb)
    else:
        _call("b200s_layer_norm_gate_fwd_ragged", L.ptr(x), L.ll(x_bs), L.ll(x_rs), L.ptr(gamma), L.ptr(beta), L.ptr(y),
              L.ll(y_bs), L.ll(y_rs), L.ptr(mean), L.ptr(rstd), i32(T), i32(B), i32(D), L.ptr(grep_w), L.ptr(grep_b),
              L.ptr(grep_a), i32(H), L.ptr(gate), L.ptr(valid), _s(), nbytes=nb)


def layer_norm_bwd(dy, dy_bs, dy_rs, x, x_bs, x_rs, mean, rstd, gamma, beta, dres, dres_bs, dres_rs, dx, dx_bs, dx_rs,
                   dgamma, dbeta, colsum, rows_per_batch, batches, D, gelu=False, valid=None):
    nb = (4.0 if dres is not None else 3.0) * 2 * rows_per_batch * batches * D
    head = (L.ptr(dy), L.ll(dy_bs), L.ll(dy_rs), L.ptr(x), L.ll(x_bs), L.ll(x_rs), L.ptr(mean), L.ptr(rstd), L.ptr(gamma),
            L.ptr(beta), L.ptr(dres), L.ll(dres_bs), L.ll(dres_rs), L.ptr(dx), L.ll(dx_bs), L.ll(dx_rs), L.ptr(dgamma),
            L.ptr(dbeta), L.ptr(colsum), i32(rows_per_batch), i32(batches), i32(D), i32(1 if gelu else 0))
    if valid is None:
        _call("b200s_layer_norm_bwd", *head, _s(), nbytes=nb)
    else:
        _call("b200s_layer_norm_bwd_ragged", *head, L.ptr(valid), _s(), nbytes=nb)


def colsum(x, x_bs, x_rs, rows_per_batch, batches, N, out, valid=None):
    nb = 2.0 * rows_per_batch * batches * N
    if valid is None:
        _call("b200s_colsum", L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(rows_per_batch), i32(batches), i32(N), L.ptr(out), _s(),
              nbytes=nb)
    else:
        _call("b200s_colsum_ragged", L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(rows_per_batch), i32(batches), i32(N), L.ptr(out),
              L.ptr(valid), _s(), nbytes=nb)


def dgelu_mul(dy, dy_bs, dy_rs, pre, pre_bs, pre_rs, out, out_bs, out_rs, rows_per_batch, batches, N, colsum_out=None,
              pre_is_grad=False):
    _call("b200s_dgelu_mul_ex", L.ptr(dy), L.ll(dy_bs), L.ll(dy_rs), L.ptr(pre), L.ll(pre_bs), L.ll(pre_rs), L.ptr(out),
           L.ll(out_bs), L.ll(out_rs), i32(rows_per_batch), i32(batches), i32(N), L.ptr(colsum_out),
           i32(1 if pre_is_grad else 0), _s())


def frame_mask_fwd(x, x_bs, x_rs, T, B, D, mask, pad, mask_emb):
    _call("b200s_frame_mask_fwd", L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(T), i32(B), i32(D), L.ptr(mask), L.ptr(pad),
           L.ptr(mask_emb), _s())


def frame_mask_bwd(dx, x_bs, x_rs, T, B, D, mask, pad, dmask_emb):
    _call("b200s_frame_mask_bwd", L.ptr(dx), L.ll(x_bs), L.ll(x_rs), i32(T), i32(B), i32(D), L.ptr(mask), L.ptr(pad),
           L.ptr(dmask_emb), _s())


def gate_fwd(x, x_bs, x_rs, T, B, H, grep_w, grep_b, grep_a, gate):
    _call("b200s_gate_fwd", L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(T), i32(B), i32(H), L.ptr(grep_w), L.ptr(grep_b),
           L.ptr(grep_a), L.ptr(gate), _s())


def gate_bwd(x, x_bs, x_rs, T, B, H, grep_w, grep_b, grep_a, dgate, dxg, dx_bs, dx_rs, dgrep_w, dgrep_b, dgrep_a, valid=None):
    head = (L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(T), i32(B), i32(H), L.ptr(grep_w), L.ptr(grep_b), L.ptr(grep_a), L.ptr(dgate),
            L.ptr(dxg), L.ll(dx_bs), L.ll(dx_rs), L.ptr(dgrep_w), L.ptr(dgrep_b), L.ptr(dgrep_a))
    nb = 2.0 * 2 * T * B * H * 64
    if valid is None:
        _call("b200s_gate_bwd", *head, _s(), nbytes=nb)
    else:
        _call("b200s_gate_bwd_ragged", *head, L.ptr(valid), _s(), nbytes=nb)


def relpos_table_fwd(emb, lut, n, H, tab):
    _call("b200s_relpos_table_fwd", L.ptr(emb), L.ptr(lut), i32(n), i32(H), L.ptr(tab), _s())


def relpos_table_bwd(dtab, lut, n, H, demb):
    _call("b200s_relpos_table_bwd", L.ptr(dtab), L.ptr(lut), i32(n), i32(H), L.ptr(demb), _s())


# ------------------------------------------------------------------------------------------------- conv layer 0
def conv0_fwd(wav, L_, B, T, Cc, k, s, w, gamma, beta, mode, stats, fmean, frstd, out, out_bs):
    _call("b200s_conv0_fwd", L.ptr(wav), L.ll(L_), i32(B), i32(T), i32(Cc), i32(k), i32(s), L.ptr(w), L.ptr(gamma),
           L.ptr(beta), i32(mode), L.ptr(stats), L.ptr(fmean), L.ptr(frstd), L.ptr(out), L.ll(out_bs), _s())


def conv0_bwd(wav, L_, B, T, Cc, k, s, w, gamma, beta, mode, stats, bstats, fmean, frstd, da, da_bs, dw, dgamma, dbeta,
              dconv_ws=None, ws_bs=0):
    """`dconv_ws` (LayerNorm mode): bf16 workspace for the gradient w.r.t. the raw convolution output; may be `da` itself."""
    if dconv_ws is None:
        _call("b200s_conv0_bwd", L.ptr(wav), L.ll(L_), i32(B), i32(T), i32(Cc), i32(k), i32(s), L.ptr(w), L.ptr(gamma),
               L.ptr(beta), i32(mode), L.ptr(stats), L.ptr(bstats), L.ptr(fmean), L.ptr(frstd), L.ptr(da), L.ll(da_bs),
               L.ptr(dw), L.ptr(dgamma), L.ptr(dbeta), _s())
    else:
        _call("b200s_conv0_bwd_ws", L.ptr(wav), L.ll(L_), i32(B), i32(T), i32(Cc), i32(k), i32(s), L.ptr(w), L.ptr(gamma),
               L.ptr(beta), i32(mode), L.ptr(stats), L.ptr(bstats), L.ptr(fmean), L.ptr(frstd), L.ptr(da), L.ll(da_bs),
               L.ptr(dconv_ws), L.ll(ws_bs), L.ptr(dw), L.ptr(dgamma), L.ptr(dbeta), _s())


# ------------------------------------------------------------------------------------------------- parameter prep
def scale_copy_f32(src, dst, n, scale=1.0):
    _call("b200s_scale_copy_f32", L.ptr(src), L.ptr(dst), L.ll(n), f32(scale), _s())


def prep_linear(src, N, K, scale, dst, ld, dstT, ldT):
    _call("b200s_prep_linear", L.ptr(src), i32(N), i32(K), f32(scale), L.ptr(dst), L.ll(ld), L.ptr(dstT), L.ll(ldT), _s())


def prep_linear_batched(descs, n_descs, total_tiles):
    _call("b200s_prep_linear_batched", L.ptr(descs), i32(n_descs), i32(total_tiles), _s())


def prep_conv_fwd(src, Co, Ci, k, dst):
    _call("b200s_prep_conv_fwd", L.ptr(src), i32(Co), i32(Ci), i32(k), L.ptr(dst), _s())


def prep_conv_dgrad(src, Co, Ci, k, s, rho, dst):
    _call("b200s_prep_conv_dgrad", L.ptr(src), i32(Co), i32(Ci), i32(k), i32(s), i32(rho), L.ptr(dst), _s())


def unprep_conv_wgrad(dwk, Co, Ci, k, dw):
    _call("b200s_unprep_conv_wgrad", L.ptr(dwk), i32(Co), i32(Ci), i32(k), L.ptr(dw), _s())


def posconv_prep(weight_v, weight_g, D, G, taps, norm2, wp_fwd, wp_dgrad):
    _call("b200s_posconv_prep", L.ptr(weight_v), L.ptr(weight_g), i32(D), i32(G), i32(taps), L.ptr(norm2),
           L.ptr(wp_fwd), L.ptr(wp_dgrad), _s())


def posconv_unprep(weight_v, weight_g, dwp, D, G, taps, work, dweight_v, dweight_g):
    _call("b200s_posconv_unprep", L.ptr(weight_v), L.ptr(weight_g), L.ptr(dwp), i32(D), i32(G), i32(taps),
           L.ptr(work), L.ptr(dweight_v), L.ptr(dweight_g), _s())


# ------------------------------------------------------------------------------------------------- attention
def attn_fwd(qkv, gate, tab, key_pad, out, lse, B, T, H, scale):
    _call("b200s_attn_fwd", L.ptr(qkv), L.ptr(gate), L.ptr(tab), L.ptr(key_pad), L.ptr(out), L.ptr(lse), i32(B), i32(T),
           i32(H), f32(scale), _s(), flops=4.0 * B * H * T * T * 64)


def attn_bwd(qkv, out, dout, gate, tab, key_pad, lse, delta, dqkv, dgate, dtab, B, T, H, scale):
    _call("b200s_attn_bwd", L.ptr(qkv), L.ptr(out), L.ptr(dout), L.ptr(gate), L.ptr(tab), L.ptr(key_pad), L.ptr(lse),
           L.ptr(delta), L.ptr(dqkv), L.ptr(dgate), L.ptr(dtab), i32(B), i32(T), i32(H), f32(scale), _s(),
          flops=10.0 * B * H * T * T * 64)


def attn_bwd_fused(qkv, out, dout, gate, tab, key_pad, lse, delta, dq_acc, dqkv, dgate, dtab, B, T, H, scale):
    _call("b200s_attn_bwd_fused", L.ptr(qkv), L.ptr(out), L.ptr(dout), L.ptr(gate), L.ptr(tab), L.ptr(key_pad), L.ptr(lse),
           L.ptr(delta), L.ptr(dq_acc), L.ptr(dqkv), L.ptr(dgate), L.ptr(dtab), i32(B), i32(T), i32(H), f32(scale), _s(),
          flops=10.0 * B * H * T * T * 64)


def attn_fwd_max_frames(has_bias: bool) -> int:
    """Longest T `attn_fwd` accepts (its shared-memory footprint grows with T)."""
    return int(L.load().b200s_attn_fwd_max_frames(int(bool(has_bias))))


def attn_fwd_long(qkv, gate, tab, tab_radius, key_pad, out, lse, B, T, H, scale):
    _call("b200s_attn_fwd_long", L.ptr(qkv), L.ptr(gate), L.ptr(tab), i32(tab_radius), L.ptr(key_pad), L.ptr(out), L.ptr(lse),
          i32(B), i32(T), i32(H), f32(scale), _s(), flops=4.0 * B * H * T * T * 64)


def attn_bwd_long(qkv, out, dout, gate, tab, tab_radius, key_pad, lse, delta, dqkv, dgate, dtab, B, T, H, scale):
    _call("b200s_attn_bwd_long", L.ptr(qkv), L.ptr(out), L.ptr(dout), L.ptr(gate), L.ptr(tab), i32(tab_radius), L.ptr(key_pad),
          L.ptr(lse), L.ptr(delta), L.ptr(dqkv), L.ptr(dgate), L.ptr(dtab), i32(B), i32(T), i32(H), f32(scale), _s(),
          flops=10.0 * B * H * T * T * 64)


# ------------------------------------------------------------------------------------------------- dropout
def u32(v) -> int:
    return int(v) & 0xFFFFFFFF


def dropout_rows(x, x_bs, x_rs, res, res_bs, res_rs, y, y_bs, y_rs, rows_per_batch, batches, N, p, key):
    """y = [res +] dropout(x) with the counter-based mask of csrc/dropout.cuh; `key` = (key0, key1).  y may alias x."""
    _call("b200s_dropout_rows", L.ptr(x), L.ll(x_bs), L.ll(x_rs), L.ptr(res), L.ll(res_bs), L.ll(res_rs), L.ptr(y), L.ll(y_bs),
           L.ll(y_rs), i32(rows_per_batch), i32(batches), i32(N), f32(p), u32(key[0]), u32(key[1]), _s())


def memset_zero(t):
    """Zero a contiguous device tensor on the current stream (cudaMemsetAsync)."""
    _call("b200s_memset_zero", L.ptr(t), int(t.numel() * t.element_size()), _s())


def sumsq_rows(x, x_bs, x_rs, rows_per_batch, batches, N, out):
    """*out (fp64, device) += sum x^2 over the bf16 rows view."""
    _call("b200s_sumsq_rows", L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(rows_per_batch), i32(batches), i32(N), L.ptr(out), _s())


def grad_multiply(g, g_bs, g_rs, x, x_bs, x_rs, rows_per_batch, batches, N, scale, pen_grad=None, pen_mul=0.0):
    """g <- scale * (g + (*pen_grad * pen_mul) * x) in place (GradMultiply backward fused with the feature-penalty gradient)."""
    _call("b200s_grad_multiply", L.ptr(g), L.ll(g_bs), L.ll(g_rs), L.ptr(x), L.ll(x_bs), L.ll(x_rs), i32(rows_per_batch),
          i32(batches), i32(N), f32(scale), L.ptr(pen_grad), f32(pen_mul), _s())


def attn_dropout_mask_words(B, T, H) -> int:
    n = (T + 127) // 128
    return B * H * (4 * n) * (128 * n)


def attn_fwd_dropout(qkv, gate, tab, key_pad, out, lse, B, T, H, scale, p, key, drop_mask):
    _call("b200s_attn_fwd_dropout", L.ptr(qkv), L.ptr(gate), L.ptr(tab), L.ptr(key_pad), L.ptr(out), L.ptr(lse), i32(B), i32(T),
           i32(H), f32(scale), f32(p), u32(key[0]), u32(key[1]), L.ptr(drop_mask), _s(), flops=4.0 * B * H * T * T * 64)


def attn_bwd_fused_dropout(qkv, out, dout, gate, tab, key_pad, lse, delta, dq_acc, dqkv, dgate, dtab, B, T, H, scale, p,
                           drop_mask):
    _call("b200s_attn_bwd_fused_dropout", L.ptr(qkv), L.ptr(out), L.ptr(dout), L.ptr(gate), L.ptr(tab), L.ptr(key_pad),
           L.ptr(lse), L.ptr(delta), L.ptr(dq_acc), L.ptr(dqkv), L.ptr(dgate), L.ptr(dtab), i32(B), i32(T), i32(H), f32(scale),
           f32(p), L.ptr(drop_mask), _s(), flops=10.0 * B * H * T * T * 64)


# ------------------------------------------------------------------------------------------------- optimizer
def sumsq_f32(g, n, out):
    _call("b200s_sumsq_f32", L.ptr(g), L.ll(n), L.ptr(out), _s())


def sumsq_table(table, n_tensors, total_chunks, g, out):
    _call("b200s_sumsq_table", L.ptr(table), i32(n_tensors), L.ll(total_chunks), L.ptr(g), L.ptr(out), _s())


def adam_step(table, n_tensors, total_chunks, g, m, v, sumsq, grad_scale, max_norm, lr, beta1, beta2, eps, weight_decay, step,
              zero_grad):
    _call("b200s_adam_step", L.ptr(table), i32(n_tensors), L.ll(total_chunks), L.ptr(g), L.ptr(m), L.ptr(v), L.ptr(sumsq),
           f32(grad_scale), f32(max_norm), f32(lr), f32(beta1), f32(beta2), f32(eps), f32(weight_decay), i32(step),
           i32(1 if zero_grad else 0), _s())


# ------------------------------------------------------------------------------------------------- masked-prediction head
def gather_rows(x, x_rs, idx, S, D, out, out_rs):
    _call("b200s_gather_rows", L.ptr(x), L.ll(x_rs), L.ptr(idx), i32(S), i32(D), L.ptr(out), L.ll(out_rs), _s())


def scatter_add_rows(src, src_rs, idx, S, D, dx, dx_rs):
    _call("b200s_scatter_add_rows", L.ptr(src), L.ll(src_rs), L.ptr(idx), i32(S), i32(D), L.ptr(dx), L.ll(dx_rs), _s())


def nce_prep(label_embs, C, Cpad, Dp, en, en_t, invn):
    _call("b200s_nce_prep", L.ptr(label_embs), i32(C), i32(Cpad), i32(Dp), L.ptr(en), L.ptr(en_t), L.ptr(invn), _s())


def nce_ce(proj, proj_rs, Dp, zraw, z_rs, target, S, C, Cpad, logit_temp, weight, g, g_rs, pn, rvec, loss_sum, correct):
    _call("b200s_nce_ce", L.ptr(proj), L.ll(proj_rs), i32(Dp), L.ptr(zraw), L.ll(z_rs), L.ptr(target), i32(S), i32(C), i32(Cpad),
           f32(logit_temp), f32(weight), L.ptr(g), L.ll(g_rs), L.ptr(pn), L.ptr(rvec), L.ptr(loss_sum), L.ptr(correct), _s())


def nce_dproj(dproj, d_rs, proj, p_rs, S, Dp, pn, rvec):
    _call("b200s_nce_dproj", L.ptr(dproj), L.ll(d_rs), L.ptr(proj), L.ll(p_rs), i32(S), i32(Dp), L.ptr(pn), L.ptr(rvec), _s())


def nce_dlabel(d_en, label_embs, invn, C, Dp, d_label_embs):
    _call("b200s_nce_dlabel", L.ptr(d_en), L.ptr(label_embs), L.ptr(invn), i32(C), i32(Dp), L.ptr(d_label_embs), _s())


# ------------------------------------------------------------------------------------------------- UniSpeech-SAT head
def sat_nce_fwd(proj, proj_rs, y, y_rs, idx, same, S, N, Dp, logit_temp, g, loss_sum, stats):
    _call("b200s_sat_nce_fwd", L.ptr(proj), L.ll(proj_rs), L.ptr(y), L.ll(y_rs), L.ptr(idx), L.ptr(same), i32(S), i32(N), i32(Dp),
          f32(logit_temp), L.ptr(g), L.ptr(loss_sum), L.ptr(stats), _s())


def w2v_nce_fwd(proj, proj_rs, y, y_rs, idx, S, N, Dp, logit_temp, g, loss_sum, stats):
    _call("b200s_w2v_nce_fwd", L.ptr(proj), L.ll(proj_rs), L.ptr(y), L.ll(y_rs), L.ptr(idx), i32(S), i32(N), i32(Dp),
          f32(logit_temp), L.ptr(g), L.ptr(loss_sum), L.ptr(stats), _s())


def sat_nce_bwd(proj, proj_rs, y, y_rs, idx, S, N, Dp, logit_temp, g, upstream, dproj_acc, dy_acc):
    _call("b200s_sat_nce_bwd", L.ptr(proj), L.ll(proj_rs), L.ptr(y), L.ll(y_rs), L.ptr(idx), i32(S), i32(N), i32(Dp),
          f32(logit_temp), L.ptr(g), L.ptr(upstream), L.ptr(dproj_acc), L.ptr(dy_acc), _s())


def f32_to_bf16_rows(src, src_rs, dst, dst_rs, rows, N):
    _call("b200s_f32_to_bf16_rows", L.ptr(src), L.ll(src_rs), L.ptr(dst), L.ll(dst_rs), L.ll(rows), i32(N), _s())


def vq_hard(logits, logits_rs, vars_, S, G, V, dv, codes, q, q_rs, counts, probs, gumbel=False, key=(0, 0)):
    _call("b200s_vq_hard", L.ptr(logits), L.ll(logits_rs), L.ptr(vars_), i32(S), i32(G), i32(V), i32(dv), L.ptr(codes), L.ptr(q),
          L.ll(q_rs), L.ptr(counts), L.ptr(probs), i32(1 if gumbel else 0), u32(key[0]), u32(key[1]), _s())


def vq_logits_bwd(logits, logits_rs, S, G, V, c, h, h_rs, tau, key, dlogits, dlogits_rs):
    _call("b200s_vq_logits_bwd", L.ptr(logits), L.ll(logits_rs), i32(S), i32(G), i32(V), L.ptr(c), L.ptr(h), L.ll(h_rs), f32(tau),
          u32(key[0]), u32(key[1]), L.ptr(dlogits), L.ll(dlogits_rs), _s())


def vq_dvars(dq, dq_rs, codes, S, G, V, dv, dvars):
    _call("b200s_vq_dvars", L.ptr(dq), L.ll(dq_rs), L.ptr(codes), i32(S), i32(G), i32(V), i32(dv), L.ptr(dvars), _s())


# ------------------------------------------------------------------------------------------------- on-device data path
def span_mask(valid_len, B, T, mask_prob, mask_length, min_masks, key, mask, counts):
    _call("b200s_span_mask", L.ptr(valid_len), i32(B), i32(T), f32(mask_prob), i32(mask_length), i32(min_masks), u32(key[0]),
          u32(key[1]), L.ptr(mask), L.ptr(counts), _s())


def row_power(x, x_bs, B, Ln, power):
    _call("b200s_row_power", L.ptr(x), L.ll(x_bs), i32(B), i32(Ln), L.ptr(power), _s())


def mix_apply(src, bs, B, Ln, plan, power, dst):
    _call("b200s_mix_apply", L.ptr(src), L.ll(bs), i32(B), i32(Ln), L.ptr(plan), L.ptr(power), L.ptr(dst), _s())


def row_normalize(x, bs, B, Ln, valid_len, stats, plan):
    _call("b200s_row_normalize", L.ptr(x), L.ll(bs), i32(B), i32(Ln), L.ptr(valid_len), L.ptr(stats), L.ptr(plan), _s())
