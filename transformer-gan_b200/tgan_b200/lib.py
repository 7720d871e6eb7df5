"""ctypes binding of libtgan_b200.so (C ABI declared in include/tgan_b200.h).

There is NO fallback: if the shared library is missing or fails to load, importing this module raises.
Tensors are passed as raw device pointers (``tensor.data_ptr()``), the stream is torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_uint64, c_ulonglong, c_void_p

import torch

F32, BF16 = 0, 1
HS = 64
EPI_BIAS, EPI_RELU, EPI_MASK_POS, EPI_ADD_AUX, EPI_ACCUM, EPI_DROPOUT, EPI_AUX_F32 = 1, 2, 4, 8, 16, 32, 64
IMPL_AUTO, IMPL_SIMT, IMPL_TC = 0, 1, 2

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtgan_b200.so")


class TganError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with transformer-gan_b200/csrc/build.sh (or __graft_entry__.build()). "
            "tgan_b200 has no CPU / eager fallback.")
    return ctypes.CDLL(LIB_PATH)


_lib = _load()
_lib.tgan_last_error.restype = c_char_p
_lib.tgan_launch_count.restype = c_ulonglong

P, I, L, F, U = c_void_p, c_int, c_int64, c_float, c_uint64
_SIGS = {
    "tgan_gemm": [I, I, I, I, I, I, I, P, L, P, L, P, L, P, P, L, I, F, F, U, U, I, P],
    "tgan_embed_fwd": [I, P, P, L, P, L, I, I, I, F, F, U, U, P],
    "tgan_embed_bwd": [I, P, P, L, P, L, I, I, I, F, F, U, U, P],
    "tgan_pos_emb": [I, P, P, L, I, I, I, I, F, U, U, P],
    "tgan_ln_fwd": [I, P, L, P, L, P, P, P, P, I, I, I, I, P],
    "tgan_ln_bwd": [I, P, L, P, L, P, P, P, P, L, P, L, P, P, P, I, I, I, F, U, U, P],
    "tgan_dropout": [I, P, L, P, L, I, I, F, U, U, P],
    "tgan_relattn_fwd": [I, P, L, P, P, L, P, L, P, P, P, P, L, P, I, I, I, I, I, I, F, F, U, U, I, P],
    "tgan_relattn_fwd_ragged": [I, P, L, P, P, L, P, L, P, P, P, P, L, P, I, I, I, I, I, I, F, F, U, U, I, P, P, L],
    "tgan_relattn_bwd": [I, P, L, P, P, L, P, L, P, P, P, P, P, L, P, P, P, P, P, L, P, L, P, P, I, I, I, I, I, I,
                         F, F, U, U, I, P],
    "tgan_relattn_bwd_step": [I, I, P, L, P, P, L, P, L, P, P, P, P, P, L, P, P, P, P, P, L, P, L, P, P, I, I, I, I, I,
                              F, F, U, U, P],
    "tgan_lamb_step": [P, P, P, P, P, P, I, P, I, F, F, F, F, F, P, F, F, I, P],
    "tgan_batch_next": [P, P, P, P, I, P, P, P, P, P, P, P, I, I, L, P],
    "tgan_batch_gather": [P, P, P, P, P, I, I, L, P],
    "tgan_ce_fwd": [P, L, P, P, P, I, I, P],
    "tgan_ce_bwd": [I, P, L, P, P, P, P, L, I, I, I, P],
    "tgan_gumbel_st_fwd": [P, L, P, L, F, P, P, L, P, L, P, I, I, U, U, P],
    "tgan_gumbel_st_bwd": [P, L, P, L, F, P, P, L, I, I, P],
    "tgan_colsum": [I, P, L, P, I, I, P],
    "tgan_convert": [I, P, L, I, P, L, L, I, I, P],
    "tgan_pack_params": [I, P, P, P, I, L, P],
    "tgan_unpack_grads": [P, P, P, I, L, I, P],
    "tgan_sumsq": [P, L, P, P],
    "tgan_adam_step": [P, P, P, P, L, F, F, F, F, F, I, P, F, F, P],
    "tgan_set_step_counter": [P],
    "tgan_ln_fwd_eps": [I, P, L, P, L, P, P, P, P, I, I, I, I, F, P],
    "tgan_gelu": [I, I, P, L, P, L, P, L, I, I, P],
    "tgan_bert_embed_rows": [I, P, L, P, P, L, P, I, P, L, I, I, P],
    "tgan_ln_jvp": [I, P, L, P, L, P, P, P, P, L, I, I, P],
    "tgan_bert_attn_fwd": [I, P, L, P, L, P, I, I, I, I, F, U, U, P],
    "tgan_bert_attn_bwd": [I, P, L, P, L, P, P, L, I, I, I, I, F, U, U, P],
    "tgan_bert_attn_jvp": [I, P, L, P, L, P, P, L, I, I, I, I, F, U, U, P],
    "tgan_sample_tokens": [P, L, P, P, P, P, L, I, I, I, I, I, I, F, F, U, U, P],
    "tgan_sample_step": [P, L, P, P, P, P, P, P, P, P, P, P, P, P, L, I, I, I, U, U, P],
    "tgan_ring_scatter": [I, P, I, I, I, P, L, P, L, I, I, P, L, P, L, I, I, I, I, P],
    "tgan_nccl_load": [c_char_p],
    "tgan_nccl_unique_id": [P],
    "tgan_nccl_init": [P, I, I, P],
    "tgan_allreduce_bucket": [P, P, L, I, P],
    "tgan_nccl_destroy": [P],
}
EXPORTS = ["tgan_last_error", "tgan_version", "tgan_has_tcgen05", "tgan_launch_count"] + list(_SIGS)
for _name, _sig in _SIGS.items():
    _fn = getattr(_lib, _name)
    _fn.argtypes = _sig
    _fn.restype = c_int


def version() -> int:
    return _lib.tgan_version()


def has_tcgen05() -> bool:
    return bool(_lib.tgan_has_tcgen05())


_replayed = 0
_step_counters = {}


def launch_count() -> int:
    """Kernels of this library enqueued so far: direct launches plus the kernel nodes of every graph replay."""
    return int(_lib.tgan_launch_count()) + _replayed


def note_graph_replay(n_kernels: int) -> None:
    global _replayed
    _replayed += n_kernels


def step_counter(device) -> torch.Tensor:
    """The process-wide device step counter (int32 [1]) registered with tgan_set_step_counter; created on first use."""
    key = torch.device(device).index or 0
    if key not in _step_counters:
        t = torch.zeros(1, dtype=torch.int32, device=device)
        set_step_counter(t)
        _step_counters[key] = t
    return _step_counters[key]


def set_step_counter(counter) -> None:
    """Register (or, with None, clear) the device uint32/int32 step counter folded into every dropout / noise key."""
    _call("tgan_set_step_counter", None if counter is None else counter.data_ptr())


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, int):
        return t
    return t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream():
    """raw handle of torch's current CUDA stream (the C accessor is ~20x cheaper than the Stream object; a decode
    step makes ~55 calls)"""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise TganError(f"unsupported dtype {dt}")


def _call(name, *args):
    rc = getattr(_lib, name)(*args)
    if rc != 0:
        raise TganError(f"{name} failed ({rc}): {_lib.tgan_last_error().decode()}")


# ---------------------------------------------------------------------------------------------------------
# thin typed wrappers (tensors in, nothing allocated)
# ---------------------------------------------------------------------------------------------------------
def gemm(A, B, C, *, transA=False, transB=True, M, N, K, lda=None, ldb=None, ldc=None, bias=None, aux=None,
         ldaux=0, flags=0, alpha=1.0, drop_p=0.0, seed=0, site=0, impl=IMPL_AUTO, a_off=0, b_off=0, c_off=0,
         aux_off=0):
    """C[M,N] = epi(op(A) op(B)).  *_off are element offsets into the tensors (row/column sub-views)."""
    ea, ec = A.element_size(), C.element_size()
    lda = lda if lda is not None else A.stride(0)
    ldb = ldb if ldb is not None else B.stride(0)
    ldc = ldc if ldc is not None else C.stride(0)
    if aux is not None and aux.dtype == torch.float32 and A.dtype != torch.float32:
        flags |= EPI_AUX_F32
    _call("tgan_gemm", dtype_code(A.dtype), dtype_code(C.dtype), int(transA), int(transB), M, N, K,
          A.data_ptr() + a_off * ea, lda, B.data_ptr() + b_off * ea, ldb, C.data_ptr() + c_off * ec, ldc,
          _ptr(bias), None if aux is None else aux.data_ptr() + aux_off * aux.element_size(), ldaux, flags,
          alpha, drop_p, seed, site, impl, _stream())


def embed_fwd(ids, E, out, rows, D, DP, scale, drop_p, seed, site, out_off=0):
    _call("tgan_embed_fwd", dtype_code(E.dtype), _ptr(ids), E.data_ptr(), DP,
          out.data_ptr() + out_off * out.element_size(), DP, rows, D, DP, scale, drop_p, seed, site, _stream())


def embed_bwd(ids, dout, dE, rows, V, D, DP, scale, drop_p, seed, site):
    _call("tgan_embed_bwd", dtype_code(dout.dtype), _ptr(ids), dout.data_ptr(), DP, dE.data_ptr(),
          DP, rows, V, D, scale, drop_p, seed, site, _stream())


def pos_emb(inv_freq, pe, klen, D, DP, clamp_len, drop_p, seed, site):
    _call("tgan_pos_emb", dtype_code(pe.dtype), _ptr(inv_freq), pe.data_ptr(), pe.stride(0), klen, D, DP,
          clamp_len, drop_p, seed, site, _stream())


def ln_fwd(z, y, gamma, beta, mean, rstd, rows, D, DP, y_off=0, pad_one=False):
    _call("tgan_ln_fwd", dtype_code(y.dtype), z.data_ptr(), z.stride(0), y.data_ptr() + y_off * y.element_size(),
          DP, _ptr(gamma), _ptr(beta), _ptr(mean), _ptr(rstd), rows, D, DP, int(pad_one), _stream())


def ln_fwd_eps(z, y, gamma, beta, mean, rstd, rows, D, eps):
    """LayerNorm with an explicit epsilon over all D columns (BERT: 1e-12); z fp32 [rows, D] -> y"""
    _call("tgan_ln_fwd_eps", dtype_code(y.dtype), z.data_ptr(), z.stride(0), y.data_ptr(), y.stride(0), _ptr(gamma),
          _ptr(beta), _ptr(mean), _ptr(rstd), rows, D, D, 0, eps, _stream())


def gelu(u, out, rows, cols, t=None):
    """t is None: out = gelu(u) (erf form);  else out = t * gelu'(u)  (input gradient and forward tangent alike)"""
    _call("tgan_gelu", dtype_code(u.dtype), 0 if t is None else 1, u.data_ptr(), u.stride(0), _ptr(t),
          0 if t is None else t.stride(0), out.data_ptr(), out.stride(0), rows, cols, _stream())


def bert_embed_rows(z, rows, cols, table, period, x=None, ids=None, E=None):
    """z[row] = (x[row] | E[ids[row]]) + table[row % period]   (z fp32)"""
    src = x if x is not None else E
    _call("tgan_bert_embed_rows", dtype_code(src.dtype), _ptr(x), 0 if x is None else x.stride(0), _ptr(ids), _ptr(E),
          0 if E is None else E.stride(0), _ptr(table), period, z.data_ptr(), z.stride(0), rows, cols, _stream())


def ln_jvp(zd, z, gamma, mean, rstd, yd, rows, D):
    _call("tgan_ln_jvp", dtype_code(yd.dtype), zd.data_ptr(), zd.stride(0), z.data_ptr(), z.stride(0), _ptr(gamma),
          _ptr(mean), _ptr(rstd), yd.data_ptr(), yd.stride(0), rows, D, _stream())


def bert_attn_fwd(qkv, ctx, lse, B, heads, T, dh, drop_p, seed, site):
    _call("tgan_bert_attn_fwd", dtype_code(qkv.dtype), qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0),
          lse.data_ptr(), B, heads, T, dh, drop_p, seed, site, _stream())


def bert_attn_bwd(qkv, dctx, lse, dqkv, B, heads, T, dh, drop_p, seed, site):
    _call("tgan_bert_attn_bwd", dtype_code(qkv.dtype), qkv.data_ptr(), qkv.stride(0), dctx.data_ptr(), dctx.stride(0),
          lse.data_ptr(), dqkv.data_ptr(), dqkv.stride(0), B, heads, T, dh, drop_p, seed, site, _stream())


def bert_attn_jvp(qkv, qkvd, lse, ctxd, B, heads, T, dh, drop_p, seed, site):
    _call("tgan_bert_attn_jvp", dtype_code(qkv.dtype), qkv.data_ptr(), qkv.stride(0), qkvd.data_ptr(), qkvd.stride(0),
          lse.data_ptr(), ctxd.data_ptr(), ctxd.stride(0), B, heads, T, dh, drop_p, seed, site, _stream())


def ln_bwd(dy, z, gamma, mean, rstd, dz, dz_drop, dgamma, dbeta, rows, D, DP, drop_p, seed, site, dy_off=0, dsum=None):
    _call("tgan_ln_bwd", dtype_code(dz.dtype), dy.data_ptr() + dy_off * dy.element_size(), DP, z.data_ptr(),
          z.stride(0), _ptr(gamma), _ptr(mean), _ptr(rstd), dz.data_ptr(), dz.stride(0),
          _ptr(dz_drop), DP, _ptr(dgamma), _ptr(dbeta), _ptr(dsum), rows, D, DP, drop_p, seed, site, _stream())


def relattn_bwd_step(phase, q, k, v, ldkv, r, u, vb, reset, out, dout, lse, scratch, dq, dk, dv, lddkv, dr, du, dvb, B, N,
                     M, msl, same_length, scale, drop_p, seed, site, k_off=0, v_off=0, dk_off=0, dv_off=0):
    """single-token (Q = 1) attention backward in two launches: phase 1 = query side (dq, du / dvb, dk / dv of the
    current row; on the dgrad chain), phase 2 = memory side (dk / dv of the rows j < M, dR; needed only by weight
    gradients: a side stream).  scratch: fp32 [2 * B * N * (M + 1) + 2 * B * N * 64]."""
    es = q.element_size()
    _call("tgan_relattn_bwd_step", phase, dtype_code(q.dtype), q.data_ptr(), q.stride(0), k.data_ptr() + k_off * es,
          v.data_ptr() + v_off * es, ldkv, r.data_ptr(), r.stride(0), _ptr(u), _ptr(vb), _ptr(reset),
          out.data_ptr(), dout.data_ptr(), out.stride(0), _ptr(lse), _ptr(scratch), dq.data_ptr(),
          dk.data_ptr() + dk_off * es, dv.data_ptr() + dv_off * es, lddkv, dr.data_ptr(), dr.stride(0),
          _ptr(du), _ptr(dvb), B, N, M, msl, int(same_length), scale, drop_p, seed, site, _stream())


def lamb_step(param, grad, m, v, upd, chunks, n_chunks, norms, n_tensors, lr, beta1, beta2, eps, weight_decay, gnorm_sq,
              clip, grad_scale, adam=False):
    _call("tgan_lamb_step", param.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), upd.data_ptr(),
          chunks.data_ptr(), n_chunks, norms.data_ptr(), n_tensors, lr, beta1, beta2, eps, weight_decay, _ptr(gnorm_sq),
          clip, grad_scale, int(adam), _stream())


def batch_next(corpus, seq_off, seq_len, perm, n_seq, tracker, data, target, reset, n_tokens, bptt, B, pad_id,
               plan_src=None, plan_n=None):
    _call("tgan_batch_next", corpus.data_ptr(), seq_off.data_ptr(), seq_len.data_ptr(), perm.data_ptr(), n_seq,
          tracker.data_ptr(), _ptr(plan_src), _ptr(plan_n), data.data_ptr(), target.data_ptr(), reset.data_ptr(),
          n_tokens.data_ptr(), bptt, B, pad_id, _stream())


def batch_gather(corpus, plan_src, plan_n, data, target, bptt, B, pad_id):
    _call("tgan_batch_gather", corpus.data_ptr(), plan_src.data_ptr(), plan_n.data_ptr(), data.data_ptr(), _ptr(target),
          bptt, B, pad_id, _stream())


def dropout(src, dst, rows, cols, lds, ldd, p, seed, site, src_off=0, dst_off=0):
    es = src.element_size()
    _call("tgan_dropout", dtype_code(src.dtype), src.data_ptr() + src_off * es, lds, dst.data_ptr() + dst_off * es,
          ldd, rows, cols, p, seed, site, _stream())


def relattn_fwd(q, k, v, ldkv, r, u, vb, reset, out, lse, B, N, Q, M, msl, same_length, scale, drop_p, seed, site,
                impl=IMPL_AUTO, k_off=0, v_off=0, key_start=None, key_base=0):
    """key_start (int32 [B]) / key_base: the per-sequence key floor of tgan_relattn_fwd_ragged (left-padded prompts);
    key_start=None calls tgan_relattn_fwd."""
    es = q.element_size()
    args = (dtype_code(q.dtype), q.data_ptr(), q.stride(0), k.data_ptr() + k_off * es, v.data_ptr() + v_off * es, ldkv,
            r.data_ptr(), r.stride(0), _ptr(u), _ptr(vb), _ptr(reset), out.data_ptr(), out.stride(0), _ptr(lse), B, N, Q,
            M, msl, int(same_length), scale, drop_p, seed, site, impl, _stream())
    if key_start is None:
        _call("tgan_relattn_fwd", *args)
    else:
        if key_start.dtype != torch.int32 or key_start.numel() != B:
            raise TganError("relattn_fwd: key_start must be an int32 tensor of B entries")
        _call("tgan_relattn_fwd_ragged", *args, key_start.data_ptr(), int(key_base))


def relattn_bwd(q, k, v, ldkv, r, u, vb, reset, out, dout, lse, delta, dq, dk, dv, lddkv, dr, du, dvb, B, N, Q, M,
                msl, same_length, scale, drop_p, seed, site, impl=IMPL_AUTO, k_off=0, v_off=0, dk_off=0, dv_off=0):
    es = q.element_size()
    _call("tgan_relattn_bwd", dtype_code(q.dtype), q.data_ptr(), q.stride(0), k.data_ptr() + k_off * es,
          v.data_ptr() + v_off * es, ldkv, r.data_ptr(), r.stride(0), _ptr(u), _ptr(vb), _ptr(reset),
          out.data_ptr(), dout.data_ptr(), out.stride(0), _ptr(lse), _ptr(delta), dq.data_ptr(),
          dk.data_ptr() + dk_off * es, dv.data_ptr() + dv_off * es, lddkv, dr.data_ptr(), dr.stride(0),
          _ptr(du), _ptr(dvb), B, N, Q, M, msl, int(same_length), scale, drop_p, seed, site, impl,
          _stream())


def ce_fwd(logits, target, nll, lse, rows, V):
    _call("tgan_ce_fwd", logits.data_ptr(), logits.stride(0), _ptr(target), _ptr(nll), _ptr(lse),
          rows, V, _stream())


def ce_bwd(logits, target, lse, dnll, dlogits, rows, V, VP):
    _call("tgan_ce_bwd", dtype_code(dlogits.dtype), logits.data_ptr(), logits.stride(0), _ptr(target),
          _ptr(lse), _ptr(dnll), dlogits.data_ptr(), dlogits.stride(0), rows, V, VP, _stream())


def _tau(tau):
    """temperature as (by-value float, device pointer): a 1-element CUDA tensor is read on the device (graph-safe)"""
    return (1.0, tau.data_ptr()) if isinstance(tau, torch.Tensor) else (float(tau), None)


def gumbel_st_fwd(logits, U, tau, y, st, ids, rows, V, seed=0, site=0):
    tv, tp = _tau(tau)
    _call("tgan_gumbel_st_fwd", logits.data_ptr(), logits.stride(0), _ptr(U), 0 if U is None else U.stride(0),
          tv, tp, y.data_ptr(), y.stride(0), _ptr(st), 0 if st is None else st.stride(0), _ptr(ids), rows, V, seed,
          site, _stream())


def gumbel_st_bwd(y, dst, tau, dlogits, rows, V):
    tv, tp = _tau(tau)
    _call("tgan_gumbel_st_bwd", y.data_ptr(), y.stride(0), dst.data_ptr(), dst.stride(0), tv, tp, dlogits.data_ptr(),
          dlogits.stride(0), rows, V, _stream())


def colsum(x, out, rows, cols, ld=None, x_off=0, out_off=0):
    _call("tgan_colsum", dtype_code(x.dtype), x.data_ptr() + x_off * x.element_size(),
          ld if ld is not None else x.stride(0), out.data_ptr() + out_off * 4, rows, cols, _stream())


def convert(src, lds, dst, ldd, rows, cols, cols_pad, src_off=0, dst_off=0):
    _call("tgan_convert", dtype_code(src.dtype), src.data_ptr() + src_off * src.element_size(), lds,
          dtype_code(dst.dtype), dst.data_ptr() + dst_off * dst.element_size(), ldd, rows, cols, cols_pad, _stream())


def pack_params(packed_mat, packed_vec, desc, n_desc, max_elems):
    _call("tgan_pack_params", dtype_code(packed_mat.dtype), packed_mat.data_ptr(), packed_vec.data_ptr(),
          desc.data_ptr(), n_desc, max_elems, _stream())


def unpack_grads(padded_mat, padded_vec, desc, n_desc, max_elems, accumulate=False):
    _call("tgan_unpack_grads", padded_mat.data_ptr(), padded_vec.data_ptr(), desc.data_ptr(), n_desc, max_elems,
          int(accumulate), _stream())


def sumsq(x, n, out):
    _call("tgan_sumsq", x.data_ptr(), n, out.data_ptr(), _stream())


def adam_step(param, grad, m, v, n, lr, beta1, beta2, eps, weight_decay, step, gnorm_sq, clip, grad_scale):
    _call("tgan_adam_step", param.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), n, lr, beta1, beta2, eps,
          weight_decay, step, _ptr(gnorm_sq), clip, grad_scale, _stream())


def sample_tokens(logits, ids, V, *, u=None, suppress_empty=None, probs_out=None, exclude_bos=True, empty_token=-1,
                  mode=1, topk=32, top_p=0.0, temperature=1.0, seed=0, site=0):
    """generate.py:228-304 for a batch of rows in one launch: logits fp32 [rows, >= V] -> ids int64 [rows].
    mode 0 random / 1 topk / 2 nucleus; u: optional injected uniforms [rows] (default: device Philox)."""
    rows = ids.numel()
    _call("tgan_sample_tokens", logits.data_ptr(), logits.stride(0), _ptr(u), _ptr(suppress_empty), ids.data_ptr(),
          _ptr(probs_out), 0 if probs_out is None else probs_out.stride(0), rows, V, int(exclude_bos), empty_token, mode,
          topk, top_p, temperature, seed, site, _stream())


def sample_step(logits, req, start, out_off, forced_next, req_i, req_f, run, cur, out, V, step, *, u=None,
                run0=None, probs_out=None, seed=0, site=0):
    """One step of generation from a request queue (tgan_sample_step): logits fp32 [B, >= V]; req / start / out_off /
    forced_next int32 [B] (forced_next may be None); req_i int32 [R, 5], req_f fp32 [R, 2]; run int32 [B] and cur int64
    [B] are updated in place; out int64 / u fp32: flat buffers indexed by out_off; run0 (int32 [R] or None): the
    empty-bar run a request starts with."""
    _call("tgan_sample_step", logits.data_ptr(), logits.stride(0), req.data_ptr(), start.data_ptr(), out_off.data_ptr(),
          _ptr(forced_next), req_i.data_ptr(), req_f.data_ptr(), _ptr(u), _ptr(run0), run.data_ptr(), cur.data_ptr(),
          out.data_ptr(), _ptr(probs_out), 0 if probs_out is None else probs_out.stride(0), req.numel(), V, step, seed,
          site, _stream())


def ring_scatter(desc, n, max_rows, dst_end, src_x, dst_x, src_kv=None, dst_kv=None, *, src_kv_stride=0,
                 dst_kv_stride=0, desc_off=0):
    """tgan_ring_scatter: descriptors desc[desc_off : desc_off + n] (int32 [*, 4]: source column, first source position,
    destination column, rows) copy rows of every slab of the ring slabs src_x [S, C, G, DP] into dst_x [S, C', B, DP],
    landing at positions [dst_end - rows, dst_end); with src_kv / dst_kv also every layer of the projected-K/V rows
    ([n_layer, *, G | B, KW] with layer strides src_kv_stride / dst_kv_stride elements, positions as in the slabs)."""
    if src_x.dtype != dst_x.dtype or (src_kv is not None and (src_kv.dtype != src_x.dtype or dst_kv.dtype != src_x.dtype)):
        raise TganError("ring_scatter: every buffer must have the same dtype")
    if src_x.shape[0] != dst_x.shape[0] or src_x.shape[3] != dst_x.shape[3]:
        raise TganError("ring_scatter: source and destination slabs differ in count or row width")
    n_kv = 0 if src_kv is None else dst_kv.shape[0]
    _call("tgan_ring_scatter", dtype_code(src_x.dtype), desc.data_ptr() + 16 * desc_off, n, max_rows, dst_end,
          src_x.data_ptr(), src_x.stride(0), dst_x.data_ptr(), dst_x.stride(0), dst_x.shape[0], dst_x.shape[3],
          _ptr(src_kv), src_kv_stride, _ptr(dst_kv), dst_kv_stride, n_kv, 0 if dst_kv is None else dst_kv.shape[-1],
          src_x.shape[2], dst_x.shape[2], _stream())


def nccl_load(path=None):
    """Bind libnccl.so.2 (default: the copy torch ships / has already loaded)."""
    if path is None:
        cand = os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "nccl", "lib", "libnccl.so.2")
        path = cand if os.path.exists(cand) else ""
    _call("tgan_nccl_load", path.encode() if path else None)


def nccl_unique_id() -> bytes:
    nccl_load()
    buf = ctypes.create_string_buffer(128)
    _call("tgan_nccl_unique_id", buf)
    return buf.raw


def nccl_init(uid: bytes, nranks: int, rank: int) -> int:
    nccl_load()
    comm = c_void_p()
    _call("tgan_nccl_init", ctypes.c_char_p(uid), nranks, rank, ctypes.byref(comm))
    return comm.value


def allreduce_bucket(comm: int, t: torch.Tensor, count=None, offset=0, stream=None):
    """in-place SUM all-reduce of t.view(-1)[offset : offset + count] on `stream` (raw handle; default: current stream)"""
    n = t.numel() - offset if count is None else count
    _call("tgan_allreduce_bucket", comm, t.data_ptr() + offset * t.element_size(), n, dtype_code(t.dtype),
          _stream() if stream is None else stream)


def nccl_destroy(comm: int):
    _call("tgan_nccl_destroy", comm)
