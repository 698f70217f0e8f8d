"""Thin ctypes wrappers of the individual-operator C-ABI entry points (include/vqacl_b200.h) for the GPU parity tests."""
import ctypes
from ctypes import c_float, c_int, c_int64, c_void_p

import torch

from vqacl_b200._lib import check, cur_stream, lib, ptr

F = c_float


def _L():
    L = lib()
    if not getattr(L, "_ops_declared", False):
        L.vqacl_rmsnorm_fwd.argtypes = [c_void_p] * 4 + [c_int, F, F, c_void_p]
        L.vqacl_rmsnorm_bwd.argtypes = [c_void_p] * 7 + [c_int, F, F, c_void_p]
        L.vqacl_attention_fwd.argtypes = [c_void_p] * 3 + [c_int] * 3 + [c_void_p, c_int, c_void_p] + [c_int] * 4 + [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]
        L.vqacl_attention_bwd.argtypes = ([c_void_p] * 3 + [c_int] * 3 + [c_void_p, c_int, c_void_p] + [c_void_p] * 3 + [c_int] * 3 + [c_int] * 4 +
                                          [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p])
        L.vqacl_attention_fwd_ex.argtypes = (L.vqacl_attention_fwd.argtypes[:-1] + [ctypes.c_uint32, F, ctypes.c_uint32] + [c_int64] * 4 +
                                             [c_int, c_void_p])
        L.vqacl_attention_bwd_ex.argtypes = L.vqacl_attention_bwd.argtypes[:-1] + [ctypes.c_uint32, F, ctypes.c_uint32, c_void_p]
        L.vqacl_proto_means.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]
        L.vqacl_proto_scatter_mean.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
        L.vqacl_proto_update.argtypes = [c_void_p] * 8 + [c_int] * 5 + [F, F, c_void_p]
        L.vqacl_proto_retrieve.argtypes = [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
        L.vqacl_ce_fwd.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
        L.vqacl_ce_bwd.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
        L.vqacl_loss_tail.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
        L.vqacl_visual_embed_fwd.argtypes = [c_void_p] * 9 + [c_int] * 5 + [F, c_void_p, c_void_p]
        L.vqacl_adamw_hf.argtypes = [c_void_p] * 5 + [c_int64, c_int64, F, F, F, F, F, c_int, c_void_p, F, c_void_p]
        L.vqacl_grad_sumsq.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]
        L.vqacl_gemm_bf16.argtypes = [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int,
                                      c_int, F, c_int, c_int, c_void_p]
        L.vqacl_gemm_bf16_ex.argtypes = [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int,
                                         c_int, F, c_int, c_int, ctypes.c_uint32, F, ctypes.c_uint32, c_void_p]
        L.vqacl_gemm_resid_rmsnorm.argtypes = [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, F, c_void_p, c_void_p]
        L.vqacl_visual_embed_fused.argtypes = [c_void_p, c_void_p, c_int] + [c_void_p] * 8 + [c_int] * 5 + [F, c_void_p, c_void_p, c_void_p]
        L.vqacl_gemm_bf16_slabs.argtypes = [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_int64, c_int, c_int, c_int, F,
                                            c_int, c_int, ctypes.POINTER(c_int), c_void_p]
        L.vqacl_set_gemm_sm_limit.argtypes = [c_int]
        L.vqacl_set_gemm_dynamic_schedule.argtypes = [c_int]
        L.vqacl_launch_count.restype = ctypes.c_longlong
        L._ops_declared = True
    return L


def rmsnorm_fwd(x, w, eps=1e-6, scale=1.0):
    M = x.shape[0]
    yb = torch.empty(M, 768, dtype=torch.bfloat16, device=x.device)
    yf = torch.empty(M, 768, dtype=torch.float32, device=x.device)
    check(_L().vqacl_rmsnorm_fwd(ptr(x), ptr(w), ptr(yb), ptr(yf), M, eps, scale, cur_stream()))
    return yb, yf


def rmsnorm_bwd(dn, x, w, g_in=None, eps=1e-6, scale=1.0):
    M = x.shape[0]
    g_out = torch.empty(M, 768, dtype=torch.float32, device=x.device)
    gb = torch.empty(M, 768, dtype=torch.bfloat16, device=x.device)
    dw = torch.zeros(768, dtype=torch.float32, device=x.device)
    check(_L().vqacl_rmsnorm_bwd(ptr(dn), ptr(x), ptr(w), ptr(g_in), ptr(g_out), ptr(gb), ptr(dw), M, eps, scale, cur_stream()))
    return g_out, gb, dw


def attention_fwd(q, k, v, B, H, Sq, Sk, rel_table=None, rel_bucket=None, rel_mode=0, Lt=0, keymask=None, causal=0):
    """q [B*Sq, H*64], k/v [B*Sk, H*64] bf16 (row pitch = stride(0))."""
    o = torch.empty(B * Sq, H * 64, dtype=torch.bfloat16, device=q.device)
    lse = torch.empty(B, H, Sq, dtype=torch.float32, device=q.device)
    check(_L().vqacl_attention_fwd(ptr(q), ptr(k), ptr(v), q.stride(0), k.stride(0), v.stride(0), ptr(o), o.stride(0), ptr(lse), B, H, Sq, Sk,
                                   ptr(rel_table), ptr(rel_bucket), rel_mode, Lt, ptr(keymask), causal, cur_stream()))
    return o, lse


def attention_bwd(q, k, v, dO, lse, B, H, Sq, Sk, rel_table=None, rel_bucket=None, rel_mode=0, Lt=0, keymask=None, causal=0, o_saved=None):
    dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    dtab = torch.zeros_like(rel_table) if rel_table is not None else None
    check(_L().vqacl_attention_bwd(ptr(q), ptr(k), ptr(v), q.stride(0), k.stride(0), v.stride(0), ptr(dO), dO.stride(0), ptr(lse),
                                   ptr(dq), ptr(dk), ptr(dv), dq.stride(0), dk.stride(0), dv.stride(0), B, H, Sq, Sk, ptr(rel_table),
                                   ptr(rel_bucket), rel_mode, Lt, ptr(keymask), causal, ptr(dtab), ptr(o_saved), cur_stream()))
    return dq, dk, dv, dtab


def _pitch(t, ld=None):
    """row pitch of a 2-D operand: stride(0) unless given; 0 for a missing (NULL) operand"""
    return ld if ld is not None else 0 if t is None else t.stride(0)


def attention_fwd_ex(q, k, v, o, lse, B, H, Sq, Sk, rel_table=None, rel_bucket=None, rel_mode=0, Lt=0, keymask=None, causal=0,
                     drop=(0, 1.0, 0), bstrides=(0, 0, 0, 0), q_off=0, ld=(None, None, None, None)):
    """vqacl_attention_fwd_ex into caller-provided o (and lse, or None). Pointers are the tensors' first elements; the row pitches
    are their stride(0) unless given in ld = (ldq, ldk, ldv, ldo). drop = (thr16, inv_keep, key)."""
    check(_L().vqacl_attention_fwd_ex(ptr(q), ptr(k), ptr(v), _pitch(q, ld[0]), _pitch(k, ld[1]), _pitch(v, ld[2]), ptr(o), _pitch(o, ld[3]),
                                      ptr(lse), B, H, Sq, Sk, ptr(rel_table), ptr(rel_bucket), rel_mode, Lt, ptr(keymask), causal,
                                      int(drop[0]), float(drop[1]), int(drop[2]), *[int(x) for x in bstrides], q_off, cur_stream()))


def attention_bwd_ex(q, k, v, dO, lse, dq, dk, dv, d_rel_table, B, H, Sq, Sk, rel_table=None, rel_bucket=None, rel_mode=0, Lt=0,
                     keymask=None, causal=0, o_saved=None, drop=(0, 1.0, 0)):
    """vqacl_attention_bwd_ex into caller-provided dq / dk / dv (row pitches = their stride(0)); d_rel_table is accumulated into."""
    check(_L().vqacl_attention_bwd_ex(ptr(q), ptr(k), ptr(v), _pitch(q), _pitch(k), _pitch(v), ptr(dO), _pitch(dO), ptr(lse),
                                      ptr(dq), ptr(dk), ptr(dv), _pitch(dq), _pitch(dk), _pitch(dv), B, H, Sq, Sk, ptr(rel_table),
                                      ptr(rel_bucket), rel_mode, Lt, ptr(keymask), causal, ptr(d_rel_table), ptr(o_saved),
                                      int(drop[0]), float(drop[1]), int(drop[2]), cur_stream()))


def proto_means(h, split):
    B, S, _ = h.shape
    mq = torch.empty(B, 768, device=h.device)
    mv = torch.empty(B, 768, device=h.device)
    check(_L().vqacl_proto_means(ptr(h), B, S, split, ptr(mq), ptr(mv), cur_stream()))
    return mq, mv


def proto_scatter_mean(mean, labels):
    B, C = labels.shape
    proto = torch.empty(C, 768, device=mean.device)
    cnt = torch.empty(C, device=mean.device)
    check(_L().vqacl_proto_scatter_mean(ptr(mean), ptr(labels), B, C, ptr(proto), ptr(cnt), cur_stream()))
    return proto, cnt


def proto_update(curQ, curV, cntQ, cntV, Q, Vp, numQ, numV, task, first, has_mem, alpha, beta):
    check(_L().vqacl_proto_update(ptr(curQ), ptr(curV), ptr(cntQ), ptr(cntV), ptr(Q), ptr(Vp), ptr(numQ), ptr(numV), Q.shape[0], Vp.shape[0],
                                  task, int(first), int(has_mem), alpha, beta, cur_stream()))


def proto_retrieve(P, x):
    B = x.shape[0]
    out = torch.empty(B, 768, device=x.device)
    idx = torch.empty(B, dtype=torch.int64, device=x.device)
    scratch = torch.empty(P.shape[0], 768, device=x.device)
    check(_L().vqacl_proto_retrieve(ptr(P), P.shape[0], ptr(x), B, None, 0, 0, ptr(idx), ptr(out), ptr(scratch), cur_stream()))
    return out, idx


def ce_fwd(logits, labels, V):
    M = logits.shape[0]
    lse = torch.empty(M, device=logits.device)
    loss = torch.empty(M, device=logits.device)
    check(_L().vqacl_ce_fwd(ptr(logits), logits.stride(0), M, V, ptr(labels), ptr(lse), ptr(loss), cur_stream()))
    return lse, loss


def ce_bwd(logits, labels, V, lse, w):
    check(_L().vqacl_ce_bwd(ptr(logits), logits.stride(0), logits.shape[0], V, ptr(labels), ptr(lse), ptr(w), cur_stream()))


def loss_tail(rows, labels, scores):
    B, T = labels.shape
    out = torch.zeros(4, device=rows.device)
    w = torch.empty(B * T, device=rows.device)
    check(_L().vqacl_loss_tail(ptr(rows), ptr(labels), ptr(scores), B, T, ptr(out), ptr(w), cur_stream()))
    return out[0], w


def visual_embed_fwd(featpre, boxes, bf, wf, Wp, bp, wp, img, shared, B, N, eps=1e-6):
    x = torch.zeros(B, N, 768, device=featpre.device)
    check(_L().vqacl_visual_embed_fwd(ptr(featpre), ptr(boxes), ptr(bf), ptr(wf), ptr(Wp), ptr(bp), ptr(wp), ptr(img), ptr(shared),
                                      shared.shape[0], B, N, N, 0, eps, ptr(x), cur_stream()))
    return x


def adamw(p, g, m, v, n_decay, lr, b1, b2, eps, wd, step, sumsq=None, max_norm=0.0, p_bf16=None):
    check(_L().vqacl_adamw_hf(ptr(p), ptr(g), ptr(m), ptr(v), ptr(p_bf16), p.numel(), n_decay, lr, b1, b2, eps, wd, step, ptr(sumsq), max_norm,
                              cur_stream()))


def grad_sumsq(g):
    partials = torch.empty(2048, device=g.device)
    out = torch.empty(1, device=g.device)
    check(_L().vqacl_grad_sumsq(ptr(g), g.numel(), ptr(partials), ptr(out), cur_stream()))
    return out


def gemm(A, a_mn, B, b_mn, C, R, M, N, K, epi, alpha=1.0, splits=1, bn=0):
    check(_L().vqacl_gemm_bf16(ptr(A), A.stride(0), int(a_mn), ptr(B), B.stride(0), int(b_mn), ptr(C), C.stride(0), ptr(R),
                               R.stride(0) if R is not None else 0, M, N, K, epi, alpha, splits, bn, cur_stream()))


def gemm_dropout(A, B, C, R, M, N, K, epi, thr16, inv_keep, key, bn=0):
    check(_L().vqacl_gemm_bf16_ex(ptr(A), A.stride(0), 0, ptr(B), B.stride(0), 0, ptr(C), C.stride(0), ptr(R),
                                  R.stride(0) if R is not None else 0, M, N, K, epi, 1.0, 1, bn, thr16, inv_keep, key, cur_stream()))


def dropout_scale_host(M, N, thr16, inv_keep, key, device):
    """Host restatement of vq_dropout_pair (csrc/common.cuh): scale (0 or inv_keep) of every element of an [M, N] matrix."""
    return dropout_scale_idx(torch.arange(M * N, device=device, dtype=torch.int64).view(M, N), thr16, inv_keep, key)


def dropout_scale_idx(idx, thr16, inv_keep, key):
    """Scale (0 or inv_keep) of the elements with int64 element indices `idx`: pair idx >> 1 is hashed with the 32-bit key, the
    low 16 bits of the hash decide the even element of the pair and the high 16 bits the odd one."""
    m32 = 0xFFFFFFFF
    x = ((idx >> 1) * 0x9E3779B1 + key) & m32
    x = x ^ (x >> 16)
    x = (x * 0x85EBCA6B) & m32
    x = x ^ (x >> 13)
    x = (x * 0xC2B2AE35) & m32
    x = x ^ (x >> 16)
    lane = torch.where((idx & 1) == 1, x >> 16, x & 0xFFFF)
    return (lane >= thr16).float() * inv_keep


def gemm_resid_rmsnorm(A, B, R, norm_w, eps=1e-6):
    M, K = A.shape
    C = torch.empty(M, 768, device=A.device)
    n = torch.empty(M, 768, device=A.device, dtype=torch.bfloat16)
    check(_L().vqacl_gemm_resid_rmsnorm(ptr(A), A.stride(0), ptr(B), B.stride(0), ptr(C), ptr(R), M, K, ptr(norm_w), eps, ptr(n), cur_stream()))
    return C, n


def visual_embed_fused(feats_bf16, Wf_bf16, boxes, bf, wf, Wp, bp, wp, img, shared, B, N, eps=1e-6):
    Fd = feats_bf16.shape[-1]
    featpre = torch.empty(B * N, 768, device=boxes.device)
    x = torch.zeros(B, N, 768, device=boxes.device)
    check(_L().vqacl_visual_embed_fused(ptr(feats_bf16), ptr(Wf_bf16), Fd, ptr(boxes), ptr(bf), ptr(wf), ptr(Wp), ptr(bp), ptr(wp), ptr(img),
                                        ptr(shared), shared.shape[0], B, N, N, 0, eps, ptr(featpre), ptr(x), cur_stream()))
    return x, featpre


def gemm_grouped_mn(As, Bs, Cs, epi=3, alpha=1.0):
    """Problem i: Cs[i][M_i, N_i] (+)= As[i]^T @ Bs[i] with As[i] stored [K, M_i], Bs[i] stored [K, N_i] (bf16); one launch."""
    n = len(As)
    K = As[0].shape[0]
    VP = ctypes.c_void_p * n
    IP = ctypes.c_int * n
    L = _L()
    L.vqacl_gemm_bf16_grouped_mn.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_void_p),
                                             ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int),
                                             ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                             ctypes.c_void_p]
    check(L.vqacl_gemm_bf16_grouped_mn(n, VP(*[a.data_ptr() for a in As]), IP(*[a.stride(0) for a in As]), VP(*[b.data_ptr() for b in Bs]),
                                       IP(*[b.stride(0) for b in Bs]), VP(*[c.data_ptr() for c in Cs]), IP(*[c.stride(0) for c in Cs]),
                                       IP(*[a.shape[1] for a in As]), IP(*[b.shape[1] for b in Bs]), K, epi, ctypes.c_float(alpha), cur_stream()))
    return Cs


def gemm_slabs(A, a_mn, B, b_mn, C, M, N, K, split_stride, alpha=1.0, splits=1, bn=0):
    """Split-K with one fp32 slab per split: slab s = C.view(-1)[s * split_stride:] with pitch C.stride(0). Returns the number of
    slabs the GEMM wrote."""
    n = c_int(-1)
    check(_L().vqacl_gemm_bf16_slabs(ptr(A), A.stride(0), int(a_mn), ptr(B), B.stride(0), int(b_mn), ptr(C), C.stride(0), split_stride,
                                     M, N, K, alpha, splits, bn, ctypes.byref(n), cur_stream()))
    return n.value


def set_gemm_sm_limit(n):
    """Process-wide: SMs the persistent GEMMs may occupy (0 = all; odd values are rounded down to even)."""
    check(_L().vqacl_set_gemm_sm_limit(int(n)))


def set_gemm_dynamic_schedule(on):
    """Process-wide: atomic-counter tile schedule of the CTA-pair kernel instead of the static round robin."""
    check(_L().vqacl_set_gemm_dynamic_schedule(int(bool(on))))


def launch_count():
    return int(_L().vqacl_launch_count())
