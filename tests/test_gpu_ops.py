"""GPU parity of every operator of the C-ABI against the oracle / a plain fp32 PyTorch statement of the same op.
Tolerances: bit-exact for indices and counts; bf16-level (stated per test) for floating point."""
import math
import os

import pytest
import torch
import torch.nn.functional as F

import cabi
from golden_fixtures import load_prototype_path
from helpers import O, cos, rel_err

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DEV = "cuda"


def test_rmsnorm_fwd_bwd_vs_oracle():
    torch.manual_seed(0)
    for M in (1, 37, 1600):
        x = (torch.randn(M, 768, device=DEV) * 3).requires_grad_()
        w = torch.randn(768, device=DEV).requires_grad_()
        ln = O.T5LayerNorm(768).to(DEV)
        ln.weight.data.copy_(w.data)
        y = ln(x)
        yb, yf = cabi.rmsnorm_fwd(x.detach(), w.detach())
        torch.testing.assert_close(yf, y.detach(), rtol=2e-6, atol=2e-6)          # fp32 path
        torch.testing.assert_close(yb.float(), y.detach(), rtol=1e-2, atol=1e-2)  # bf16 rounding of the same value
        dn = torch.randn(M, 768, device=DEV).bfloat16()
        gin = torch.randn(M, 768, device=DEV)
        y.backward(dn.float())
        g_out, gb, dw = cabi.rmsnorm_bwd(dn, x.detach(), w.detach(), gin)
        torch.testing.assert_close(g_out, gin + x.grad, rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(dw, ln.weight.grad, rtol=1e-3, atol=1e-3 * max(1.0, math.sqrt(M)))
        assert rel_err(gb, g_out) < 1e-2


def _attn_ref(q, k, v, B, H, Sq, Sk, bias):
    qh = q.float().view(B, Sq, H, 64).transpose(1, 2)
    kh = k.float().view(B, Sk, H, 64).transpose(1, 2)
    vh = v.float().view(B, Sk, H, 64).transpose(1, 2)
    s = qh @ kh.transpose(2, 3) + bias          # no 1/sqrt(d) (T5)
    p = torch.softmax(s, dim=-1)
    return (p @ vh).transpose(1, 2).reshape(B * Sq, H * 64)


@pytest.mark.parametrize("mode", ["enc", "dec_self", "cross", "enc_many"])
def test_attention_fwd_bwd_vs_torch(mode):
    from vqacl_b200.engine import rel_bucket_table
    torch.manual_seed(1)
    B, H = 5, 12
    if mode == "enc_many":      # more (batch, head-pair) items than SMs: the persistent tcgen05 kernels pipeline several per CTA
        B, mode = 110, "enc"
    if mode == "enc":
        Sq = Sk = 56; Lt = 20
    elif mode == "dec_self":
        Sq = Sk = 5; Lt = 0
    else:
        Sq, Sk, Lt = 5, 58, 0
    q = (torch.randn(B * Sq, H * 64, device=DEV) * 0.3).bfloat16().requires_grad_()
    k = (torch.randn(B * Sk, H * 64, device=DEV) * 0.3).bfloat16().requires_grad_()
    v = torch.randn(B * Sk, H * 64, device=DEV).bfloat16().requires_grad_()
    table = (torch.randn(32, H, device=DEV) * 0.5).requires_grad_()
    bias = torch.zeros(B, H, Sq, Sk, device=DEV)
    keymask = None
    kw = {}
    if mode == "enc":
        bucket = rel_bucket_table(True)          # host table
        att = O.T5Attention(O.VLT5Config(), False, True).to(DEV)
        att.relative_attention_bias.weight = torch.nn.Parameter(table.detach().clone())
        tb = att.compute_bias(Lt, Lt)
        full = torch.zeros(1, H, Sq, Sk, device=DEV)
        full[:, :, :Lt, :Lt] = tb
        pad = torch.zeros(B, Sk, device=DEV)
        pad[1, 9:20] = -10000.0
        pad[3, 15:20] = -10000.0
        keymask = pad.contiguous()
        bias = full + pad[:, None, None, :]
        kw = dict(rel_table=table.detach(), rel_bucket=bucket, rel_mode=1, Lt=Lt, keymask=keymask)
    elif mode == "dec_self":
        bucket = rel_bucket_table(False)
        att = O.T5Attention(O.VLT5Config(), True, True).to(DEV)
        att.relative_attention_bias.weight = torch.nn.Parameter(table.detach().clone())
        causal = torch.tril(torch.ones(Sq, Sk, device=DEV))
        bias = att.compute_bias(Sq, Sk) + (1.0 - causal)[None, None] * -10000.0
        kw = dict(rel_table=table.detach(), rel_bucket=bucket, rel_mode=2, causal=1)
    else:
        pad = torch.zeros(B, Sk, device=DEV)
        pad[2, 7:20] = -1e9
        keymask = pad.contiguous()
        bias = pad[:, None, None, :].expand(B, H, Sq, Sk)
        kw = dict(keymask=keymask)
    ref = _attn_ref(q, k, v, B, H, Sq, Sk, bias)
    o, lse = cabi.attention_fwd(q.detach(), k.detach(), v.detach(), B, H, Sq, Sk, **kw)
    assert rel_err(o, ref.detach()) < 1e-2
    dO = torch.randn_like(ref).bfloat16()
    if mode != "cross":
        att.relative_attention_bias.weight.grad = None
    ref.backward(dO.float())
    dq, dk, dv, dtab = cabi.attention_bwd(q.detach(), k.detach(), v.detach(), dO, lse, B, H, Sq, Sk, **kw)
    for mine, theirs, nm in ((dq, q.grad, "dq"), (dk, k.grad, "dk"), (dv, v.grad, "dv")):
        assert cos(mine, theirs) > 0.999 and rel_err(mine, theirs) < 2e-2, nm
    if mode != "cross":
        tg = att.relative_attention_bias.weight.grad
        assert cos(dtab, tg) > 0.999 and rel_err(dtab, tg) < 2e-2
    else:
        # the key-split backward (few queries x many keys; uses the saved forward output instead of a row reduction)
        dq2, dk2, dv2, _ = cabi.attention_bwd(q.detach(), k.detach(), v.detach(), dO, lse, B, H, Sq, Sk, o_saved=o, **kw)
        for mine, theirs, nm in ((dq2, q.grad, "dq"), (dk2, k.grad, "dk"), (dv2, v.grad, "dv")):
            assert cos(mine, theirs) > 0.999 and rel_err(mine, theirs) < 2e-2, "key-split " + nm


def test_prototype_kernels_match_reference_fixture_bit_exact_bookkeeping():
    """calculate_current_prototype / update_prototype / cosine_similarity_multi through the C-ABI against the fixture
    produced by executing the reference's own source (tools/gen_golden.py): counts, slot routing and argmax indices are
    compared bit-exact, prototype values to fp32 round-off (summation order differs)."""
    d = load_prototype_path()
    Q = torch.zeros(10, 768, device=DEV)
    Vp = torch.zeros(80, 768, device=DEV)
    numQ = torch.zeros(10, device=DEV)
    numV = torch.zeros(80, device=DEV)
    seen, mem = set(), set()
    for st in d["steps"]:
        h = st["hidden"].float().to(DEV).contiguous()
        mq, mv = cabi.proto_means(h, 20)
        torch.testing.assert_close(mq.cpu(), st["hidden"].float()[:, :20].mean(1), rtol=1e-5, atol=1e-6)
        curQ, cntQ = cabi.proto_scatter_mean(mq, st["ques_labels"].to(DEV))
        curV, cntV = cabi.proto_scatter_mean(mv, st["cate_labels"].to(DEV))
        assert torch.equal(cntQ.cpu(), st["numQ"]) and torch.equal(cntV.cpu(), st["numV"])
        torch.testing.assert_close(curQ.cpu(), st["curQ"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(curV.cpu(), st["curV"], rtol=1e-5, atol=1e-6)
        t = st["task"]
        first, has_mem = t not in seen, t in mem
        cabi.proto_update(curQ, curV, cntQ, cntV, Q, Vp, numQ, numV, t, first, has_mem, d["alpha"], d["beta"])
        if first:
            seen.add(t)
        elif t != 0:
            mem.add(t)
        torch.testing.assert_close(Q.cpu(), st["Q_prototype"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(Vp.cpu(), st["V_prototype"], rtol=1e-5, atol=1e-6)
        assert torch.equal(numQ.cpu(), st["Q_num"]) and torch.equal(numV.cpu(), st["V_num"])
        rq, iq = cabi.proto_retrieve(Q, mq)
        rv, iv = cabi.proto_retrieve(Vp, mv)
        assert torch.equal(iq.cpu(), st["idx_Q"]) and torch.equal(iv.cpu(), st["idx_V"])
        torch.testing.assert_close(rq.cpu(), st["retr_Q"], rtol=1e-5, atol=1e-6)
    r, i = cabi.proto_retrieve(d["eval_P"].to(DEV), d["eval_x"].to(DEV))
    assert torch.equal(i.cpu(), d["eval_idx"])          # zero rows / first-max tie-break
    assert torch.equal(r.cpu(), d["eval_retr"])


def test_retrieve_first_max_on_exact_ties():
    P = torch.zeros(10, 768, device=DEV)        # every similarity is exactly 0 -> lowest index, like torch.argmax
    x = torch.randn(4, 768, device=DEV)
    _, idx = cabi.proto_retrieve(P, x)
    assert torch.equal(idx.cpu(), torch.zeros(4, dtype=torch.long))
    P[3] = x[0]; P[6] = x[0]                     # duplicate rows -> first of the two
    _, idx = cabi.proto_retrieve(P, x[:1].contiguous())
    assert idx.item() == 3


def test_visual_embedding_matches_reference_fixture():
    d = torch.load(os.path.join(G, "visual_embedding.pt"))
    s = {k: v.to(DEV) for k, v in d["state"].items()}
    feats, boxes = d["feats"].to(DEV), d["boxes"].to(DEV)
    B, N, _ = feats.shape
    featpre = (feats.view(B * N, -1) @ s["feat_embedding.0.weight"].t()).contiguous()      # the GEMM is tested separately
    x = cabi.visual_embed_fwd(featpre, boxes.contiguous(), s["feat_embedding.0.bias"], s["feat_embedding.1.weight"],
                              s["absolute_vis_pos_embedding.0.weight"].contiguous(), s["absolute_vis_pos_embedding.0.bias"],
                              s["absolute_vis_pos_embedding.1.weight"], s["img_order_embedding.weight"].contiguous(),
                              s["obj_order_embedding.weight"].contiguous(), B, N)
    torch.testing.assert_close(x.cpu(), d["out"], rtol=1e-4, atol=1e-4)


def test_visual_embedding_fused_single_launch():
    """The whole VisualEmbedding as one launch (tcgen05 GEMM + row tail) against the fixture made by executing the reference
    class, and bit-identical to GEMM + vis_embed_fwd_kernel on the same bf16 operands; also on a multi-block shape."""
    d = torch.load(os.path.join(G, "visual_embedding.pt"))
    s = {k: v.to(DEV) for k, v in d["state"].items()}
    feats, boxes = d["feats"].to(DEV), d["boxes"].to(DEV).contiguous()
    B, N, _ = feats.shape
    args = (s["feat_embedding.0.bias"], s["feat_embedding.1.weight"], s["absolute_vis_pos_embedding.0.weight"].contiguous(),
            s["absolute_vis_pos_embedding.0.bias"], s["absolute_vis_pos_embedding.1.weight"], s["img_order_embedding.weight"].contiguous(),
            s["obj_order_embedding.weight"].contiguous())
    fb = feats.view(B * N, -1).bfloat16().contiguous()
    Wb = s["feat_embedding.0.weight"].bfloat16().contiguous()
    x, featpre = cabi.visual_embed_fused(fb, Wb, boxes, *args, B, N)
    torch.testing.assert_close(x.cpu(), d["out"], rtol=2e-2, atol=2e-2)          # bf16 operands vs the fp32 reference
    ref_pre = (fb.float() @ Wb.float().t()).contiguous()
    torch.testing.assert_close(featpre, ref_pre, rtol=1e-5, atol=1e-5)
    x2 = cabi.visual_embed_fwd(featpre, boxes, *args, B, N)                       # the stand-alone tail kernel on the same projection
    assert torch.equal(x, x2)
    # 3 row blocks of 256 (two CTA pairs busy + a ragged one), real feature width
    torch.manual_seed(9)
    B2, N2 = 17, 36
    f2 = torch.relu(torch.randn(B2 * N2, 2048, device=DEV)).bfloat16()
    W2 = (torch.randn(768, 2048, device=DEV) * 0.02).bfloat16()
    bx = torch.rand(B2, N2, 4, device=DEV)
    xa, pa = cabi.visual_embed_fused(f2, W2, bx, *args, B2, N2)
    xb = cabi.visual_embed_fwd(pa, bx, *args, B2, N2)
    assert torch.equal(xa, xb) and rel_err(pa, f2.float() @ W2.float().t()) < 3e-5


def test_ce_and_loss_tail():
    torch.manual_seed(2)
    M, V, ld = 40, 32200, 32256
    logits = torch.zeros(M, ld, device=DEV, dtype=torch.bfloat16)
    logits[:, :V] = (torch.randn(M, V, device=DEV) * 3).bfloat16()
    labels = torch.randint(0, V, (M,), device=DEV)
    labels[::7] = -100
    ref = logits[:, :V].float().requires_grad_()
    loss_ref = F.cross_entropy(ref, labels, ignore_index=-100, reduction="none")
    lse, loss = cabi.ce_fwd(logits, labels, V)
    torch.testing.assert_close(loss, loss_ref.detach(), rtol=1e-4, atol=1e-4)
    w = torch.rand(M, device=DEV)
    (loss_ref * w).sum().backward()
    cabi.ce_bwd(logits, labels, V, lse, w)
    assert rel_err(logits[:, :V], ref.grad) < 1e-2
    assert logits[:, V:].abs().max().item() == 0.0
    # loss tail against the fixture made from vqa_model.py:46-54
    d = torch.load(os.path.join(G, "loss_tail.pt"))
    out, wr = cabi.loss_tail(d["loss_rows"].to(DEV), d["labels"].to(DEV), d["scores"].to(DEV))
    torch.testing.assert_close(out.cpu(), d["loss"], rtol=1e-6, atol=1e-7)
    rows = d["loss_rows"].clone().requires_grad_()
    B, T = d["labels"].shape
    m = (d["labels"] != -100).float()
    ((rows.view(B, T) * m).sum(1) / m.sum(1).clamp(min=1) * d["scores"]).mean().backward()
    torch.testing.assert_close(wr.cpu() * m.view(-1), rows.grad * m.view(-1), rtol=1e-6, atol=1e-8)


def test_clip_adamw_matches_hf_semantics():
    torch.manual_seed(3)
    n, n_decay = 4096 * 3, 4096 * 2
    p0 = torch.randn(n)
    pa, pb = torch.nn.Parameter(p0[:n_decay].clone()), torch.nn.Parameter(p0[n_decay:].clone())
    opt = O.HFAdamW([("w", pa), ("b.bias", pb)], lr=1e-3, eps=1e-6, weight_decay=0.01)
    p = p0.clone().to(DEV)
    m = torch.zeros(n, device=DEV)
    v = torch.zeros(n, device=DEV)
    pb16 = torch.zeros(n, device=DEV, dtype=torch.bfloat16)
    for step in range(1, 4):
        g = torch.randn(n) * (10.0 if step == 2 else 0.01)       # step 2 exceeds the clip norm
        pa.grad, pb.grad = g[:n_decay].clone(), g[n_decay:].clone()
        gn = torch.nn.utils.clip_grad_norm_([pa, pb], 5.0)
        opt.step()
        gd = g.to(DEV)
        ss = cabi.grad_sumsq(gd)
        torch.testing.assert_close(ss.sqrt().cpu(), gn.reshape(1), rtol=1e-5, atol=1e-6)
        cabi.adamw(p, gd, m, v, n_decay, 1e-3, 0.9, 0.999, 1e-6, 0.01, step, ss, 5.0, pb16)
        ref = torch.cat([pa.data, pb.data])
        torch.testing.assert_close(p.cpu(), ref, rtol=2e-6, atol=2e-7)
        torch.testing.assert_close(pb16.cpu().float(), ref.bfloat16().float(), rtol=0, atol=0)


def _pack_bits(bits):
    """[M, N] bool -> [M, ceil(N/32)] int32, bit i of word w = column 32 w + i (the ReLU mask layout of the GEMM epilogues)."""
    M, N = bits.shape
    W = (N + 31) // 32
    b = torch.zeros(M, W * 32, device=bits.device, dtype=torch.int64)
    b[:, :N] = bits
    v = (b.view(M, W, 32) << torch.arange(32, device=bits.device)).sum(-1)
    return torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32)


@pytest.mark.parametrize("epi", [0, 1, 2, 3, 4, 5])
def test_gemm_epilogues_ragged(epi):
    torch.manual_seed(4 + epi)
    M, N, K = 1000, 776, 520
    A = torch.randn(M, K, device=DEV).bfloat16()
    Bm = torch.randn(N, K, device=DEV).bfloat16()
    ref = A.float() @ Bm.float().t()
    f32 = epi in (2, 3, 5)
    C = torch.full((M, N), 0.5, device=DEV, dtype=torch.float32 if f32 else torch.bfloat16)
    R = None
    if epi == 1:
        ref = ref.relu()
        R = torch.zeros(M, (N + 31) // 32, device=DEV, dtype=torch.int32)       # sign bitmask output
    elif epi == 2:
        R = torch.randn(M, N, device=DEV)
        ref = ref + R
    elif epi == 3:
        ref = ref + 0.5
    elif epi == 4:
        keep = torch.rand(M, N, device=DEV) > 0.5
        R = _pack_bits(keep)
        ref = ref * keep
    for bn in (64, 128, 256, 512):        # 512 = 256 x 256 tiles on CTA pairs (cta_group::2)
        C.fill_(0.5)
        if epi == 1:
            R.zero_()
        cabi.gemm(A, 0, Bm, 0, C, R, M, N, K, epi, bn=bn)
        torch.cuda.synchronize()
        assert rel_err(C, ref) < (3e-5 if f32 else 1e-2), (epi, bn)
        if epi == 1:
            # the mask marks exactly the stored non-zero activations (bits past column N are don't-care)
            W = R.shape[1]
            got = ((R.long().unsqueeze(-1) >> torch.arange(32, device=DEV)) & 1).view(M, W * 32)[:, :N].bool()
            assert torch.equal(got, C.float() > 0), (epi, bn)


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize("splits", [1, 4])
def test_gemm_operand_majors_and_split_k(a_mn, b_mn, splits):
    """The three operand layouts of the step — forward X W^T (K-major / K-major), dX = dY W (B MN-major), dW = dY^T X (both
    MN-major) — on ragged sizes, every tile shape incl. the CTA-pair kernel, plain and split-K with the atomic fp32 epilogue."""
    torch.manual_seed(20 + a_mn * 2 + b_mn + splits)
    M, N, K = 392, 520, 1000            # ragged in all three dimensions (K not a multiple of 64)
    At = torch.randn(M, K, device=DEV).bfloat16()
    Bt = torch.randn(N, K, device=DEV).bfloat16()
    ref = At.float() @ Bt.float().t()
    A = At.t().contiguous() if a_mn else At          # MN-major = stored transposed ([K, M])
    Bm = Bt.t().contiguous() if b_mn else Bt
    for bn in (64, 128, 256, 512):
        C = torch.full((M, N), 0.25, device=DEV, dtype=torch.float32)
        cabi.gemm(A, a_mn, Bm, b_mn, C, None, M, N, K, 3, splits=splits, bn=bn)      # C += A B^T
        torch.cuda.synchronize()
        assert rel_err(C, ref + 0.25) < 3e-5, (a_mn, b_mn, splits, bn)
        if splits == 1:
            Cb = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
            cabi.gemm(A, a_mn, Bm, b_mn, Cb, None, M, N, K, 0, bn=bn)
            assert rel_err(Cb, ref) < 1e-2, (a_mn, b_mn, bn)


@pytest.mark.parametrize("epi", [1, 2])
def test_gemm_dropout_epilogues_match_host_hash(epi):
    """The ReLU(+dropout) and residual(+dropout) epilogues against a host restatement of the counter-based mask
    (cabi.dropout_scale_host == vq_dropout_pair): same kept set bit for bit, values to bf16 / fp32 round-off."""
    torch.manual_seed(30 + epi)
    M, N, K = 520, 776, 264
    p = 0.1
    thr = int(p * 65536 + 0.5)
    inv = 65536.0 / (65536.0 - thr)
    key = 0x1234ABCD
    A = torch.randn(M, K, device=DEV).bfloat16()
    Bm = torch.randn(N, K, device=DEV).bfloat16()
    acc = A.float() @ Bm.float().t()
    scale = cabi.dropout_scale_host(M, N, thr, inv, key, DEV)
    assert abs((scale == 0).float().mean().item() - p) < 5e-3
    for bn in (128, 256, 512):
        if epi == 1:
            C = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
            R = torch.zeros(M, (N + 31) // 32, device=DEV, dtype=torch.int32)
            cabi.gemm_dropout(A, Bm, C, R, M, N, K, 1, thr, inv, key, bn=bn)
            ref = acc.relu() * scale
            assert rel_err(C, ref) < 1e-2, bn
            W = R.shape[1]
            got = ((R.long().unsqueeze(-1) >> torch.arange(32, device=DEV)) & 1).view(M, W * 32)[:, :N].bool()
            assert torch.equal(got, C.float() > 0), bn
            # dropped positions are exactly zero wherever the pre-dropout activation is clearly positive
            clear = acc > 0.5
            assert torch.equal((C.float() == 0) & clear, (scale == 0) & clear), bn
        else:
            R = torch.randn(M, N, device=DEV)
            C = torch.empty(M, N, device=DEV)
            cabi.gemm_dropout(A, Bm, C, R, M, N, K, 2, thr, inv, key, bn=bn)
            ref = R + acc * scale
            assert rel_err(C, ref) < 3e-5, bn


@pytest.mark.parametrize("bn", [256, 512])
def test_gemm_fused_argmax_epilogue_first_max(bn):
    """EPI_ARGMAX: the greedy token choice straight from the fp32 accumulators (what replaces logits -> argmax in
    generate, vqa_model.py:112-116): per-tile maxima merged = torch.argmax of the fp32 product, including exact ties
    (duplicate vocabulary rows -> lowest index) and a ragged last tile."""
    torch.manual_seed(40)
    M, N, K = 200, 32200, 768
    A = torch.randn(M, K, device=DEV).bfloat16()
    Bm = torch.randn(N, K, device=DEV).bfloat16()
    Bm[777] = Bm[31999]                              # exact tie between two columns for whatever row prefers them
    A[5] = Bm[31999] * 0.5                           # row 5's maximum is that tied pair
    ref = (A.float() @ Bm.float().t()) * 0.125
    slots = ((N + 255) // 256) * 2
    pitch = (slots + 7) // 8 * 8
    pv = torch.full((M, pitch), float("nan"), device=DEV)
    pi = torch.full((M, pitch), -1, device=DEV, dtype=torch.int32)
    cabi.gemm(A, 0, Bm, 0, pv, pi, M, N, K, 6, alpha=0.125, bn=bn)
    v, slot = pv[:, :slots].max(dim=1)
    # lowest index among the slots holding the row maximum
    cand = torch.where(pv[:, :slots] == v[:, None], pi[:, :slots].long(), torch.full_like(pi[:, :slots].long(), 1 << 40))
    idx = cand.min(dim=1).values
    want = ref.argmax(dim=1)
    assert idx[5].item() == 777
    agree = (idx == want)
    # fp32 accumulation order differs from torch's: allow a mismatch only where torch's own top-2 are within round-off
    top2 = ref.topk(2, dim=1).values
    assert bool((agree | ((top2[:, 0] - top2[:, 1]) < 1e-4)).all())
    torch.testing.assert_close(v, ref.max(dim=1).values, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("K,epi", [(1600, 3), (1600, 5), (333 * 8, 3), (64, 5)])
def test_gemm_grouped_weight_gradients_vs_torch(K, epi):
    """Several dW = dY^T X problems in one CTA-pair launch (the decoder's six per layer, plus ragged sizes): every problem's tiles
    land in its own output, accumulate (epi 3) adds to what is there, store (epi 5) overwrites."""
    torch.manual_seed(K + epi)
    shapes = [(768, 3072), (3072, 768), (768, 768), (2304, 768), (200, 520), (768, 768), (8, 8)]
    As = [(torch.randn(K, m, device=DEV) * 0.5).bfloat16() for m, _ in shapes]
    Bs = [(torch.randn(K, n, device=DEV) * 0.5).bfloat16() for _, n in shapes]
    Cs = [torch.randn(m, n, device=DEV) for m, n in shapes]
    before = [c.clone() for c in Cs]
    guard = [torch.full((m + 3, n + 8), 7.0, device=DEV) for m, n in shapes]     # the outputs live inside larger buffers: nothing outside is touched
    for gbuf, c in zip(guard, Cs):
        gbuf[:c.shape[0], :c.shape[1]] = c
    views = [gbuf[:c.shape[0], :c.shape[1]] for gbuf, c in zip(guard, Cs)]
    cabi.gemm_grouped_mn(As, Bs, views, epi=epi, alpha=0.5)
    for i, (a, b) in enumerate(zip(As, Bs)):
        ref = 0.5 * (a.float().t() @ b.float()) + (before[i] if epi == 3 else 0.0)
        assert rel_err(views[i], ref) < 2e-3, (i, shapes[i])
        assert (guard[i][shapes[i][0]:, :] == 7.0).all() and (guard[i][:, shapes[i][1]:] == 7.0).all(), i


@pytest.mark.parametrize("S,Lt,B,masked", [(33, 20, 3, True), (40, 1, 7, False), (64, 32, 4, True), (56, 20, 200, True), (47, 9, 26, False)])
def test_attention_tcgen05_shapes_vs_torch(S, Lt, B, masked):
    """The whole shape range the tcgen05 encoder kernels accept (33..64 positions, 1..32 text tokens, fewer and more items than
    SMs, with and without masked keys): forward, dQ / dK / dV and the bias-table gradient against the fp32 torch formulation."""
    from vqacl_b200.engine import rel_bucket_table
    torch.manual_seed(S * 100 + Lt)
    H = 12
    q = (torch.randn(B * S, H * 64, device=DEV) * 0.3).bfloat16().requires_grad_()
    k = (torch.randn(B * S, H * 64, device=DEV) * 0.3).bfloat16().requires_grad_()
    v = torch.randn(B * S, H * 64, device=DEV).bfloat16().requires_grad_()
    table = (torch.randn(32, H, device=DEV) * 0.5)
    att = O.T5Attention(O.VLT5Config(), False, True).to(DEV)
    att.relative_attention_bias.weight = torch.nn.Parameter(table.clone())
    full = torch.zeros(1, H, S, S, device=DEV)
    full[:, :, :Lt, :Lt] = att.compute_bias(Lt, Lt)
    pad = torch.zeros(B, S, device=DEV)
    if masked:
        pad[B // 2, max(1, Lt // 2):Lt] = -10000.0
        pad[B - 1, Lt - 1:Lt] = -10000.0
    bias = full + pad[:, None, None, :]
    kw = dict(rel_table=table, rel_bucket=rel_bucket_table(True), rel_mode=1, Lt=Lt, keymask=pad.contiguous() if masked else None)
    ref = _attn_ref(q, k, v, B, H, S, S, bias)
    o, lse = cabi.attention_fwd(q.detach(), k.detach(), v.detach(), B, H, S, S, **kw)
    assert rel_err(o, ref.detach()) < 1e-2
    ps = torch.softmax((q.float().view(B, S, H, 64).transpose(1, 2) @ k.float().view(B, S, H, 64).transpose(1, 2).transpose(2, 3) + bias).detach(), -1)
    lse_ref = torch.logsumexp((q.float().view(B, S, H, 64).transpose(1, 2) @ k.float().view(B, S, H, 64).transpose(1, 2).transpose(2, 3) + bias).detach(), -1)
    assert (lse.view(B, H, S) - lse_ref).abs().max() < 2e-2 and ps.isfinite().all()
    dO = torch.randn_like(ref).bfloat16()
    ref.backward(dO.float())
    dq, dk, dv, dtab = cabi.attention_bwd(q.detach(), k.detach(), v.detach(), dO, lse, B, H, S, S, **kw)
    for mine, theirs, nm in ((dq, q.grad, "dq"), (dk, k.grad, "dk"), (dv, v.grad, "dv")):
        assert mine.float().isfinite().all(), nm
        assert cos(mine, theirs) > 0.999 and rel_err(mine, theirs) < 2e-2, nm
    tg = att.relative_attention_bias.weight.grad
    assert cos(dtab, tg) > 0.999 and rel_err(dtab, tg) < 2e-2


@pytest.mark.parametrize("Sq,Sk,mode", [(150, 150, "enc"), (100, 200, "plain"), (5, 152, "cross"), (256, 256, "enc"), (70, 33, "plain")])
def test_attention_multi_tile_fwd_bwd_vs_torch(Sq, Sk, mode):
    """The generic multi-tile kernels (Sq or Sk > 64): encoder form (text x text bias corner + key padding mask), a plain
    rectangular problem and the decoder's cross-attention form (few queries, many keys, -1e9 mask), forward and backward."""
    from vqacl_b200.engine import rel_bucket_table
    torch.manual_seed(7)
    B, H, Lt = 3, 12, 23
    q = (torch.randn(B * Sq, H * 64, device=DEV) * 0.3).bfloat16().requires_grad_()
    k = (torch.randn(B * Sk, H * 64, device=DEV) * 0.3).bfloat16().requires_grad_()
    v = torch.randn(B * Sk, H * 64, device=DEV).bfloat16().requires_grad_()
    table = (torch.randn(32, H, device=DEV) * 0.5)
    pad = torch.zeros(B, Sk, device=DEV)
    kw = {}
    att = None
    if mode == "enc":
        att = O.T5Attention(O.VLT5Config(), False, True).to(DEV)
        att.relative_attention_bias.weight = torch.nn.Parameter(table.clone())
        full = torch.zeros(1, H, Sq, Sk, device=DEV)
        full[:, :, :Lt, :Lt] = att.compute_bias(Lt, Lt)
        pad[1, 9:Lt] = -10000.0
        bias = full + pad[:, None, None, :]
        kw = dict(rel_table=table, rel_bucket=rel_bucket_table(True), rel_mode=1, Lt=Lt, keymask=pad.contiguous())
    elif mode == "cross":
        pad[2, 7:20] = -1e9
        bias = pad[:, None, None, :].expand(B, H, Sq, Sk)
        kw = dict(keymask=pad.contiguous())
    else:
        bias = torch.zeros(B, H, Sq, Sk, device=DEV)
    ref = _attn_ref(q, k, v, B, H, Sq, Sk, bias)
    o, lse = cabi.attention_fwd(q.detach(), k.detach(), v.detach(), B, H, Sq, Sk, **kw)
    assert rel_err(o, ref.detach()) < 1e-2
    dO = torch.randn_like(ref).bfloat16()
    ref.backward(dO.float())
    dq, dk, dv, dtab = cabi.attention_bwd(q.detach(), k.detach(), v.detach(), dO, lse, B, H, Sq, Sk, o_saved=o, **kw)
    for mine, theirs, nm in ((dq, q.grad, "dq"), (dk, k.grad, "dk"), (dv, v.grad, "dv")):
        assert cos(mine, theirs) > 0.999 and rel_err(mine, theirs) < 2e-2, nm
    if att is not None:
        tg = att.relative_attention_bias.weight.grad
        assert cos(dtab, tg) > 0.999 and rel_err(dtab, tg) < 2e-2


@pytest.mark.parametrize("M,K", [(17920, 768), (1000, 3072), (300, 520)])
def test_gemm_residual_with_rmsnorm_row_tail(M, K):
    """The RMSNorm that opens a sub-layer folded into the residual GEMM that closes the previous one (CTA pairs own whole
    256-row blocks and normalise them from L2): C equals the plain residual epilogue bit for bit, the bf16 norm output equals
    the stand-alone rmsnorm kernel on that C bit for bit, and both match torch."""
    torch.manual_seed(50 + K)
    A = (torch.randn(M, K, device=DEV) * 0.5).bfloat16()
    Bm = (torch.randn(768, K, device=DEV) * 0.05).bfloat16()
    R = torch.randn(M, 768, device=DEV) * 3
    w = torch.rand(768, device=DEV) + 0.5
    C, n = cabi.gemm_resid_rmsnorm(A, Bm, R, w)
    C2 = torch.empty(M, 768, device=DEV)
    cabi.gemm(A, 0, Bm, 0, C2, R, M, 768, K, 2, bn=512)
    assert torch.equal(C, C2)
    nb, _ = cabi.rmsnorm_fwd(C, w)
    assert torch.equal(n, nb)
    ref = R + A.float() @ Bm.float().t()
    assert rel_err(C, ref) < 3e-5
    refn = ref * torch.rsqrt(ref.pow(2).mean(-1, keepdim=True) + 1e-6) * w
    assert rel_err(n, refn) < 1e-2
