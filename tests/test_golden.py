"""Pin the oracle against outputs of the reference's own source (tests/golden, made by tools/gen_golden.py)."""
import os

import pytest
import torch

from golden_fixtures import assert_close_to_sample, load_prototype_path, load_vlt5_forward
from helpers import O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_visual_embedding_matches_reference():
    d = torch.load(os.path.join(G, "visual_embedding.pt"))
    cfg = O.VLT5Config(vocab_size=d["vocab"], feat_dim=d["feat_dim"])
    shared = torch.nn.Embedding(d["vocab"], 768)
    ve = O.VisualEmbedding(cfg, shared)
    ve.load_state_dict(d["state"])
    with torch.no_grad():
        out = ve(d["feats"], d["boxes"])
    torch.testing.assert_close(out, d["out"], rtol=1e-6, atol=1e-6)


def test_prototype_state_machine_matches_reference():
    d = load_prototype_path()
    bank = O.PrototypeBank()
    for st in d["steps"]:
        h = st["hidden"].float()
        curQ, numQ = O.calculate_current_prototype(h[:, :20], st["ques_labels"])
        curV, numV = O.calculate_current_prototype(h[:, 20:], st["cate_labels"])
        torch.testing.assert_close(curQ, st["curQ"], rtol=0, atol=0)
        torch.testing.assert_close(curV, st["curV"], rtol=0, atol=0)
        assert torch.equal(numQ, st["numQ"]) and torch.equal(numV, st["numV"])
        bank.update(curQ, curV, numQ, numV, st["task"], d["alpha"], d["beta"])
        torch.testing.assert_close(bank.Q_prototype, st["Q_prototype"], rtol=0, atol=0)
        torch.testing.assert_close(bank.V_prototype, st["V_prototype"], rtol=0, atol=0)
        assert torch.equal(bank.Q_prototype_num, st["Q_num"]) and torch.equal(bank.V_prototype_num, st["V_num"])
        rq, iq = O.cosine_similarity_multi(bank.Q_prototype, h[:, :20].mean(1))
        rv, iv = O.cosine_similarity_multi(bank.V_prototype, h[:, 20:].mean(1))
        assert torch.equal(iq, st["idx_Q"]) and torch.equal(iv, st["idx_V"])
        torch.testing.assert_close(rq, st["retr_Q"], rtol=0, atol=0)
        torch.testing.assert_close(rv, st["retr_V"], rtol=0, atol=0)
    r, i = O.cosine_similarity_multi(d["eval_P"], d["eval_x"])
    assert torch.equal(i, d["eval_idx"])
    torch.testing.assert_close(r, d["eval_retr"], rtol=0, atol=0)


def test_loss_tail_matches_reference():
    d = torch.load(os.path.join(G, "loss_tail.pt"))
    labels, rows, scores = d["labels"], d["loss_rows"], d["scores"]
    B, T = labels.shape
    m = (labels != -100).float()
    loss = ((rows.view(B, T) * m).sum(1) / m.sum(1).clamp(min=1) * scores).mean()
    torch.testing.assert_close(loss, d["loss"], rtol=0, atol=0)


def test_full_forward_glue_matches_reference():
    """JointEncoder.forward + VLT5.forward executed from the reference's text (tools/gen_golden_forward.py): encoder bias /
    mask construction (a3), SI path in place (a9-a13), shift-right, cross mask with the two prototype rows attendable,
    decoder, x d^-1/2, tied LM head, CE(reduction='none') (a7, a8, a14), over four consecutive calls on one model, then one
    step through the reference's VLT5VQA.train_step text (a1)."""
    d = load_vlt5_forward()
    cfg = O.VLT5Config(dropout_rate=0.0, **d["cfg"])
    om = O.VLT5VQA(cfg).eval()
    missing, unexpected = om.load_state_dict(d["state"], strict=False)
    assert not unexpected, unexpected
    assert all(k.startswith(("prototype_fc", "lm_head", "encoder.embed_tokens", "decoder.embed_tokens")) for k in missing), missing
    for c in d["calls"]:
        with torch.no_grad():
            # the additive bias + mask tensor the reference hands to its first encoder block (modeling_t5_our.py:258-273)
            L, S = c["input_ids"].size(1), c["input_ids"].size(1) + c["vis_feats"].size(1)
            mask = torch.cat([c["input_ids"].ne(0).float(), torch.ones(c["input_ids"].size(0), S - L)], 1)
            bias = torch.zeros(1, cfg.num_heads, S, S)
            bias[:, :, :L, :L] = om.encoder.block[0].layer[0].SelfAttention.compute_bias(L, L)
            torch.testing.assert_close(bias + (1.0 - mask[:, None, None, :]) * -10000.0, c["position_bias"], rtol=0, atol=0)
            kw = dict(cate_labels=c["cate_labels"], ques_labels=c["ques_labels"], proto_update=True, task_id=c["task"],
                      alpha=d["alpha"], beta=d["beta"]) if c["proto_update"] else {}
            out = om(c["input_ids"], c["vis_feats"], c["boxes"], c["labels"], **kw)
        assert_close_to_sample(out["encoder_hidden_states"], c["encoder_hidden_states"], rtol=1e-5, atol=1e-5)
        assert torch.equal(out["encoder_attention_mask"], c["encoder_attention_mask"])
        torch.testing.assert_close(out["logits"], c["logits"], rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(out["loss"], c["loss"], rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(om.bank.Q_prototype, c["Q_prototype"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(om.bank.V_prototype, c["V_prototype"], rtol=1e-5, atol=1e-6)
        assert torch.equal(om.bank.Q_prototype_num, c["Q_num"]) and torch.equal(om.bank.V_prototype_num, c["V_num"])
    # one more step through the reference's VLT5VQA.train_step text (vqa_model.py:18-65) on the same model state
    t = d["train_call"]
    with torch.no_grad():
        res = om.train_step({k: t[k] for k in ("input_ids", "vis_feats", "boxes", "target_ids", "cate_labels", "ques_labels", "scores")},
                            t["task"], d["alpha"], d["beta"], 3, 1000)
    assert set(t["keys"]) <= set(res.keys()) and tuple(res["BL"]) == tuple(t["BL"])
    torch.testing.assert_close(res["loss"], t["loss"], rtol=1e-5, atol=1e-6)
    assert_close_to_sample(res["encoder_hidden_states"], t["encoder_hidden_states"], rtol=1e-5, atol=1e-5)
    assert torch.equal(res["encoder_attention_mask"], t["encoder_attention_mask"])
    torch.testing.assert_close(om.bank.Q_prototype, t["Q_prototype"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(om.bank.V_prototype, t["V_prototype"], rtol=1e-5, atol=1e-6)


def test_memory_loss_matches_reference_fixture():
    """oracle.memory_loss against the fixture made by executing the reference's own text of
    VL-T5/nextqa/modeling_t5_nextqa.py:544-555 (tools/gen_golden_memory_loss.py): both losses and the gradient of
    lambda_Q * loss_Q + lambda_V * loss_V with respect to the encoder hidden states."""
    d = torch.load(os.path.join(G, "memory_loss.pt"))
    om = O.VLT5VQA(O.VLT5Config(num_layers=1, num_decoder_layers=1, vocab_size=64))
    om.bank.Q_prototype, om.bank.V_prototype = d["Q_prototype"], d["V_prototype"]
    h = d["hidden"].float().requires_grad_()
    lq, lv = om.memory_loss(h[:, :20], h[:, 20:], d["ques_labels"], d["cate_labels"])
    torch.testing.assert_close(lq.detach(), d["loss_Q"], rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(lv.detach(), d["loss_V"], rtol=1e-6, atol=1e-6)
    (d["lambda_Q"] * lq + d["lambda_V"] * lv).backward()
    torch.testing.assert_close(h.grad[:, 0], d["grad_hidden_q_row"], rtol=1e-6, atol=1e-8)
    torch.testing.assert_close(h.grad[:, 25], d["grad_hidden_v_row"], rtol=1e-6, atol=1e-8)
