"""Generate tests/golden/vlt5_forward.pt by EXECUTING the reference's own `JointEncoder.forward` and `VLT5.forward` text
(VL-T5/src/modeling_t5_our.py:175-339 and :514-713) — the glue of SURVEY.md §8 a3, a7, a8, a13, a14 — in the build
container. Companion of tools/gen_golden.py (which pins a2, a9-a12 and the loss tail).

The two methods are lifted from the file with `ast` and run unmodified. What they call into is provided as follows:
  * VisualEmbedding, calculate_current_prototype / update_prototype / cosine_similarity_multi, VLSeq2SeqLMOutput:
    the reference's own text, lifted the same way (only edit: the hard-coded torch.device('cuda') at :504 -> 'cpu');
  * T5Block / decoder T5Stack / T5LayerNorm / _shift_right / compute_bias: the installed transformers-5.5 modules, whose
    arithmetic equals the 4.2.1 release the reference imports (SURVEY.md §8c), behind two thin adapters that translate the
    4.2.1 calling convention the reference uses (keyword `head_mask`, `past_key_value`; block returns
    (hidden, present_key_value, position_bias)) to 5.5's;
  * `get_extended_attention_mask(mask, shape, device)`: the 4.2.1 value (1 - mask[:, None, None, :]) * -10000.0 (5.5 changed
    the signature and the constant); `get_head_mask`: [None] * n. These two lines are restated, not executed.
Weights are tiny (d_model must stay 768 — the reference hard-codes it at :503 — but 2 heads x 16, d_ff 64, 1 + 1 layers) and
stored in the fixture under the reference's state_dict names; tests/test_golden.py loads them into the oracle and compares
every output of four consecutive forward calls (first step of task 0, two steps of task 2 incl. a rehearsal batch, an eval
call with frozen banks) and of one more step through the reference's VLT5VQA.train_step text (vqa_model.py:18-65).

    python tools/gen_golden_forward.py [/root/reference]
"""
import os
import sys
import types
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gen_golden import lift  # noqa: E402
from golden_fixtures import pack_vlt5_forward  # noqa: E402  (gen_golden puts tests/ on the path)

REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
SRC = os.path.join(REF, "VL-T5", "src", "modeling_t5_our.py")

D, DKV, H, FF, VOCAB, FEAT, LT, NB, T = 768, 16, 2, 64, 120, 32, 20, 6, 4


def main():
    from transformers import T5Config
    from transformers.modeling_outputs import BaseModelOutput, BaseModelOutputWithPastAndCrossAttentions
    from transformers.models.t5 import modeling_t5 as hf
    from transformers.utils import ModelOutput

    ns = dict(torch=torch, nn=nn, F=F, T5LayerNorm=hf.T5LayerNorm, BaseModelOutput=BaseModelOutput,
              BaseModelOutputWithPastAndCrossAttentions=BaseModelOutputWithPastAndCrossAttentions, ModelOutput=ModelOutput,
              CrossEntropyLoss=nn.CrossEntropyLoss, dataclass=dataclass, Optional=Optional, Tuple=Tuple, List=List, Dict=Dict,
              Any=Any)
    exec(lift(SRC, "VisualEmbedding"), ns)
    exec(lift(SRC, "VLSeq2SeqLMOutput"), ns)
    ns["VLSeq2SeqLMOutput"] = dataclass(ns["VLSeq2SeqLMOutput"])   # `lift` starts at the `class` line: re-apply the decorator of :774
    enc_forward_src = lift(SRC, "JointEncoder", only=["forward"])
    exec(enc_forward_src, ns)
    vlt5_src = lift(SRC, "VLT5", only=["forward", "cosine_similarity_multi", "update_prototype", "calculate_current_prototype"])
    assert "torch.device('cuda')" in vlt5_src
    exec(vlt5_src.replace("torch.device('cuda')", "torch.device('cpu')"), ns)
    VisualEmbedding, JointEncoder, VLT5 = ns["VisualEmbedding"], ns["JointEncoder"], ns["VLT5"]
    # VLT5VQA.train_step (vqa_model.py:18-65) on top of that forward: `self(...)` and `self.parameters()` are all it needs
    VLT5.__call__ = VLT5.forward
    exec(lift(os.path.join(REF, "VL-T5", "src", "vqa_model.py"), "VLT5VQA", only=["train_step"]).replace(
        "class VLT5VQA:", "class VLT5VQA(VLT5):"), ns)
    VLT5VQA = ns["VLT5VQA"]

    cfg = T5Config(vocab_size=VOCAB, d_model=D, d_kv=DKV, d_ff=FF, num_layers=1, num_decoder_layers=1, num_heads=H,
                   relative_attention_num_buckets=32, relative_attention_max_distance=128, dropout_rate=0.0,
                   feed_forward_proj="relu", tie_word_embeddings=True, decoder_start_token_id=0, pad_token_id=0, eos_token_id=1,
                   use_cache=False)
    cfg.feat_dim, cfg.pos_dim, cfg.n_images = FEAT, 4, 2
    cfg.individual_vis_layer_norm = cfg.use_vis_layer_norm = cfg.use_vis_order_embedding = True
    g = torch.Generator().manual_seed(404)
    shared = nn.Embedding(VOCAB, D)

    # ---- encoder object the reference's JointEncoder.forward runs on
    class Block421(nn.Module):
        """transformers-5.5 T5Block called the 4.2.1 way."""
        def __init__(self, blk):
            super().__init__()
            self.blk = blk
            self.layer = blk.layer
            self.seen_bias = None

        def forward(self, hidden_states, attention_mask=None, position_bias=None, encoder_hidden_states=None,
                    encoder_attention_mask=None, encoder_decoder_position_bias=None, head_mask=None, past_key_value=None,
                    use_cache=None, output_attentions=None):
            assert head_mask is None and past_key_value is None and encoder_hidden_states is None
            self.seen_bias = position_bias.detach().clone()
            out = self.blk(hidden_states, attention_mask=attention_mask, position_bias=position_bias)
            return (out[0], None, out[1])

    enc_cfg = T5Config(**{**cfg.to_dict(), "is_decoder": False, "use_cache": False})
    enc = types.SimpleNamespace(
        embed_tokens=shared, visual_embedding=VisualEmbedding(cfg, shared),
        block=nn.ModuleList([Block421(hf.T5Block(enc_cfg, has_relative_attention_bias=True, layer_idx=0))]),
        final_layer_norm=hf.T5LayerNorm(D, eps=1e-6), dropout=nn.Dropout(0.0), config=enc_cfg, is_decoder=False,
        get_extended_attention_mask=lambda mask, shape, device: (1.0 - mask[:, None, None, :]) * -10000.0,   # HF 4.2.1
        get_head_mask=lambda head_mask, n: [None] * n)

    # ---- decoder: transformers-5.5 T5Stack behind the 4.2.1 keyword set
    dec_cfg = T5Config(**{**cfg.to_dict(), "is_decoder": True, "use_cache": False, "num_layers": 1})
    dec_stack = hf.T5Stack(dec_cfg)
    dec_stack.set_input_embeddings(shared)
    dec_stack.eval()

    def decoder(input_ids=None, attention_mask=None, inputs_embeds=None, past_key_values=None, encoder_hidden_states=None,
                encoder_attention_mask=None, head_mask=None, use_cache=None, output_attentions=None, output_hidden_states=None,
                return_dict=None):
        assert head_mask is None and past_key_values is None and attention_mask is None and inputs_embeds is None
        return dec_stack(input_ids=input_ids, encoder_hidden_states=encoder_hidden_states,
                         encoder_attention_mask=encoder_attention_mask, use_cache=False, return_dict=True)

    # ---- the VLT5 object the reference's VLT5.forward runs on (no __init__: exactly the attributes the method touches)
    m = VLT5VQA.__new__(VLT5VQA)
    m.parameters = lambda: iter([shared.weight])
    m.config = cfg
    m.encoder = lambda **kw: JointEncoder.forward(enc, **kw)
    m.decoder = decoder
    m.lm_head = nn.Linear(D, VOCAB, bias=False)
    m.lm_head.weight = shared.weight
    m.model_dim = D
    m.L = 20
    m.Q_task_mem_proto, m.Q_task_cur_proto = {}, {}
    m._shift_right = types.MethodType(hf.T5PreTrainedModel._shift_right, types.SimpleNamespace(config=cfg))

    # ---- weights: HF init scheme at these sizes (any values pin the glue; N(0,1) visual linears as in the reference, H14)
    mods = dict(shared=shared, ve=enc.visual_embedding, eblk=enc.block[0].blk, efin=enc.final_layer_norm, dec=dec_stack)
    with torch.no_grad():
        for name, mod in mods.items():
            for pn, p in mod.named_parameters():
                if "shared" in pn or "embed_tokens" in pn or "obj_order_embedding" in pn:
                    continue
                std = 1.0 if p.dim() == 1 else 0.06
                p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=g) if "layer_norm" in pn or pn == "weight" and p.dim() == 1
                        else torch.randn(p.shape, generator=g) * std)
        shared.weight.copy_(torch.randn(VOCAB, D, generator=g))

    def batch(seed, task, rehearsal):
        gg = torch.Generator().manual_seed(seed)
        B = 5
        ids = torch.zeros(B, LT, dtype=torch.long)
        for b in range(B):
            n = LT if b == 0 else int(torch.randint(6, LT + 1, (1,), generator=gg))
            ids[b, :n - 1] = torch.randint(3, VOCAB - 1, (n - 1,), generator=gg)
            ids[b, n - 1] = 1
        feats = torch.relu(torch.randn(B, NB, FEAT, generator=gg))
        xy = torch.rand(B, NB, 2, generator=gg) * 0.7
        boxes = torch.cat([xy, xy + torch.rand(B, NB, 2, generator=gg) * 0.25 + 0.05], dim=2)
        labels = torch.full((B, T), -100, dtype=torch.long)
        for b in range(B):
            n = int(torch.randint(2, T + 1, (1,), generator=gg))
            labels[b, :n - 1] = torch.randint(3, VOCAB - 1, (n - 1,), generator=gg)
            labels[b, n - 1] = 1
        ql = torch.zeros(B, 10)
        qcls = torch.randint(0, task, (B,), generator=gg) if rehearsal else torch.full((B,), task)
        ql[torch.arange(B), qcls] = 1
        cl = torch.zeros(B, 80)
        cl[torch.arange(B), torch.randint(0, 80, (B,), generator=gg)] = 1
        return dict(input_ids=ids, vis_feats=feats, boxes=boxes, labels=labels, ques_labels=ql, cate_labels=cl)

    calls = []
    schedule = [(0, False, True), (2, False, True), (2, True, True), (2, False, False)]   # (task, rehearsal batch, proto_update)
    with torch.no_grad():
        for i, (task, reh, upd) in enumerate(schedule):
            b = batch(500 + i, task, reh)
            kw = dict(cate_labels=b["cate_labels"], ques_labels=b["ques_labels"], proto_update=True, current_task_id=task,
                      proto_alpha=0.5, proto_beta=0.3) if upd else {}
            out = m.forward(input_ids=b["input_ids"], vis_inputs=(b["vis_feats"], b["boxes"]), labels=b["labels"],
                            return_dict=True, **kw)
            calls.append(dict(task=task, proto_update=upd, **b, loss=out.loss.clone(), logits=out.logits.clone(),
                              encoder_hidden_states=out.encoder_hidden_states.clone(),
                              encoder_attention_mask=out.encoder_attention_mask.clone(),
                              position_bias=enc.block[0].seen_bias.clone(), Q_prototype=m.Q_prototype.clone(),
                              V_prototype=m.V_prototype.clone(), Q_num=m.Q_prototype_num.clone(), V_num=m.V_prototype_num.clone()))
    # one more training call through the reference's VLT5VQA.train_step text (kwargs plumbing, loss tail, result dict)
    with torch.no_grad():
        b = batch(510, 2, False)
        b["target_ids"] = b.pop("labels")
        b["scores"] = torch.tensor([0.3, 0.6, 0.9, 1.0, 0.6])
        res = m.train_step(b, 2, 0.5, 0.3, 3, 1000)
    train_call = dict(task=2, **b, loss=res["loss"].clone(), BL=res["BL"], keys=sorted(res.keys()),
                      encoder_hidden_states=res["encoder_hidden_states"].clone(),
                      encoder_attention_mask=res["encoder_attention_mask"].clone(), Q_prototype=m.Q_prototype.clone(),
                      V_prototype=m.V_prototype.clone())
    # state under the reference's names (modeling_t5_our.py state_dict layout, SURVEY.md §8b)
    state = {"shared.weight": shared.weight.detach().clone()}
    for k, v in enc.visual_embedding.state_dict().items():
        state["encoder.visual_embedding." + k] = v.clone()
    for k, v in enc.block[0].blk.state_dict().items():
        state["encoder.block.0." + k] = v.clone()
    state["encoder.final_layer_norm.weight"] = enc.final_layer_norm.weight.detach().clone()
    for k, v in dec_stack.state_dict().items():
        if not k.startswith("embed_tokens"):
            state["decoder." + k] = v.clone()
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, "vlt5_forward.pt")
    torch.save(pack_vlt5_forward(calls, train_call, state, dict(vocab_size=VOCAB, d_model=D, d_kv=DKV, d_ff=FF, num_heads=H, feat_dim=FEAT,
                                                                num_layers=1, num_decoder_layers=1), 0.5, 0.3), path)
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
