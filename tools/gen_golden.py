"""Generate tests/golden/*.pt by EXECUTING the reference's own source text (run in the build container only).

The reference module cannot be imported here (transformers 5.5 != 4.2.1, SURVEY.md H3), but the classes / methods on the
hot path that do not depend on the 4.2.1 internals can be lifted out of the file with `ast` and executed unmodified:
  * class VisualEmbedding                      VL-T5/src/modeling_t5_our.py:27-143  (against transformers-5.5 T5LayerNorm,
                                                whose arithmetic equals 4.2.1's)
  * VLT5.cosine_similarity_multi / update_prototype / calculate_current_prototype     :434-511
    (the only edit: the hard-coded torch.device('cuda') string at :504 is evaluated on CPU)
  * the loss tail of VLT5VQA.train_step         VL-T5/src/vqa_model.py:46-54
The fixtures hold seeded inputs and the reference's outputs; tests/test_golden.py checks the oracle against them on CPU
and tests/test_gpu_ops.py checks the CUDA path. Nothing is copied into the repo except these tensors (prototype_path.pt
in the compact layout of tests/golden_fixtures.py: seeded inputs are regenerated, not stored). (tools/gen_golden_forward.py does the same for the glue of a whole
call: JointEncoder.forward + VLT5.forward.)

    python tools/gen_golden.py [/root/reference]
"""
import ast
import os
import sys
import types

import torch
import torch.nn as nn

REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
sys.path.insert(0, os.path.dirname(OUT))
from golden_fixtures import pack_prototype_path, prototype_inputs  # noqa: E402  (seeded inputs + the stored layout)
SRC = os.path.join(REF, "VL-T5", "src", "modeling_t5_our.py")
SRC_VQA = os.path.join(REF, "VL-T5", "src", "vqa_model.py")


def lift(path, class_name, only=None):
    """Source text of `class_name` (optionally only the listed methods) from the reference file."""
    text = open(path).read()
    tree = ast.parse(text)
    lines = text.splitlines()
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name == class_name:
            if only is None:
                return "\n".join(lines[node.lineno - 1:node.end_lineno])
            out = [f"class {class_name}:"]
            for f in node.body:
                if isinstance(f, ast.FunctionDef) and f.name in only:
                    out.append("\n".join(lines[f.lineno - 1:f.end_lineno]))
            return "\n".join(out)
    raise KeyError(class_name)


def main():
    from transformers.models.t5.modeling_t5 import T5LayerNorm
    import torch.nn.functional as F
    ns = dict(torch=torch, nn=nn, F=F, T5LayerNorm=T5LayerNorm)
    exec(lift(SRC, "VisualEmbedding"), ns)
    proto_src = lift(SRC, "VLT5", only=["cosine_similarity_multi", "update_prototype", "calculate_current_prototype"])
    # the only edit: run the hard-coded 'cuda' device on CPU (SURVEY.md H8)
    assert "torch.device('cuda')" in proto_src
    proto_src = proto_src.replace("torch.device('cuda')", "torch.device('cpu')")
    exec(proto_src, ns)
    VisualEmbedding, VLT5 = ns["VisualEmbedding"], ns["VLT5"]
    os.makedirs(OUT, exist_ok=True)

    # ---------------------------------------------------------------- VisualEmbedding
    g = torch.Generator().manual_seed(101)
    cfg = types.SimpleNamespace(feat_dim=64, pos_dim=4, n_images=2, d_model=768, layer_norm_epsilon=1e-6,
                                individual_vis_layer_norm=True, use_vis_layer_norm=True, use_vis_order_embedding=True)
    shared = nn.Embedding(200, 768)
    ve = VisualEmbedding(cfg, shared)
    with torch.no_grad():
        for p in ve.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.05 if p.dim() > 1 else 1.0))
    B, N = 3, 7
    feats = torch.relu(torch.randn(B, N, 64, generator=g))
    xy = torch.rand(B, N, 2, generator=g) * 0.7
    boxes = torch.cat([xy, xy + torch.rand(B, N, 2, generator=g) * 0.25 + 0.05], dim=2)
    with torch.no_grad():
        out = ve(feats, boxes)
    torch.save(dict(state={k: v.clone() for k, v in ve.state_dict().items()}, feats=feats, boxes=boxes, out=out,
                    vocab=200, feat_dim=64), os.path.join(OUT, "visual_embedding.pt"))

    # ---------------------------------------------------------------- prototype functions
    m = VLT5.__new__(VLT5)          # no __init__: only the dict/attribute state the three methods touch
    m.Q_task_mem_proto, m.Q_task_cur_proto = {}, {}
    # task 0: two steps; task 2: three steps (first / first-mem / EMA); task 5: one step. alpha .5 beta .3
    steps, P, x = prototype_inputs()
    for st in steps:
        hidden, ql, cl, task = st["hidden"], st["ques_labels"], st["cate_labels"], st["task"]
        curQ, numQ = m.calculate_current_prototype(hidden[:, :20, :], ql)
        curV, numV = m.calculate_current_prototype(hidden[:, 20:, :], cl)
        m.update_prototype(curQ, curV, numQ, numV, task, 0.5, 0.3)
        rq, iq, _ = m.cosine_similarity_multi(m.Q_prototype, torch.mean(hidden[:, :20, :], dim=1), ql)
        rv, iv, _ = m.cosine_similarity_multi(m.V_prototype, torch.mean(hidden[:, 20:, :], dim=1), cl)
        st.update(curQ=curQ.clone(), curV=curV.clone(), numQ=numQ.clone(), numV=numV.clone(), Q_prototype=m.Q_prototype.clone(),
                  V_prototype=m.V_prototype.clone(), Q_num=m.Q_prototype_num.clone(), V_num=m.V_prototype_num.clone(),
                  retr_Q=rq.clone(), idx_Q=iq.clone(), retr_V=rv.clone(), idx_V=iv.clone())
    # eval-time retrieval without labels, with an all-zero row present (tie-break / zero-row behaviour, SURVEY.md a12)
    rq, iq, _ = m.cosine_similarity_multi(P, x)
    torch.save(pack_prototype_path(steps, 0.5, 0.3, P, x, rq, iq), os.path.join(OUT, "prototype_path.pt"))

    # ---------------------------------------------------------------- loss tail (vqa_model.py:46-54)
    text = open(SRC_VQA).read().splitlines()
    i0 = next(i for i, l in enumerate(text) if "lm_mask = (lm_labels != -100).float()" in l)
    i1 = next(i for i, l in enumerate(text) if l.strip() == "loss = loss.mean()")
    import textwrap
    tail = textwrap.dedent("\n".join(text[i0:i1 + 1]))
    g = torch.Generator().manual_seed(303)
    Bt, T = 7, 5
    lm_labels = torch.randint(3, 100, (Bt, T), generator=g)
    lm_labels[0, 2:] = -100
    lm_labels[3, 1:] = -100
    lm_labels[5, :] = -100                      # a row with no valid label: clamp(min=1) path
    rows = torch.rand(Bt * T, generator=g) * 5
    rows = rows * (lm_labels.view(-1) != -100).float()   # CE(reduction='none') gives 0 at ignored positions
    scores = torch.tensor([0.3, 0.6, 0.9, 1.0, 0.3, 0.6, 0.9])
    env = dict(torch=torch, lm_labels=lm_labels, output={"loss": rows.clone()}, batch={"scores": scores}, device="cpu")
    exec(tail, env)
    torch.save(dict(labels=lm_labels, loss_rows=rows, scores=scores, loss=env["loss"].clone()), os.path.join(OUT, "loss_tail.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
