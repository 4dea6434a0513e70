"""Generates tests/golden/*.npz by executing the REFERENCE's own Python code (a checkout of thunlp/OpenMatch):

    python tests/golden/make_golden.py <path to the OpenMatch checkout>

The tests do not need the reference, so the vectors are committed.  The models' weights are stored as recipes
(openmatch_b200.synthetic.recipe_state_dict, with the standard deviations of HF's initialisation) from which the
tests rebuild them bit for bit; inputs and the reference's outputs are stored as arrays.  What is executed
unmodified from the reference:
  * openmatch.modeling.DRModelForInference.encode_passage / encode_query  (dense_retrieval_model.py:133-161,261-282)
  * openmatch.loss.SimpleContrastiveLoss                                 (loss.py:7-15)  + torch autograd
  * openmatch.modeling.DRModel.forward (training loss)                    (dense_retrieval_model.py:89-131)
  * openmatch.utils.mean_pooling, merge_retrieval_results_by_score        (utils.py:215-235)
  * openmatch.retriever.Retriever.build_all / retrieve                    (dense_retriever.py:60-206) with the
    oracle's FlatIPIndex injected as the `faiss` module (faiss itself is not installable here).
Models are randomly initialised HF modules (no checkpoints on disk, no network).
"""
import json
import os
import sys
import tempfile
import types
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF_SRC = os.path.join(os.path.abspath(sys.argv[1]), "src") if len(sys.argv) == 2 else None
if REF_SRC is None or not os.path.isdir(os.path.join(REF_SRC, "openmatch")):
    sys.exit("usage: make_golden.py <path to the OpenMatch checkout>")
sys.path.insert(0, REF_SRC)

import importlib.machinery  # noqa: E402

from oracle.flat_index import FlatIPIndex  # noqa: E402
from openmatch_b200.synthetic import recipe_state_dict  # noqa: E402

# faiss shim so that `import faiss` in openmatch.retriever succeeds (datasets probes find_spec -> needs __spec__)
faiss = types.ModuleType("faiss")
faiss.__spec__ = importlib.machinery.ModuleSpec("faiss", None)
faiss.IndexFlatIP = FlatIPIndex
sys.modules["faiss"] = faiss

from transformers import BertConfig, BertModel, T5Config, T5EncoderModel  # noqa: E402

from openmatch.arguments import DataArguments, ModelArguments  # noqa: E402
from openmatch.loss import SimpleContrastiveLoss  # noqa: E402
from openmatch.modeling import DRModel, DRModelForInference  # noqa: E402
from openmatch.modeling.linear import LinearHead  # noqa: E402
from openmatch.utils import mean_pooling, merge_retrieval_results_by_score  # noqa: E402


def synth_ids(gen, B, L, vocab, cls_id, sep_id, ragged):
    ids = torch.randint(10, vocab, (B, L), generator=gen)
    mask = torch.ones(B, L, dtype=torch.long)
    if ragged:
        lens = torch.randint(3, L + 1, (B,), generator=gen)
        lens[0] = L
        for b in range(B):
            mask[b, lens[b]:] = 0
            ids[b, lens[b]:] = 0
            ids[b, lens[b] - 1] = sep_id
    else:
        ids[:, -1] = sep_id
    if cls_id is not None:
        ids[:, 0] = cls_id
    return ids, mask


def set_recipe_weights(module):
    """Replaces every floating-point tensor of the module's state dict with zero-mean recipe weights of the tensor's
    standard deviation (constant tensors keep their value, tied tensors share one seed) and returns the recipe as JSON."""
    recipe, seeds = [], {}
    sd = module.state_dict()
    for name, t in sd.items():
        if not t.is_floating_point():
            continue
        seed = seeds.setdefault(t.data_ptr(), zlib.crc32(name.encode()))
        std = float("%.4g" % float(t.std())) if t.numel() > 1 else 0.0
        recipe.append([name, list(t.shape), float(t.flatten()[0]) if std == 0.0 else 0.0, std, seed])
    with torch.no_grad():
        for name, w in recipe_state_dict(recipe).items():
            sd[name].copy_(w)
    return json.dumps(recipe)


def main():
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(1234)
    out = {}

    # ---------------- BERT, CLS pooling, no head (the reference's default DR config) ----------------
    bcfg = BertConfig(vocab_size=512, hidden_size=128, num_hidden_layers=2, num_attention_heads=2,
                      intermediate_size=512, max_position_embeddings=128)
    bert = BertModel(bcfg).eval()
    bert_recipe = set_recipe_weights(bert)
    margs = ModelArguments(model_name_or_path="unused", pooling="first", normalize=False)
    model = DRModelForInference(lm_q=bert, lm_p=bert, tied=True, pooling="first", normalize=False, model_args=margs)
    ids, mask = synth_ids(gen, 6, 32, 512, 101, 102, ragged=True)
    tt = torch.zeros_like(ids)
    hidden, reps = model.encode_passage({"input_ids": ids, "attention_mask": mask, "token_type_ids": tt})
    np.savez_compressed(os.path.join(HERE, "bert_small.npz"), input_ids=ids.numpy(), attention_mask=mask.numpy(),
                        token_type_ids=tt.numpy(), hidden=hidden.numpy(), reps=reps.numpy(), sd_recipe=bert_recipe)

    # ---------------- T5 encoder, mean pooling + linear head + normalise (GTR-style) ----------------
    tcfg = T5Config(vocab_size=512, d_model=128, d_kv=64, d_ff=512, num_layers=2, num_heads=2,
                    feed_forward_proj="relu")
    t5 = T5EncoderModel(tcfg).eval()
    t5_recipe = set_recipe_weights(t5)
    head = LinearHead(128, 128)
    head_recipe = set_recipe_weights(head)  # one entry: "linear.weight"
    margs = ModelArguments(model_name_or_path="unused", pooling="mean", normalize=True, encoder_only=True)
    model = DRModelForInference(lm_q=t5, lm_p=t5, tied=True, pooling="mean", normalize=True, head_q=head, head_p=head,
                                model_args=margs)
    ids, mask = synth_ids(gen, 6, 32, 512, None, 1, ragged=True)
    hidden, reps = model.encode_passage({"input_ids": ids, "attention_mask": mask})
    np.savez_compressed(os.path.join(HERE, "t5_small.npz"), input_ids=ids.numpy(), attention_mask=mask.numpy(),
                        hidden=hidden.numpy(), reps=reps.numpy(), sd_recipe=t5_recipe, head_recipe=head_recipe)

    # ---------------- T5 relative-position buckets for every distance the encoder can see ----------------
    from transformers.models.t5.modeling_t5 import T5Attention
    rel = torch.arange(-600, 601)
    out["t5_bucket_rel"] = rel.numpy()
    out["t5_bucket"] = T5Attention._relative_position_bucket(rel, bidirectional=True, num_buckets=32,
                                                              max_distance=128).numpy()

    # ---------------- mean_pooling ----------------
    h = torch.randn(4, 7, 16, generator=gen)
    m = torch.tensor([[1] * 7, [1, 1, 1, 0, 0, 0, 0], [1, 0, 0, 0, 0, 0, 0], [0] * 7])
    out["mp_hidden"], out["mp_mask"], out["mp_out"] = h.numpy(), m.numpy(), mean_pooling(h, m).numpy()

    # ---------------- SimpleContrastiveLoss forward + autograd backward ----------------
    for tag, nq, n_p, d in (("a", 8, 64, 32), ("b", 5, 15, 24)):
        x = (torch.randn(nq, d, generator=gen) * 0.5).requires_grad_()
        y = (torch.randn(n_p, d, generator=gen) * 0.5).requires_grad_()
        loss = SimpleContrastiveLoss()(x, y)
        loss.backward()
        out[f"loss_{tag}_x"], out[f"loss_{tag}_y"] = x.detach().numpy(), y.detach().numpy()
        out[f"loss_{tag}_loss"] = np.float32(loss.item())
        out[f"loss_{tag}_dx"], out[f"loss_{tag}_dy"] = x.grad.numpy(), y.grad.numpy()
    # explicit target + reduction='sum'
    x = torch.randn(4, 16, generator=gen).requires_grad_()
    y = torch.randn(12, 16, generator=gen).requires_grad_()
    tgt = torch.tensor([3, 0, 11, 7])
    loss = SimpleContrastiveLoss()(x, y, target=tgt, reduction="sum")
    loss.backward()
    out.update(loss_c_x=x.detach().numpy(), loss_c_y=y.detach().numpy(), loss_c_target=tgt.numpy(),
               loss_c_loss=np.float32(loss.item()), loss_c_dx=x.grad.numpy(), loss_c_dy=y.grad.numpy())

    # ---------------- DRModel.forward training loss (encode both sides, scores, CE) ----------------
    margs = ModelArguments(model_name_or_path="unused", pooling="first", normalize=False)
    dargs = DataArguments(train_n_passages=4)
    targs = types.SimpleNamespace(negatives_x_device=False, per_device_train_batch_size=3)
    train_model = DRModel(lm_q=bert, lm_p=bert, tied=True, pooling="first", normalize=False, model_args=margs,
                          data_args=dargs, train_args=targs).eval()
    qids, qmask = synth_ids(gen, 3, 16, 512, 101, 102, ragged=True)
    pids, pmask = synth_ids(gen, 12, 32, 512, 101, 102, ragged=True)
    o = train_model(query={"input_ids": qids, "attention_mask": qmask, "token_type_ids": torch.zeros_like(qids)},
                    passage={"input_ids": pids, "attention_mask": pmask, "token_type_ids": torch.zeros_like(pids)})
    out.update(fwd_q_ids=qids.numpy(), fwd_q_mask=qmask.numpy(), fwd_p_ids=pids.numpy(), fwd_p_mask=pmask.numpy(),
               fwd_loss=np.float32(o.loss.item()), fwd_scores=o.scores.detach().numpy(),
               fwd_q_reps=o.q_reps.detach().numpy(), fwd_p_reps=o.p_reps.detach().numpy())

    # ---------------- merge_retrieval_results_by_score ----------------
    r1 = {"q1": {"d1": 3.0, "d2": 1.0, "d3": 2.0}, "q2": {"d9": 0.5}}
    r2 = {"q1": {"d2": 9.0, "d4": 2.5, "d5": 2.0}, "q3": {"d1": 1.0}}
    merged = merge_retrieval_results_by_score([r1, r2], topk=3)
    out["merge_repr"] = np.array(repr({k: list(v.items()) for k, v in merged.items()}))

    # ---------------- Retriever.build_all + retrieve, unmodified, over the faiss shim ----------------
    from torch.utils.data import IterableDataset

    from openmatch.retriever import Retriever

    class Synth(IterableDataset):
        def __init__(self, prefix, ids, mask):
            self.prefix, self.ids, self.mask = prefix, ids, mask

        def __iter__(self):
            for i in range(self.ids.shape[0]):
                yield {"text_id": f"{self.prefix}{i}", "input_ids": self.ids[i].tolist(),
                       "attention_mask": self.mask[i].tolist(), "token_type_ids": [0] * self.ids.shape[1]}

    cids, cmask = synth_ids(gen, 50, 32, 512, 101, 102, ragged=True)
    qids, qmask = synth_ids(gen, 3, 16, 512, 101, 102, ragged=True)
    with tempfile.TemporaryDirectory() as tmp:
        args = types.SimpleNamespace(device=torch.device("cpu"), fp16=False, per_device_eval_batch_size=16,
                                     dataloader_num_workers=0, dataloader_pin_memory=False, output_dir=tmp,
                                     process_index=0, local_process_index=0, world_size=1, use_gpu=False)
        model = DRModelForInference(lm_q=bert, lm_p=bert, tied=True, pooling="first", normalize=False,
                                    model_args=margs)
        retriever = Retriever.build_all(model, Synth("d", cids, cmask), args)
        result = retriever.retrieve(Synth("q", qids, qmask), topk=5)
    out.update(ret_c_ids=cids.numpy(), ret_c_mask=cmask.numpy(), ret_q_ids=qids.numpy(), ret_q_mask=qmask.numpy())
    out["ret_docids"] = np.array([[d for d in result[f"q{i}"]] for i in range(3)])
    out["ret_scores"] = np.array([[result[f"q{i}"][d] for d in result[f"q{i}"]] for i in range(3)], dtype=np.float32)

    np.savez_compressed(os.path.join(HERE, "misc.npz"), **out)
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
