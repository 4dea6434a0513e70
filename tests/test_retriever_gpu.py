"""GPU, end to end through the drop-in Python API: DRModelForInference (CUDA encoder) + Retriever (HBM index)
against what the REFERENCE's unmodified Retriever.build_all / retrieve produced for the same weights and
inputs (tests/golden/misc.npz, made by tests/golden/make_golden.py), and DRModel.forward's training loss
against the reference's."""
import os
import pickle
import types

import numpy as np
import pytest
import torch
from torch.utils.data import IterableDataset

pytestmark = pytest.mark.gpu


class Synth(IterableDataset):
    def __init__(self, prefix, ids, mask):
        self.prefix, self.ids, self.mask = prefix, ids, mask

    def __iter__(self):
        for i in range(self.ids.shape[0]):
            yield {"text_id": f"{self.prefix}{i}", "input_ids": self.ids[i].tolist(),
                   "attention_mask": self.mask[i].tolist(), "token_type_ids": [0] * self.ids.shape[1]}


@pytest.fixture(scope="module")
def small_bert(golden_dir):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from transformers import BertConfig, BertModel

    from openmatch_b200.synthetic import recipe_state_dict
    z = np.load(os.path.join(golden_dir, "bert_small.npz"))
    cfg = BertConfig(vocab_size=512, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
                     max_position_embeddings=128)
    lm = BertModel(cfg)
    sd = recipe_state_dict(z["sd_recipe"])
    missing, unexpected = lm.load_state_dict(sd, strict=False)
    assert not [m for m in missing if "position_ids" not in m], missing
    return lm.eval()


def _args(tmp, **kw):
    base = dict(device=torch.device("cuda"), fp16=False, bf16=False, per_device_eval_batch_size=16, dataloader_num_workers=0,
                dataloader_pin_memory=False, output_dir=str(tmp), process_index=0, local_process_index=0, world_size=1,
                use_gpu=True)
    base.update(kw)
    return types.SimpleNamespace(**base)


def test_retriever_matches_reference_run(small_bert, golden_dir, tmp_path):
    from openmatch.arguments import ModelArguments
    from openmatch.modeling import DRModelForInference
    from openmatch.retriever import Retriever
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    margs = ModelArguments(model_name_or_path="unused", pooling="first", normalize=False)
    model = DRModelForInference(lm_q=small_bert, lm_p=small_bert, tied=True, pooling="first", normalize=False,
                                model_args=margs)
    args = _args(tmp_path)
    retriever = Retriever.build_all(model, Synth("d", z["ret_c_ids"], z["ret_c_mask"]), args)
    # reference-compatible pickle: (float32 [n, d], list[str]) at protocol 4
    with open(tmp_path / "embeddings.corpus.rank.0", "rb") as f:
        enc, ids = pickle.load(f)
    assert enc.dtype == np.float32 and enc.shape == (50, 128) and ids[:3] == ["d0", "d1", "d2"]
    result = retriever.retrieve(Synth("q", z["ret_q_ids"], z["ret_q_mask"]), topk=5)
    assert list(result.keys()) == ["q0", "q1", "q2"]
    for qi in range(3):
        want_ids, want_scores = list(z["ret_docids"][qi]), z["ret_scores"][qi]
        got = result[f"q{qi}"]
        assert len(got) == 5 and all(isinstance(v, float) for v in got.values())
        # bf16 encoder vs the reference's fp32: scores agree to 1e-2 relative, so near-ties may swap ranks
        overlap = [d for d in got if d in want_ids]
        assert len(overlap) >= 4 and list(got)[0] in want_ids[:2]
        for d in overlap:
            ref = float(want_scores[want_ids.index(d)])
            assert abs(got[d] - ref) <= 2e-2 * max(1.0, abs(ref))
        assert list(got.values()) == sorted(got.values(), reverse=True)

    # from_embeddings + retrieve reads the pickles back (the reference's two-step workflow)
    model2 = DRModelForInference(lm_q=small_bert, lm_p=small_bert, tied=True, pooling="first", model_args=margs)
    r2 = Retriever.from_embeddings(model2, args)
    assert r2.index.ntotal == 50
    again = r2.retrieve(Synth("q", z["ret_q_ids"], z["ret_q_mask"]), topk=5)
    assert again == result


def test_successive_retriever_equals_single_index(small_bert, golden_dir, tmp_path):
    from openmatch.arguments import ModelArguments
    from openmatch.modeling import DRModelForInference
    from openmatch.retriever import Retriever, SuccessiveRetriever
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    margs = ModelArguments(model_name_or_path="unused")
    args = _args(tmp_path)
    model = DRModelForInference(lm_q=small_bert, lm_p=small_bert, model_args=margs)
    Retriever.build_embeddings(model, Synth("d", z["ret_c_ids"], z["ret_c_mask"]), args)
    # split the corpus pickle into two partitions like scripts/split_embeddings.py would
    with open(tmp_path / "embeddings.corpus.rank.0", "rb") as f:
        enc, ids = pickle.load(f)
    for r, sl in enumerate((slice(0, 20), slice(20, 50))):
        with open(tmp_path / f"embeddings.corpus.rank.{r}", "wb") as f:
            pickle.dump((enc[sl], ids[sl]), f, protocol=4)
    single = Retriever.from_embeddings(DRModelForInference(lm_q=small_bert, lm_p=small_bert, model_args=margs), args)
    want = single.retrieve(Synth("q", z["ret_q_ids"], z["ret_q_mask"]), topk=7)
    succ = SuccessiveRetriever.from_embeddings(DRModelForInference(lm_q=small_bert, lm_p=small_bert, model_args=margs), args)
    got = succ.retrieve(Synth("q", z["ret_q_ids"], z["ret_q_mask"]), topk=7)
    assert {q: list(v) for q, v in got.items()} == {q: list(v) for q, v in want.items()}


def test_training_forward_matches_reference_loss(small_bert, golden_dir):
    from openmatch.arguments import DataArguments, ModelArguments
    from openmatch.modeling import DRModel
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    targs = types.SimpleNamespace(negatives_x_device=False, per_device_train_batch_size=3)
    model = DRModel(lm_q=small_bert, lm_p=small_bert, tied=True, pooling="first", model_args=ModelArguments("unused"),
                    data_args=DataArguments(train_n_passages=4), train_args=targs).cuda()
    model.train()
    for m in model.modules():  # dropout off so that the comparison with the reference's eval-mode run holds
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0

    def batch(ids, mask):
        return {"input_ids": torch.from_numpy(ids).cuda(), "attention_mask": torch.from_numpy(mask).cuda(),
                "token_type_ids": torch.zeros_like(torch.from_numpy(ids)).cuda()}

    out = model(query=batch(z["fwd_q_ids"], z["fwd_q_mask"]), passage=batch(z["fwd_p_ids"], z["fwd_p_mask"]))
    assert abs(out.loss.item() - float(z["fwd_loss"])) <= 2e-2 * max(1.0, abs(float(z["fwd_loss"])))
    np.testing.assert_allclose(out.scores.cpu().numpy(), z["fwd_scores"], rtol=2e-2, atol=0.3)  # bf16-rounded reps
    out.loss.backward()
    g = small_bert.encoder.layer[0].attention.self.query.weight.grad
    assert g is not None and torch.isfinite(g).all() and g.abs().sum() > 0
    small_bert.zero_grad(set_to_none=True)
    model.eval()
    small_bert.cpu()


def test_block_ingest_writes_index_rows_in_place(small_bert, tmp_path):
    # PretokenizedDataset.iter_batches -> pinned staging -> encoder writing straight into reserve_rows: same embeddings,
    # ids and row order as the per-example DataLoader path, and index.ntotal == len(doc_lookup)
    from openmatch.arguments import DataArguments, ModelArguments
    from openmatch.dataset import InferenceDataset
    from openmatch.modeling import DRModelForInference
    from openmatch.retriever import Retriever
    rng = np.random.default_rng(1)
    n, L = 75, 24
    ids = rng.integers(5, 500, (n, L)).astype(np.int32)
    for r in range(n):
        ids[r, rng.integers(4, L):] = 0
    np.save(tmp_path / "c.npy", ids)
    (tmp_path / "c.ids.txt").write_text("\n".join("p%d" % i for i in range(n)))
    dargs = DataArguments(corpus_path=str(tmp_path / "c.npy"), p_max_len=32)
    margs = ModelArguments(model_name_or_path="unused")
    model = DRModelForInference(lm_q=small_bert, lm_p=small_bert, model_args=margs)
    assert model.rep_dim() == 128
    out_a, out_b = tmp_path / "a", tmp_path / "b"
    ds = InferenceDataset.load(None, dargs, is_query=False, batch_size=16)
    fast = Retriever.build_all(model, ds, _args(out_a))
    assert fast.index.ntotal == n == len(fast.doc_lookup) and fast.doc_lookup[:2] == ["p0", "p1"]

    class PerExample(torch.utils.data.IterableDataset):  # hides iter_batches: forces the DataLoader + collator path
        def __iter__(self):
            return iter(InferenceDataset.load(None, dargs, is_query=False, batch_size=16))

    slow = Retriever.build_all(DRModelForInference(lm_q=small_bert, lm_p=small_bert, model_args=margs), PerExample(),
                               _args(out_b))
    assert slow.doc_lookup == fast.doc_lookup
    a, b = fast.index.master_rows().cpu(), slow.index.master_rows().cpu()
    assert torch.equal(a, b), "block ingest and per-example ingest disagree"
    with open(out_a / "embeddings.corpus.rank.0", "rb") as f:
        enc, names = pickle.load(f)
    assert enc.shape == (n, 128) and names == fast.doc_lookup and np.array_equal(enc, a.numpy())
    small_bert.cpu()
