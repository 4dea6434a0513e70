"""CPU: pins the oracle (oracle/*.py) against golden vectors produced by the REFERENCE's own code
(tests/golden/make_golden.py, executed against a checkout of thunlp/OpenMatch)."""
import os

import numpy as np
import torch

import oracle
from openmatch_b200.synthetic import recipe_state_dict
from oracle.encoder import EncoderSpec


def _load(golden_dir, name):
    z = np.load(os.path.join(golden_dir, name), allow_pickle=False)
    return z, recipe_state_dict(z["sd_recipe"])


def test_bert_encoder_matches_reference(golden_dir):
    z, sd = _load(golden_dir, "bert_small.npz")
    spec = EncoderSpec("bert", layers=2, hidden=128, heads=2, ffn=512, ln_eps=1e-12, pooling="first")
    hidden, reps = oracle.encode_reps(sd, spec, torch.from_numpy(z["input_ids"]), torch.from_numpy(z["attention_mask"]),
                                      torch.from_numpy(z["token_type_ids"]))
    m = z["attention_mask"].astype(bool)
    # padded query rows are never pooled; HF leaves implementation-defined values there
    np.testing.assert_allclose(hidden.numpy()[m], z["hidden"][m], rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(reps.numpy(), z["reps"], rtol=2e-4, atol=2e-5)


def test_t5_encoder_matches_reference(golden_dir):
    z, sd = _load(golden_dir, "t5_small.npz")
    spec = EncoderSpec("t5", layers=2, hidden=128, heads=2, ffn=512, ln_eps=1e-6, pooling="mean", normalize=True)
    hidden, reps = oracle.encode_reps(sd, spec, torch.from_numpy(z["input_ids"]), torch.from_numpy(z["attention_mask"]),
                                      head_weight=recipe_state_dict(z["head_recipe"])["linear.weight"])
    m = z["attention_mask"].astype(bool)
    np.testing.assert_allclose(hidden.numpy()[m], z["hidden"][m], rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(reps.numpy(), z["reps"], rtol=2e-4, atol=2e-6)


def test_t5_buckets_match_hf(golden_dir):
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    got = oracle.t5_relative_position_bucket(torch.from_numpy(z["t5_bucket_rel"]), 32, 128).numpy()
    np.testing.assert_array_equal(got, z["t5_bucket"])


def test_mean_pooling(golden_dir):
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    got = oracle.pool_head_normalize(torch.from_numpy(z["mp_hidden"]), torch.from_numpy(z["mp_mask"]), "mean", None,
                                     False)
    np.testing.assert_allclose(got.numpy(), z["mp_out"], rtol=1e-6, atol=1e-7)


def test_contrastive_loss_matches_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    for tag in ("a", "b"):
        loss, dx, dy, _ = oracle.contrastive_loss_fwd_bwd(z[f"loss_{tag}_x"], z[f"loss_{tag}_y"])
        assert abs(loss - float(z[f"loss_{tag}_loss"])) < 2e-6 * max(1.0, abs(loss))
        np.testing.assert_allclose(dx, z[f"loss_{tag}_dx"], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(dy, z[f"loss_{tag}_dy"], rtol=1e-4, atol=1e-6)
    loss, dx, dy, _ = oracle.contrastive_loss_fwd_bwd(z["loss_c_x"], z["loss_c_y"], z["loss_c_target"], "sum")
    assert abs(loss - float(z["loss_c_loss"])) < 2e-6 * max(1.0, abs(loss))
    np.testing.assert_allclose(dx, z["loss_c_dx"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(dy, z["loss_c_dy"], rtol=1e-4, atol=1e-6)


def test_training_forward_matches_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    _, sd = _load(golden_dir, "bert_small.npz")
    spec = EncoderSpec("bert", layers=2, hidden=128, heads=2, ffn=512, ln_eps=1e-12, pooling="first")
    _, q = oracle.encode_reps(sd, spec, torch.from_numpy(z["fwd_q_ids"]), torch.from_numpy(z["fwd_q_mask"]))
    _, p = oracle.encode_reps(sd, spec, torch.from_numpy(z["fwd_p_ids"]), torch.from_numpy(z["fwd_p_mask"]))
    np.testing.assert_allclose(q.numpy(), z["fwd_q_reps"], rtol=2e-4, atol=2e-5)
    loss, _, _, scores = oracle.contrastive_loss_fwd_bwd(q.numpy(), p.numpy())  # target = i * (12 // 3)
    np.testing.assert_allclose(scores, z["fwd_scores"], rtol=2e-4, atol=2e-4)
    assert abs(loss - float(z["fwd_loss"])) < 1e-4


def test_merge_results_matches_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    r1 = {"q1": {"d1": 3.0, "d2": 1.0, "d3": 2.0}, "q2": {"d9": 0.5}}
    r2 = {"q1": {"d2": 9.0, "d4": 2.5, "d5": 2.0}, "q3": {"d1": 1.0}}
    merged = oracle.merge_retrieval_results_by_score([r1, r2], topk=3)
    assert repr({k: list(v.items()) for k, v in merged.items()}) == str(z["merge_repr"])


def test_retriever_flow_matches_reference(golden_dir):
    """encode corpus + queries with the oracle encoder, flat-IP search, compare with what the reference's
    unmodified Retriever.build_all/retrieve produced over the same inputs."""
    z = np.load(os.path.join(golden_dir, "misc.npz"))
    _, sd = _load(golden_dir, "bert_small.npz")
    spec = EncoderSpec("bert", layers=2, hidden=128, heads=2, ffn=512, ln_eps=1e-12, pooling="first")
    _, c = oracle.encode_reps(sd, spec, torch.from_numpy(z["ret_c_ids"]), torch.from_numpy(z["ret_c_mask"]))
    _, q = oracle.encode_reps(sd, spec, torch.from_numpy(z["ret_q_ids"]), torch.from_numpy(z["ret_q_mask"]))
    D, I = oracle.flat_ip_search(q.numpy(), c.numpy(), 5)
    want_ids = z["ret_docids"]
    got_ids = np.array([[f"d{j}" for j in row] for row in I])
    assert (got_ids == want_ids).all()
    np.testing.assert_allclose(D, z["ret_scores"], rtol=2e-4, atol=2e-4)


def test_flat_index_semantics():
    rng = np.random.default_rng(0)
    x = rng.integers(-8, 9, size=(300, 16)).astype(np.float32)  # exact arithmetic, many ties
    q = rng.integers(-8, 9, size=(7, 16)).astype(np.float32)
    D, I = oracle.flat_ip_search(q, x, 10, block_rows=64)  # blocked == unblocked
    D2, I2 = oracle.flat_ip_search(q, x, 10, block_rows=1 << 20)
    assert (I == I2).all() and (D == D2).all()
    s = q @ x.T
    for r in range(7):
        order = sorted(range(300), key=lambda j: (-s[r, j], j))[:10]
        assert list(I[r]) == order
    # k > ntotal pads with -1 / lowest(float)
    D, I = oracle.flat_ip_search(q, x[:4], 6)
    assert (I[:, 4:] == -1).all() and (D[:, 4:] == np.float32(-3.4028234663852886e38)).all()
    idx = oracle.FlatIPIndex(16)
    idx.add(x[:100]); idx.add(x[100:])
    assert idx.ntotal == 300
    D3, I3 = idx.search(q, 10)
    assert (I3 == I2).all()
    idx.reset()
    assert idx.ntotal == 0


def test_t5_encoder_decoder_pooling_matches_the_reference(golden_dir):
    # the reference's default T5 mode (encoder_only=False, dense_retrieval_model.py:137-141): reps of DRModel.encode
    # (HF module path, CPU is fine here) against the reference's own run on the same weights
    import torch
    from transformers import T5Config, T5Model

    from openmatch_b200.arguments import ModelArguments
    from openmatch_b200.modeling import DRModelForInference
    z = np.load(os.path.join(golden_dir, "t5dec_small.npz"))
    cfg = T5Config(vocab_size=120, d_model=32, d_kv=8, d_ff=64, num_layers=2, num_decoder_layers=2, num_heads=4,
                   feed_forward_proj="relu", dropout_rate=0.0)
    lm = T5Model(cfg).eval()
    lm.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")})
    batch = {"input_ids": torch.from_numpy(z["ids"]), "attention_mask": torch.from_numpy(z["mask"])}
    for normalize in (False, True):
        model = DRModelForInference(lm_q=lm, lm_p=lm, tied=True, pooling="first", normalize=normalize,
                                    model_args=ModelArguments(model_name_or_path="unused", encoder_only=False))
        hidden, reps = model.encode_passage(batch)
        assert hidden.shape == (5, 1, 32)
        np.testing.assert_allclose(reps.numpy(), z["reps_norm%d" % int(normalize)], rtol=1e-5, atol=1e-6)
        out = torch.empty(5, 32)
        model.encode_into(batch, out)
        np.testing.assert_allclose(out.numpy(), z["reps_norm%d" % int(normalize)], rtol=1e-5, atol=1e-6)
