"""Generates tests/golden/t5dec_small.npz by executing the REFERENCE's DRModelForInference in its default T5 mode
(encoder_only=False: full encoder-decoder, one zero decoder token, reps = decoder last_hidden_state[:, 0];
src/openmatch/modeling/dense_retrieval_model.py:137-141) on a randomly initialised tiny T5Model:

    python tests/golden/make_golden_t5dec.py <path to the OpenMatch checkout>
"""
import os
import sys

import numpy as np
import torch

REF_SRC = os.path.join(os.path.abspath(sys.argv[1]), "src") if len(sys.argv) == 2 else None
if REF_SRC is None or not os.path.isdir(os.path.join(REF_SRC, "openmatch")):
    sys.exit("usage: make_golden_t5dec.py <path to the OpenMatch checkout>")
sys.path.insert(0, REF_SRC)
from transformers import T5Config, T5Model  # noqa: E402

from openmatch.arguments import ModelArguments  # noqa: E402
from openmatch.modeling import DRModelForInference  # noqa: E402

torch.manual_seed(11)
cfg = T5Config(vocab_size=120, d_model=32, d_kv=8, d_ff=64, num_layers=2, num_decoder_layers=2, num_heads=4,
               feed_forward_proj="relu", dropout_rate=0.0)
lm = T5Model(cfg).eval()
g = torch.Generator().manual_seed(3)
ids = torch.randint(3, 120, (5, 12), generator=g)
mask = torch.ones_like(ids)
mask[1, 7:] = 0
mask[3, 4:] = 0
ids = ids * mask
out = {}
for normalize in (False, True):
    model = DRModelForInference(lm_q=lm, lm_p=lm, tied=True, pooling="first", normalize=normalize,
                                model_args=ModelArguments(model_name_or_path="unused", encoder_only=False))
    _, reps = model.encode_passage({"input_ids": ids, "attention_mask": mask})
    out["reps_norm%d" % int(normalize)] = reps.detach().numpy()
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "t5dec_small.npz"),
                    ids=ids.numpy(), mask=mask.numpy(), **out,
                    **{"sd." + k: v.numpy() for k, v in lm.state_dict().items()})
print("wrote t5dec_small.npz", {k: v.shape for k, v in out.items()})
