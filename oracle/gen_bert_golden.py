"""Generate tests/golden/bert_text.pt and tests/golden/bert_state_keys.json from HF transformers' own BertModel.

    python oracle/gen_bert_golden.py

Needs `transformers` only (not the reference checkout); the tests read the files and never import it.
  * BertModel(BertConfig()) in fp32 on the CPU, eval mode, with synthetic.bert_state_dict(0) loaded strict=True
    (which also pins the key layout; the listing goes to bert_state_keys.json, 199 keys, pooler included);
  * 6 transcripts of 1, 2, 63, 64, 65 and 512 seeded ids (synthetic.transcript_ids(..., seed=0));
  * per transcript the sum of hidden_states[-4:];
  * transcript 2's rows aligned to T = 100, 63, 20 frames with numpy.array_split blocks (T > n, T = n, T < n);
  * the transformers version.
To keep the file small, the sums and aligned rows are stored for every 12th of the 768 features (`columns`); the
tests compare those columns and take each row's scale from their own full rows.
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from feature_vs_text_compound_emotion_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
LENGTHS = (1, 2, 63, 64, 65, 512)
COLUMNS = torch.arange(0, 768, 12)


def main():
    import transformers
    from transformers import BertConfig, BertModel
    torch.set_grad_enabled(False)
    m = BertModel(BertConfig()).eval()
    sd = synthetic.bert_state_dict(0)
    m.load_state_dict(sd, strict=True)
    keys = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert list(keys) == list(sd), "synthetic key order differs from BertModel's"
    json.dump(keys, open(os.path.join(OUT, "bert_state_keys.json"), "w"), indent=0)
    ids = synthetic.transcript_ids(LENGTHS, seed=0)
    sums = []
    for x in ids:
        hs = m(x[None], output_hidden_states=True).hidden_states
        sums.append(sum(hs[-4:])[0])
    aligned = {}
    for T in (100, 63, 20):
        blocks = np.array_split(np.arange(T), len(ids[2]))
        idx = np.concatenate([np.full(len(b), i) for i, b in enumerate(blocks)])
        aligned[T] = sums[2][torch.from_numpy(idx)][:, COLUMNS].clone()
    torch.save({"transformers": transformers.__version__, "weights_seed": 0, "std": 0.02, "ids_seed": 0,
                "lengths": list(LENGTHS), "ids": ids, "columns": COLUMNS.clone(),
                "sums": [s[:, COLUMNS].clone() for s in sums], "aligned_index": 2, "aligned": aligned},
               os.path.join(OUT, "bert_text.pt"))
    print("bert", transformers.__version__, [tuple(t.shape) for t in sums], len(keys), "keys")


if __name__ == "__main__":
    main()
