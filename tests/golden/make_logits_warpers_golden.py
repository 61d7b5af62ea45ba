"""Generate tests/golden/logits_warpers_hf.pt: which tokens HuggingFace's TopKLogitsWarper / TopPLogitsWarper (an
INDEPENDENT implementation of top-k / nucleus filtering) leave drawable, on 64 random distributions over 16 candidates --
the subsets `sonar_b200/sampling.py` is held to in tests/test_oracle_decoder.py.

    python tests/golden/make_logits_warpers_golden.py"""

import os

import torch
from transformers.generation.logits_process import TopKLogitsWarper, TopPLogitsWarper

TOP_K = (1, 3, 8, 14)
TOP_P = (0.3, 0.6, 0.9, 0.99)


def main() -> None:
    g = torch.Generator().manual_seed(11)
    logits = torch.randn((64, 16), generator=g) * 2.5
    ids = torch.zeros((64, 1), dtype=torch.long)
    out = {"logits": logits}
    for k in TOP_K:
        out[f"top_k={k}"] = TopKLogitsWarper(top_k=k)(ids, logits.clone()) > float("-inf")
    for p in TOP_P:
        out[f"top_p={p}"] = TopPLogitsWarper(top_p=p)(ids, logits.clone()) > float("-inf")
    here = os.path.dirname(os.path.abspath(__file__))
    torch.save(out, os.path.join(here, "logits_warpers_hf.pt"))
    print("wrote logits_warpers_hf.pt", list(out))


if __name__ == "__main__":
    main()
