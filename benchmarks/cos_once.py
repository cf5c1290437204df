#!/usr/bin/env python
"""Development helper: two br_cosine_topk calls on the config-5 shard (for ncu captures of single launches)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from document_retrieval_b200.cosine import CosineIndex  # noqa: E402

dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(20241105 + 5)
docs = torch.empty(1_250_000, 768, device=dev, dtype=torch.bfloat16)
for a in range(0, docs.shape[0], 1 << 18):
    b = min(docs.shape[0], a + (1 << 18))
    docs[a:b] = torch.randn(b - a, 768, generator=g, device=dev).to(torch.bfloat16)
qs = torch.randn(10_000, 768, generator=g, device=dev).to(torch.bfloat16)
ix = CosineIndex(docs)
for _ in range(2):
    ids, sims = ix.topk(qs, 10)
torch.cuda.synchronize()
print("ok", ids.shape)
