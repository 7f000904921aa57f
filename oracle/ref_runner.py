"""Drive the UNMODIFIED reference modules (`oracle/_ref/src`, staged by oracle/make_ref.py; `/root/reference/src` in the
build container) through the retrieve-then-read step that bench.py measures: reference `Contriever.forward`
(src/retrievers.py:22-60) -> reference `DistributedIndex.search_knn` (src/index.py:122-157: `matmul` + `topk`, the
reference's `--index_mode flat`) -> reference `FiD.forward` (src/fid.py:28-120 over src/modeling_t5.py) + loss.

TEST / BENCH INFRASTRUCTURE: used only by `bench.py --impl reference` (CPU, all host threads) and by the
`gpu_reference` leg (the same modules on cuda:0, eager PyTorch + cuBLAS: the comparator of north_star's ">= 10x").
Nothing here is on the product path; `atlas_b200/` never imports it.
"""
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

DIM = 768


def reference_root():
    """Where the reference sources are importable from: the copy oracle/make_ref.py staged inside the tree, or None."""
    staged = os.path.join(HERE, "_ref")
    if os.path.isfile(os.path.join(staged, "src", "index.py")):
        return staged
    return None


class LazyDocMap:
    """id -> synthetic passage dict without materialising millions of dicts (what `doc_map[x]` returns)."""

    def __init__(self, n, base=0, stride=1):
        self.n, self.base, self.stride = n, base, stride

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        g = self.base + self.stride * int(i)
        return {"id": str(g), "title": f"t{g}", "text": f"passage {g}"}


class ReferenceStep:
    """Reference Contriever-base + flat DistributedIndex + FiD-base (random init, the BASELINE configs[1]+[3] shapes)."""

    def __init__(self, rows, device="cpu", dtype=None, n_docs=40, text_len=384, seed=0, bank=None, embeddings=None, bank_seed=1234):
        import torch

        import ref_shims

        root = reference_root()
        if root is None:
            raise RuntimeError("reference sources not staged (run `python oracle/make_ref.py` in the build container)")
        ref_shims.install(root)
        from transformers import BertConfig, T5Config
        from src.fid import FiD
        from src.index import DistributedIndex
        from src.retrievers import Contriever

        self.torch = torch
        self.device = torch.device(device)
        self.dtype = dtype or (torch.float32 if self.device.type == "cpu" else torch.bfloat16)
        self.n_docs, self.text_len = n_docs, text_len
        torch.manual_seed(seed)
        self.retriever = Contriever(BertConfig()).eval().to(self.dtype).to(self.device)      # bert-base-uncased shapes
        cfg = T5Config(vocab_size=32128, d_model=768, d_kv=64, d_ff=2048, num_layers=12, num_decoder_layers=12,
                       num_heads=12, relative_attention_num_buckets=32, dropout_rate=0.1, layer_norm_epsilon=1e-6,
                       feed_forward_proj="gated-gelu", decoder_start_token_id=0, pad_token_id=0, eos_token_id=1,
                       is_encoder_decoder=True, use_cache=False)
        cfg.tie_word_embeddings = False                                                        # T5 v1.1 (lm-adapt)
        self.reader = FiD(cfg).eval().to(self.dtype).to(self.device)
        self.index = DistributedIndex()
        self.index.is_in_gpu = self.device.type == "cuda"
        self.index.doc_map = LazyDocMap(rows)
        if embeddings is not None:
            self.index.embeddings = embeddings.to(self.device)       # already [768, N] fp16
        elif bank is not None:
            # reference layout [768, N] fp16 (src/index.py:51); `bank` is the product arm's [N, 768] tensor
            self.index.embeddings = bank.t().contiguous()
        else:
            gen = torch.Generator().manual_seed(bank_seed)
            emb = torch.empty(DIM, rows, dtype=torch.float16)
            step = 1 << 16
            for s in range(0, rows, step):
                e = min(rows, s + step)
                emb[:, s:e] = (torch.randn(DIM, e - s, generator=gen) / (DIM ** 0.5)).half()
            self.index.embeddings = emb.to(self.device)
        self.pos = torch.arange(text_len, dtype=torch.long)

    def step(self, q_ids, q_mask, dec, labels, topk=40):
        """One retrieve-then-read step of `len(q_ids)` queries; returns (loss float, ids [B, k] list, phase seconds)."""
        torch = self.torch
        dev = self.device
        t0 = time.perf_counter()
        with torch.no_grad():
            q_emb = self.retriever(input_ids=q_ids.to(dev), attention_mask=q_mask.to(dev))
            if dev.type == "cuda":
                torch.cuda.synchronize()
            t1 = time.perf_counter()
            docs, _ = self.index.search_knn(q_emb, topk)
            gids = torch.tensor([[int(d["id"]) for d in row] for row in docs], dtype=torch.long)
            t2 = time.perf_counter()
            B = gids.shape[0]
            # reader tokens: the tokenizer stand-in bench.py uses for both arms (ids keyed by the retrieved passage id)
            reader_ids = ((gids[:, :, None] * 1315423911 + self.pos * 2654435761) % 32000 + 2).view(B, -1).to(dev)
            mask = torch.ones(B, self.n_docs * self.text_len, dtype=torch.bool, device=dev)
            self.reader.encoder.config.n_context = self.n_docs
            self.reader.encoder.config.bsz = B
            out = self.reader(input_ids=reader_ids, attention_mask=mask, decoder_input_ids=dec.to(dev),
                              labels=labels.to(dev), use_cache=False)
            loss = float(out[0])
            t3 = time.perf_counter()
        return loss, gids.tolist(), (t1 - t0, t2 - t1, t3 - t2)
