"""Generate tests/golden/{fid_base_full,contriever_base_full,untied_tiny}.npz by running the UNMODIFIED reference modules on
CPU (oracle/ref_shims.py) at the BASELINE shapes (VERDICT r1 "next round" item 1):

  fid_base_full         `src.fid.FiD`, T5-v1.1-base dims (12 + 12 layers, d 768, 12 heads, d_ff 2048, vocab 32128), ONE query x
                        n_context 40 x text_maxlength 384 tokens (ragged passage lengths), 32 target tokens: fp32 logits
                        (a strided column sample: every 32nd vocabulary entry + the 64 largest of every row), loss, a row
                        sample of the encoder states - and the SAME quantities with the reference's parameters cast to bf16
                        (how far the reference itself drifts at 16 bits = the accuracy budget of the GPU test).  The
                        samples keep the file under 1 MB; the 16-bit runs are stored as float16 (checked lossless).
  contriever_base_full  `src.retrievers.Contriever`, BERT-base dims, 64 passages x <= 192 tokens: fp32 embeddings + the
                        reference's own bf16 run.
  untied_tiny           `src.retrievers.UntiedDualEncoderRetriever` (src/retrievers.py:108-135) with
                        query_side_retriever_training on / off: embeddings of both towers, and for the loss sum(q . p) the
                        gradient norms of every parameter (the frozen passage tower has none under query-side training).

Weights / inputs are seeded (oracle/model_synth.py); the tests regenerate them and fill atlas_b200's modules with the same
values.  Runs in the build container only (`/root/reference` is not on the GPU box): python oracle/make_golden_fullsize.py
"""
import os
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import model_synth  # noqa: E402
import ref_shims  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(HERE), "tests", "golden")

T5_BASE = dict(model_synth.T5_CFG, vocab_size=32128, num_layers=12, num_decoder_layers=12)
BERT_BASE = dict(model_synth.CONTRIEVER_CFG, vocab_size=30522, num_hidden_layers=12)


def fid_base_inputs():
    return model_synth.fid_inputs(seed=77, B=1, n_ctx=40, L=384, T=32, vocab=32128)


def contriever_base_inputs(B=64):
    return model_synth.contriever_inputs(seed=55, B=B, L=192, vocab=30522)


def logit_sample(logits):
    """[B, T, V] -> (strided columns, top-64 indices per row from the fp32 run are chosen by the caller)."""
    return logits[..., ::32]


def fid_base():
    from transformers import T5Config
    from src.fid import FiD

    cfg = T5Config(**T5_BASE)
    cfg.tie_word_embeddings = False
    ids, mask, labels = fid_base_inputs()
    out = {}
    sd = sha = None
    top_idx = None
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16), ("fp16", torch.float16)):
        t0 = time.time()
        model = FiD(cfg).eval()
        if sd is None:
            sd, sha = model_synth.fill_state_dict(model.state_dict(), seed=303)
        model.load_state_dict(sd)
        model = model.to(dt)
        model.encoder.config.n_context = 40
        model.encoder.config.bsz = 1
        with torch.no_grad():
            res = model(input_ids=ids, attention_mask=mask, decoder_input_ids=model._shift_right(labels), labels=labels,
                        use_cache=False)
        logits = res[1].float()
        if top_idx is None:
            top_idx = logits.topk(64, dim=-1)[1]
            out["top_idx"] = top_idx.numpy().astype(np.int32)
        out[f"loss_{name}"] = np.array(float(res[0]))
        out[f"logits_strided_{name}"] = logit_sample(logits).numpy()
        out[f"logits_top_{name}"] = torch.gather(logits, -1, top_idx).numpy()
        out[f"argmax_{name}"] = logits.argmax(-1).numpy().astype(np.int32)
        enc = res.encoder_last_hidden_state.float()[0]
        out[f"enc_rows_{name}"] = enc[::122].numpy()                          # 126 of the 15 360 rows
        out[f"enc_absmax_{name}"] = np.array(float(enc.abs().max()))
        print(f"fid_base {name}: {time.time() - t0:.1f} s, loss {float(res[0]):.5f}", flush=True)
    for k in ("logits_strided", "logits_top", "enc_rows"):
        for h16 in ("bf16", "fp16"):
            d = np.abs(out[f"{k}_{h16}"] - out[k + "_fp32"])
            print(f"  reference {h16} vs fp32 {k}: max abs diff {d.max():.4e}, mean {d.mean():.4e}, "
                  f"scale {np.abs(out[k + '_fp32']).max():.3f}")
            half = out[f"{k}_{h16}"].astype(np.float16)
            assert np.array_equal(half.astype(np.float32), out[f"{k}_{h16}"]), f"{k}_{h16} is not float16-exact"
            out[f"{k}_{h16}"] = half
    np.savez_compressed(os.path.join(GOLDEN_DIR, "fid_base_full.npz"), weights_sha256=sha, **out)


def contriever_base():
    from transformers import BertConfig
    from src.retrievers import Contriever

    cfg = BertConfig(**BERT_BASE)
    ids, mask = contriever_base_inputs()
    out = {}
    sd = sha = None
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16), ("fp16", torch.float16)):
        t0 = time.time()
        model = Contriever(cfg).eval()
        if sd is None:
            sd, sha = model_synth.fill_state_dict(model.state_dict(), seed=404)
        model.load_state_dict(sd)
        model = model.to(dt)
        with torch.no_grad():
            out[f"emb_{name}"] = model(input_ids=ids, attention_mask=mask).float().numpy()
        print(f"contriever_base {name}: {time.time() - t0:.1f} s", flush=True)
    for h16 in ("bf16", "fp16"):
        d = np.abs(out[f"emb_{h16}"] - out["emb_fp32"])
        print(f"  reference {h16} vs fp32 emb: max abs diff {d.max():.4e} mean {d.mean():.4e} scale",
              float(np.abs(out["emb_fp32"]).max()))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "contriever_base_full.npz"), weights_sha256=sha, **out)


def untied():
    from transformers import BertConfig
    from src.retrievers import Contriever, UntiedDualEncoderRetriever

    cfg = BertConfig(**model_synth.CONTRIEVER_CFG)
    ids, mask = model_synth.contriever_inputs()
    pids, pmask = model_synth.contriever_inputs(seed=22, B=6, L=40)
    out = {}
    for mode in (True, False):
        q_enc, p_enc = Contriever(cfg), Contriever(cfg)
        sdq, _ = model_synth.fill_state_dict(q_enc.state_dict(), seed=111)
        sdp, _ = model_synth.fill_state_dict(p_enc.state_dict(), seed=112)
        q_enc.load_state_dict(sdq)
        p_enc.load_state_dict(sdp)
        for m in (q_enc, p_enc):
            m.config.hidden_dropout_prob = 0.0
            m.config.attention_probs_dropout_prob = 0.0
            for mod in m.modules():
                if isinstance(mod, torch.nn.Dropout):
                    mod.p = 0.0
        opt = SimpleNamespace(query_side_retriever_training=mode)
        r = UntiedDualEncoderRetriever(opt, q_enc, p_enc).train()
        q = r(input_ids=ids, attention_mask=mask, is_passages=False)
        p = r(input_ids=pids, attention_mask=pmask, is_passages=True)
        loss = (q * p).sum()
        loss.backward()
        tag = "qside" if mode else "both"
        out[f"q_emb_{tag}"] = q.detach().numpy()
        out[f"p_emb_{tag}"] = p.detach().numpy()
        out[f"loss_{tag}"] = np.array(float(loss))
        out[f"p_requires_grad_{tag}"] = np.array(bool(p.requires_grad))
        for tower, mod in (("query", r.query_contriever), ("passage", r.passage_contriever)):
            names, norms = [], []
            for n, prm in mod.named_parameters():
                names.append(n)
                norms.append(float(prm.grad.norm()) if prm.grad is not None else -1.0)
            out[f"grad_names_{tower}"] = np.array(names)
            out[f"grad_norms_{tower}_{tag}"] = np.array(norms, dtype=np.float64)
        out[f"passage_training_flag_after_{tag}"] = np.array(bool(r.passage_contriever.training))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "untied_tiny.npz"), **out)
    print("untied:", {k: (v.shape if hasattr(v, "shape") else v) for k, v in out.items() if "emb" in k or "loss" in k})


if __name__ == "__main__":
    ref_shims.install()
    torch.manual_seed(0)
    which = sys.argv[1:] or ["untied", "contriever", "fid"]
    if "untied" in which:
        untied()
    if "contriever" in which:
        contriever_base()
    if "fid" in which:
        fid_base()
