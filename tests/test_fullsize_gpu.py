"""Parity at the BASELINE shapes, on hardware (VERDICT r1 item 1): FiD-base (12 + 12 layers, n_context 40, text_maxlength 384,
32 target tokens) and Contriever-base (12 layers, 512 passages x <= 192 tokens) against goldens produced by the UNMODIFIED
reference on CPU (oracle/make_golden_fullsize.py: fp32 outputs plus the reference's own bf16 / fp16 runs), and against the
CPU oracle restatement (oracle/fid_cpu.py, itself pinned to the reference's goldens) where the golden holds a sample.

Accuracy budget: a 16-bit run here may sit as far from the reference's fp32 outputs as the reference's OWN 16-bit run does
(x 2 on the maximum, x 1.5 on the mean).  The measured numbers are printed (pytest -s) and recorded in DESIGN.md §5;
north_star's "1e-3 fp16" is below the reference's own fp16 drift at this depth (4.1e-2 on the logits), see DESIGN.md.
Also here: the untied dual encoder (src/retrievers.py:108-135) against the reference's embeddings and gradient norms."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import model_synth
from conftest import GOLDEN_DIR

pytestmark = pytest.mark.gpu

T5_BASE = {k: v for k, v in dict(model_synth.T5_CFG, vocab_size=32128, num_layers=12, num_decoder_layers=12).items()
           if k not in ("dropout_rate", "is_encoder_decoder", "use_cache")}
BERT_BASE = dict(model_synth.CONTRIEVER_CFG, vocab_size=30522, num_hidden_layers=12)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from atlas_b200._lib import lib

    lib()
    return torch.device("cuda:0")


def _drift(a, ref):
    d = np.abs(np.asarray(a, dtype=np.float64) - np.asarray(ref, dtype=np.float64))
    return float(d.max()), float(d.mean())


@pytest.mark.parametrize("dtype,key", [(torch.float16, "fp16"), (torch.bfloat16, "bf16")])
def test_fid_base_full_size_matches_reference(dev, dtype, key):
    from atlas_b200.fid import FiD, T5ConfigLite

    g = np.load(os.path.join(GOLDEN_DIR, "fid_base_full.npz"))
    model = FiD(T5ConfigLite(**T5_BASE))
    sd, sha = model_synth.fill_state_dict(model.state_dict(), 303)
    assert sha == str(g["weights_sha256"]), "seeded weights differ from the golden generator's"
    model.load_state_dict(sd)
    model = model.to(dtype).to(dev).eval()
    ids, mask, labels = model_synth.fid_inputs(seed=77, B=1, n_ctx=40, L=384, T=32, vocab=32128)
    model.encoder.config.n_context, model.encoder.config.bsz = 40, 1
    with torch.no_grad():
        out = model(input_ids=ids.to(dev), attention_mask=mask.to(dev), decoder_input_ids=model._shift_right(labels.to(dev)),
                    labels=labels.to(dev), use_cache=False)
    logits = out[1].float().cpu()
    assert logits.shape == (1, 32, 32128)
    top_idx = torch.from_numpy(g["top_idx"].astype(np.int64))
    got = {"logits_strided": logits[..., ::32].numpy(), "logits_top": torch.gather(logits, -1, top_idx).numpy(),
           "enc_rows": out.encoder_last_hidden_state.float().cpu()[0][::122].numpy()}
    # encoder states: the padding-compacted encoder (FiD._encode_rows) returns zeros at the 64-row tiles behind a passage's last
    # real token - positions whose values in the reference nothing reads (the cross-attention masks them); the kept rows are
    # compared, the dropped ones must be exactly 0
    from atlas_b200 import ops

    live = ops.key_block_live((1.0 - mask.view(40, 384).float().to(dev)) * -10000.0)
    kept = (ops.segment_tile_scan(live)[0].bool().cpu().repeat_interleave(64, dim=1).reshape(-1)[::122].numpy()
            if ops._ENC_PACKED and live is not None else np.ones(len(got["enc_rows"]), dtype=bool))
    assert kept.sum() >= len(kept) // 2 and float(np.abs(got["enc_rows"][~kept]).max(initial=0.0)) == 0.0
    report = {}
    for name, val in got.items():
        ref32 = g[f"{name}_fp32"]
        ref16 = g[f"{name}_{key}"]
        if name == "enc_rows":
            val, ref32, ref16 = val[kept], ref32[kept], ref16[kept]
        mx, mean = _drift(val, ref32)
        rmx, rmean = _drift(ref16, ref32)
        report[name] = (mx, mean, rmx, rmean)
        assert mx <= 2.0 * rmx + 1e-3 and mean <= 1.5 * rmean + 1e-4, (name, key, mx, mean, rmx, rmean)
    print(f"\nFiD-base full size [{key}] |ours - ref fp32| (max, mean) vs the reference's own {key} drift (max, mean): "
          + "; ".join(f"{n}: {a:.3e} {b:.3e} vs {c:.3e} {d:.3e}" for n, (a, b, c, d) in report.items()))
    assert abs(float(out[0]) - float(g["loss_fp32"])) <= 2.0 * abs(float(g[f"loss_{key}"]) - float(g["loss_fp32"])) + 2e-2
    # the greedy token of every target position agrees wherever the reference's top-2 logit gap exceeds its 16-bit drift
    top2 = np.sort(g["logits_top_fp32"], axis=-1)[..., -2:]
    safe = (top2[..., 1] - top2[..., 0]) > 4.0 * report["logits_top"][2]
    assert np.array_equal(logits.argmax(-1).numpy()[safe], g["argmax_fp32"][safe])


@pytest.mark.parametrize("dtype,key", [(torch.float16, "fp16"), (torch.bfloat16, "bf16")])
def test_contriever_base_full_size_matches_reference(dev, dtype, key):
    """512 passages x <= 192 tokens (one index-refresh embedder batch): the first 64 rows are the golden's passages
    (unmodified reference, fp32 + its own 16-bit runs); all 512 rows against the CPU oracle restatement on a row sample."""
    import fid_cpu
    from atlas_b200.retrievers import BertConfigLite, Contriever

    g = np.load(os.path.join(GOLDEN_DIR, "contriever_base_full.npz"))
    model = Contriever(BertConfigLite(**BERT_BASE))
    sd, sha = model_synth.fill_state_dict(model.state_dict(), 404)
    assert sha == str(g["weights_sha256"])
    model.load_state_dict(sd)
    ids64, mask64 = model_synth.contriever_inputs(seed=55, B=64, L=192, vocab=30522)
    ids_more, mask_more = model_synth.contriever_inputs(seed=56, B=448, L=192, vocab=30522)
    ids, mask = torch.cat([ids64, ids_more]), torch.cat([mask64, mask_more])
    model = model.to(dtype).to(dev).eval()
    with torch.no_grad():
        emb = model(input_ids=ids.to(dev), attention_mask=mask.to(dev)).float().cpu().numpy()
    assert emb.shape == (512, 768)
    ref32 = g["emb_fp32"]
    mx, mean = _drift(emb[:64], ref32)
    rmx, rmean = _drift(g[f"emb_{key}"], ref32)
    print(f"\nContriever-base [{key}] |ours - ref fp32| max {mx:.3e} mean {mean:.3e}; reference's own {key} drift "
          f"max {rmx:.3e} mean {rmean:.3e}")
    assert mx <= 2.0 * rmx + 1e-3 and mean <= 1.5 * rmean + 1e-4, (mx, mean, rmx, rmean)
    # rows 64.. against the CPU restatement (fp32) on a sample of 32 rows (batch rows are independent)
    sel = torch.arange(64, 512, 14)
    with torch.no_grad():
        want = fid_cpu.contriever_forward({k: v.float() for k, v in sd.items()}, BERT_BASE, ids[sel], mask[sel]).numpy()
    mx2, mean2 = _drift(emb[sel.numpy()], want)
    assert mx2 <= 2.0 * rmx + 1e-3 and mean2 <= 1.5 * rmean + 1e-4, (mx2, mean2)


@pytest.mark.parametrize("qside", [True, False])
def test_untied_dual_encoder_matches_reference(dev, qside):
    """`UntiedDualEncoderRetriever` (src/retrievers.py:108-135): separate query / passage towers; under
    `query_side_retriever_training` the passage tower embeds in eval mode under no_grad (frozen: no gradients) and its
    training flag is restored.  Embeddings and per-parameter gradient norms against the unmodified reference."""
    from atlas_b200.retrievers import BertConfigLite, Contriever, UntiedDualEncoderRetriever

    g = np.load(os.path.join(GOLDEN_DIR, "untied_tiny.npz"))
    tag = "qside" if qside else "both"
    q_enc = Contriever(BertConfigLite(**model_synth.CONTRIEVER_CFG))
    p_enc = Contriever(BertConfigLite(**model_synth.CONTRIEVER_CFG))
    sdq, _ = model_synth.fill_state_dict(q_enc.state_dict(), 111)
    sdp, _ = model_synth.fill_state_dict(p_enc.state_dict(), 112)
    q_enc.load_state_dict(sdq)
    p_enc.load_state_dict(sdp)
    r = UntiedDualEncoderRetriever(SimpleNamespace(query_side_retriever_training=qside), q_enc, p_enc).to(dev).train()
    ids, mask = model_synth.contriever_inputs()
    pids, pmask = model_synth.contriever_inputs(seed=22, B=6, L=40)
    q = r(input_ids=ids.to(dev), attention_mask=mask.to(dev), is_passages=False)
    p = r(input_ids=pids.to(dev), attention_mask=pmask.to(dev), is_passages=True)
    assert p.requires_grad == bool(g[f"p_requires_grad_{tag}"]) and q.requires_grad
    assert r.passage_contriever.training == bool(g[f"passage_training_flag_after_{tag}"])
    # fp32 master parameters train through bf16 activations (retrievers.py): the embedding budget is the bf16 one
    for got, name in ((q, "q_emb"), (p, "p_emb")):
        ref = g[f"{name}_{tag}"]
        err = np.abs(got.detach().float().cpu().numpy() - ref).max()
        assert err <= 3e-2 * max(1.0, np.abs(ref).max()), (name, err)
    loss = (q.float() * p.float()).sum()
    loss.backward()
    # sum of 6 x 768 signed products: the budget scales with sum |q . p| (the terms cancel), bf16 activations
    scale = float(np.abs(g[f"q_emb_{tag}"] * g[f"p_emb_{tag}"]).sum())
    assert abs(float(loss) - float(g[f"loss_{tag}"])) <= 1e-2 * scale, (float(loss), float(g[f"loss_{tag}"]), scale)
    for tower, mod in (("query", r.query_contriever), ("passage", r.passage_contriever)):
        names = [str(n) for n in g[f"grad_names_{tower}"]]
        norms = g[f"grad_norms_{tower}_{tag}"]
        params = dict(mod.named_parameters())
        for n, want in zip(names, norms):
            prm = params[n]
            if want < 0:
                assert prm.grad is None, (tower, n)          # frozen tower: the reference left .grad unset
            else:
                assert prm.grad is not None, (tower, n)
                got = float(prm.grad.float().norm())
                if n.endswith("attention.self.key.bias"):
                    # softmax is invariant to a per-query shift of the scores: this gradient is identically zero in exact
                    # arithmetic (the reference's 1e-7 is fp32 rounding noise, ours is bf16 rounding noise of the dS tile);
                    # it must stay noise-sized next to the query bias of the same layer
                    qb = float(params[n.replace("key.bias", "query.bias")].grad.float().norm())
                    assert got <= 0.05 * qb + 1e-4, (tower, n, got, qb)
                    continue
                assert abs(got - want) <= 0.08 * want + 1e-4, (tower, n, got, want)
