#!/usr/bin/env python
"""bench.py — the driver's measurement contract for atlas_b200 (see DESIGN.md §6).

Metric (BASELINE.json): end-to-end queries/sec of the retrieve-then-read step — Contriever query embedding,
exact top-40 search over the GPU-resident 768-d fp16 passage bank (BASELINE configs[1]: 4 Mi passages per GPU,
configs[2] at 8 GPUs = 32 Mi), FiD-base forward over the 40 retrieved passages (configs[3]: T5-v1.1-base, n_docs 40,
text_maxlength 384, 32 target tokens) — plus the MIPS scan against the HBM roofline.

  value         queries/s of the whole job, step inputs already resident in HBM, CUDA events, max over ranks
  e2e           the same step with HOST inputs: pinned token ids are copied H2D and the retrieved ids / scores and the
                loss are copied D2H inside the timed region
  roofline      the dominant kernel of the step (tcgen05 GEMM): FLOPs / CUDA-event time, against the measured bf16 peak
  mips          the retrieval kernel alone at its BASELINE batch (256 queries): queries/s, C-ABI e2e with host buffers,
                and the bank sweep against the measured HBM peak (`mips.roofline`)
  train         supplementary: FiD-base forward + BACKWARD step (the training path's kernels), reader tokens/s
  refresh       supplementary: index refresh in place (Contriever-base passage embedding into bank rows), passages/s
  cpu_baseline  the reference's CPU path (oracle/: torch-CPU restatements pinned to the reference's goldens) on this
                box's host cores, bounded sample
  gpu_reference the UNMODIFIED reference modules (oracle/_ref/src, staged by oracle/make_ref.py) on cuda:0 in bf16 eager
                PyTorch (`--index_mode flat`: matmul + topk; eager FiD / Contriever) on the same step: the comparator of
                north_star's ">= 10x" target, plus the fp32 matmul + topk stand-in for FAISS-GPU flat (faiss is absent)
  parity_check  before timing: the distributed search's ids / scores against torch `matmul(q.half(), E)` + `topk`
                (src/index.py:117-118) recomputed on every shard and merged (runs at every N)
`--impl reference` times the reference's own CPU path (the same unmodified modules, all host threads; one query per
step, real steps - nothing stitched or extrapolated at N = 1).  One process per GPU; weak scaling (per-GPU batch and
per-GPU bank shard fixed).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_LOCAL = 4 * 1024 * 1024   # passages per GPU  (BASELINE.json configs[1])
DIM = 768
NQ = 256                    # global query batch
TOPK = 40
CPU_SAMPLE_ROWS = 1 << 20   # bounded CPU sample: 1 Mi of the 4 Mi rows (scaled linearly, stated)
METRIC = "end-to-end queries/sec (retrieve top-40 + FiD-base fwd)"
N_DOCS, TEXT_LEN, TARGET_LEN, QUERY_TOKENS = 40, 384, 32, 20   # BASELINE configs[3] / finetune_qa defaults
FID_FLOPS_PER_QUERY = 3.29e12                                   # SURVEY.md §8(d)
PASSAGE_TOKENS = 256                                            # token-bank row width (passage part of the reader input)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8, help="queries per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=N_LOCAL, help="passages per GPU (default: the BASELINE config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-xl", action="store_true", help="skip the Atlas-xl training leg (BASELINE configs[4])")
    ap.add_argument("--ref-budget-s", type=float, default=150.0,
                    help="--impl reference: wall-clock budget of the timed CPU steps (each step = one query)")
    ap.add_argument("--profile-step", action="store_true",
                    help="run warm-up + the timed steps inside an NVTX range 'atlas_b200_timed' and exit (for ncu "
                         "--nvtx --nvtx-include 'atlas_b200_timed/'; no JSON line is printed)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 / "
                         "float64, at most 64 MB): the same arguments give the same inputs, so two builds can be "
                         "compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def peaks(kind="hbm"):
    """(peak, source).  hbm: GB/s (burst copy figure: the sweep is timed alone); tensor: dense bf16 TFLOP/s,
    the SUSTAINED figure (the GEMMs are timed inside a long step)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    key = "hbm_gbs" if kind == "hbm" else "bf16_tflops_sustained"
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        if key in d:
            return float(d[key]), f"measured (MEASURED_PEAKS.json {key})"
    return (6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)") if kind == "hbm" else \
        (1500.0, "fallback (B200_PROFILING.md dense bf16)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md):
    one `nvidia-smi -lms 20` process is started before the region and stopped after it."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.15)  # let the first samples land before the region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 6:
                self.samples.append(parts)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[j] for s in self.samples for j in range(4) if s[2 + j].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.samples)}


def make_bank(rows, device, seed):
    """Unit-scale Gaussian passages (norm ~1, Contriever-like), generated on the device in chunks."""
    import torch

    gen = torch.Generator(device=device).manual_seed(seed)
    bank = torch.empty(rows, DIM, dtype=torch.float16, device=device)
    step = 1 << 18
    for s in range(0, rows, step):
        e = min(rows, s + step)
        bank[s:e] = (torch.randn(e - s, DIM, device=device, generator=gen) / (DIM ** 0.5)).half()
    return bank


def make_queries():
    import torch

    return torch.randn(NQ, DIM, generator=torch.Generator().manual_seed(4321))


def _all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1: the CPU arm must still use every host core (VERDICT r1, weak item 7)."""
    import torch

    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def cpu_reference_leg(rows_total, budget_s=40.0, max_steps=1, warmup=0):
    """The reference's CPU path, REAL steps: the unmodified reference `Contriever` -> `DistributedIndex.search_knn`
    (matmul + topk over the whole `rows_total` x 768 fp16 bank, CPU-resident) -> `FiD` fp32 forward + loss
    (oracle/ref_runner.py over oracle/_ref/src), ONE query per step (the bounded sample), all host threads.  Falls back
    to the torch-CPU restatements (oracle/fid_cpu.py, kind "port") only when the reference sources are not staged."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    cores = _all_host_threads()
    import ref_runner

    if ref_runner.reference_root() is None:
        return _cpu_port_leg(rows_total, cores)
    # bank: a 256 Ki-column Gaussian block tiled to the full width (the arithmetic cost does not depend on the values);
    # capped by the host's free memory (stated) - the reference keeps the bank as ONE [768, N] fp16 tensor
    rows = rows_total
    try:
        import psutil

        free = psutil.virtual_memory().available
        while rows * DIM * 2 * 2.5 > free and rows > (1 << 20):
            rows //= 2
    except Exception:
        pass
    block = min(rows, 1 << 18)
    gen = torch.Generator().manual_seed(1234)
    blk = (torch.randn(DIM, block, generator=gen) / (DIM ** 0.5)).half()
    emb = torch.empty(DIM, rows, dtype=torch.float16)          # the reference layout, src/index.py:51
    for s in range(0, rows, block):
        e = min(rows, s + block)
        emb[:, s:e] = blk[:, :e - s]
    t_build = time.perf_counter()
    ref = ref_runner.ReferenceStep(rows, "cpu", torch.float32, N_DOCS, TEXT_LEN, embeddings=emb)
    del emb
    t_build = time.perf_counter() - t_build
    q_ids, q_mask, dec, labels = make_step_inputs(1, 0)
    for _ in range(warmup):
        ref.step(q_ids, q_mask, dec, labels, TOPK)
    times, phases = [], []
    t_start = time.perf_counter()
    while len(times) < max_steps and (not times or time.perf_counter() - t_start + times[-1] < budget_s):
        t0 = time.perf_counter()
        loss, _, ph = ref.step(q_ids, q_mask, dec, labels, TOPK)
        times.append(time.perf_counter() - t0)
        phases.append(ph)
    assert loss == loss, "non-finite reference loss"
    per_query = sum(times) / len(times)
    ph = [sum(p[i] for p in phases) / len(phases) for i in range(3)]
    scale_note = "" if rows == rows_total else f"; bank capped at {rows} of {rows_total} rows by host memory (search time NOT scaled)"
    return {"value": 1.0 / per_query, "unit": "queries/s", "cores": cores, "kind": "reference",
            "sample": f"{len(times)} timed step(s) of 1 query each (+{warmup} warm-up) through the UNMODIFIED reference "
                      f"(oracle/_ref/src: Contriever-base fp32 embed {ph[0]:.3f} s, DistributedIndex.search_knn over "
                      f"{rows} x 768 fp16 CPU bank {ph[1]:.3f} s, FiD-base fp32 forward n_docs {N_DOCS} x {TEXT_LEN} "
                      f"tokens {ph[2]:.3f} s); torch-CPU {torch.get_num_threads()} threads{scale_note}",
            "s_per_query": per_query, "steps": len(times), "model_build_s": t_build}


def _cpu_port_leg(rows_full, cores, batch=1):
    """Fallback when oracle/_ref is absent: the torch-CPU restatements (pinned to the reference's goldens)."""
    import torch

    import fid_cpu
    import ref_cpu_path

    rows = min(CPU_SAMPLE_ROWS, rows_full)
    gen = torch.Generator().manual_seed(1234)
    emb = (torch.randn(DIM, rows, generator=gen) / (DIM ** 0.5)).half()
    doc_map = ref_cpu_path.LazyDocMap(rows)
    bert = fid_cpu.bert_random_state(fid_cpu.BERT_BASE)
    t5 = fid_cpu.t5_random_state(fid_cpu.T5_BASE)
    q_ids, q_mask, dec, labels = make_step_inputs(batch, 0)
    with torch.no_grad():
        t0 = time.perf_counter()
        q = fid_cpu.contriever_forward(bert, fid_cpu.BERT_BASE, q_ids, q_mask)
        t_embed = (time.perf_counter() - t0) / batch
        t0 = time.perf_counter()
        ref_cpu_path.reference_search_cpu(emb, doc_map, q, TOPK)
        t_search = (time.perf_counter() - t0) * (rows_full / rows) / batch
        ids = torch.randint(2, 32000, (1, N_DOCS * TEXT_LEN))
        mask = torch.ones(1, N_DOCS * TEXT_LEN, dtype=torch.bool)
        t0 = time.perf_counter()
        fid_cpu.fid_forward(t5, fid_cpu.T5_BASE, ids, mask, dec[:1], labels[:1], n_context=N_DOCS)
        t_read = time.perf_counter() - t0
    per_query = t_embed + t_search + t_read
    return {"value": 1.0 / per_query, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"reference sources not staged: torch-CPU restatements (oracle/fid_cpu.py, oracle/ref_cpu_path.py), "
                      f"1 query: embed {t_embed:.3f} s + search {t_search:.3f} s ({rows} of {rows_full} rows, scaled) + "
                      f"FiD-base fp32 forward {t_read:.3f} s",
            "s_per_query": per_query, "steps": 1, "model_build_s": 0.0}


def make_step_inputs(batch, seed):
    """Synthetic NQ-shaped batch: queries of ~20 tokens padded to text_maxlength like the reference does
    (src/atlas.py:187-199), 32 target tokens."""
    import torch

    g = torch.Generator().manual_seed(777 + seed)
    q_ids = torch.zeros(batch, TEXT_LEN, dtype=torch.long)
    q_mask = torch.zeros(batch, TEXT_LEN, dtype=torch.long)
    q_ids[:, :QUERY_TOKENS] = torch.randint(1000, 30000, (batch, QUERY_TOKENS), generator=g)
    q_mask[:, :QUERY_TOKENS] = 1
    labels = torch.randint(2, 32000, (batch, TARGET_LEN), generator=g)
    dec = torch.cat([torch.zeros(batch, 1, dtype=torch.long), labels[:, :-1]], dim=1)
    return q_ids, q_mask, dec, labels


def workload_config(args):
    return {"workload": f"BASELINE configs[1]+[3]: per GPU a {args.rows}x768 fp16 passage bank (exact top-{TOPK}) and "
                        f"{args.batch} queries/step through Contriever-base query embedding -> search_knn -> FiD-base "
                        f"(T5-v1.1-base, n_docs {N_DOCS}, text_maxlength {TEXT_LEN}, {TARGET_LEN} target tokens) forward + loss",
            "bank_rows_per_gpu": args.rows, "bank_rows_total": args.rows * args.gpus,
            "queries_per_step": args.batch * args.gpus, "per_gpu_batch": args.batch, "topk": TOPK,
            "parallelism": f"dp{args.gpus}: bank sharded over {args.gpus} GPU(s) (queries all-gathered, one all-gather "
                           f"of per-shard top-k), reader data-parallel",
            "reader_tokens": f"synthetic device-resident token bank: {PASSAGE_TOKENS}-token rows keyed by global passage "
                             f"id (lengths U[{PASSAGE_TOKENS // 2}, {PASSAGE_TOKENS}]), spliced behind the query tokens "
                             "on the GPU (atlas_b200_splice_tokens); no tokenizer vocabulary offline",
            "padding": "every reader passage is padded to text_maxlength like src/atlas.py:261-270 pads (148 - 276 of 384 positions "
                       "real); the repo arm encodes each passage's 64-position tiles up to its last real token (same logits / loss, "
                       "DESIGN.md 3.10) and also reports the step with every padded position encoded (`padded_encoder`)",
            "weights": "random init (Contriever-base / T5-v1.1-base shapes), bf16 reader + retriever, fp16 bank",
            "l2": "bank (6.4 GB) and per-step activations (> 1 GB) exceed the 126 MB L2; no explicit flush"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the step on this box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    leg = cpu_reference_leg(args.rows * args.gpus, budget_s=args.ref_budget_s, max_steps=max(1, args.steps),
                            warmup=1 if args.warmup > 0 else 0)
    line = {
        "impl": "reference", "metric": METRIC, "value": leg["value"], "unit": "queries/s", "n_gpus": args.gpus,
        "steps": leg["steps"], "warmup": 1 if args.warmup > 0 else 0, "ms_per_step": leg["s_per_query"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args), reference_step="1 query per step (bounded sample of the "
                       f"{args.batch * args.gpus}-query step); steps capped by --ref-budget-s {args.ref_budget_s:g}"),
        "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": leg["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


class HashTokenizer:
    """Deterministic word-hash tokenizer with the call surface Atlas uses (no vocabulary files offline): the bench's
    stand-in for BertTokenizer / T5Tokenizer, used identically by the product arm and the gpu_reference leg."""

    def __init__(self, kind, vocab_size):
        import zlib

        self.kind, self.vocab_size, self._crc = kind, vocab_size, zlib.crc32
        self.pad_token_id, self.eos_token_id, self.cls_token_id, self.sep_token_id = 0, 1, 2, 3
        self.vocab = {f"tok{i}": i for i in range(vocab_size)}

    def _encode(self, text, special):
        ids = [self.eos_token_id if w == "</s>" else 10 + self._crc(w.lower().encode()) % (self.vocab_size - 10)
               for w in text.replace("</s>", " </s> ").split()]
        if special:
            ids = [self.cls_token_id] + ids + [self.sep_token_id] if self.kind == "bert" else ids + [self.eos_token_id]
        return ids

    def __call__(self, texts, padding=False, max_length=None, truncation=False, return_tensors=None,
                 add_special_tokens=True):
        import torch

        single = isinstance(texts, str)
        rows = [self._encode(t, add_special_tokens) for t in ([texts] if single else texts)]
        if truncation and max_length is not None:
            last = self.sep_token_id if self.kind == "bert" else self.eos_token_id
            rows = [r if len(r) <= max_length else (r[:max_length - 1] + [last] if add_special_tokens else r[:max_length])
                    for r in rows]
        if return_tensors is None:
            masks = [[1] * len(r) for r in rows]
            return {"input_ids": rows[0] if single else rows, "attention_mask": masks[0] if single else masks}
        width = max_length if padding == "max_length" else max((len(r) for r in rows), default=0)
        ids = torch.full((len(rows), width), self.pad_token_id, dtype=torch.long)
        mask = torch.zeros((len(rows), width), dtype=torch.long)
        for i, r in enumerate(rows):
            ids[i, :len(r)] = torch.tensor(r, dtype=torch.long)
            mask[i, :len(r)] = 1
        return {"input_ids": ids, "attention_mask": mask}

    def batch_encode_plus(self, texts, **kw):
        return self(texts, **kw)


class LazyDocs:
    """doc_map stand-in: local row -> synthetic passage dict, generated on demand (no 32 M python dicts)."""

    def __init__(self, n, base=0, stride=1):
        self.n, self.base, self.stride = n, base, stride

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        g = self.base + self.stride * int(i)
        return {"id": str(g), "title": f"t{g}", "text": f"passage {g}"}


def bench_opt(batch):
    """The option fields `Atlas` reads on the measured path (defaults of src/options.py at BASELINE configs[3])."""
    from types import SimpleNamespace

    return SimpleNamespace(
        retriever_format="{title} {text}", encoder_format="{query} title: {title} context: {text}",
        text_maxlength=TEXT_LEN, target_maxlength=TARGET_LEN, retriever_n_context=N_DOCS, n_context=N_DOCS,
        filtering_overretrieve_ratio=2, retrieve_with_rerank=False, n_to_rerank_with_retrieve_with_rerank=128,
        per_gpu_embedder_batch_size=512, per_gpu_batch_size=batch, decoder_prompt_format=None, decoder_format=None,
        use_file_passages=False, gold_score_mode="ppmean", use_gradient_checkpoint_retriever=False,
        use_gradient_checkpoint_reader=False, compute_crossattention_stats=False, temperature_gold=0.01,
        temperature_score=0.01, generation_max_length=TARGET_LEN, generation_min_length=1, generation_num_beams=1,
        generation_length_penalty=1.0, query_side_retriever_training=False, device_token_bank=True)


def make_token_bank(rows_total, dev):
    """Synthetic device-resident reader token bank: int32 [rows_total, PASSAGE_TOKENS] rows keyed by global passage id,
    lengths U[PASSAGE_TOKENS/2, PASSAGE_TOKENS] (replicated on every rank, atlas_b200/token_bank.py)."""
    import torch

    from atlas_b200.token_bank import DeviceTokenBank

    gen = torch.Generator(device=dev).manual_seed(4242)
    ids = torch.empty(rows_total, PASSAGE_TOKENS, dtype=torch.int32, device=dev)
    step = 1 << 20
    for s in range(0, rows_total, step):
        e = min(rows_total, s + step)
        ids[s:e] = torch.randint(10, 32000, (e - s, PASSAGE_TOKENS), device=dev, generator=gen, dtype=torch.int32)
    lens = torch.randint(PASSAGE_TOKENS // 2, PASSAGE_TOKENS + 1, (rows_total,), device=dev, generator=gen,
                         dtype=torch.int32)
    return DeviceTokenBank(ids, lens, eos_id=1, pad_id=0, parts=("{query} ", "title: {title} context: {text}"))


def make_query_strings(batch, seed):
    import random

    rnd = random.Random(9000 + seed)
    queries = [" ".join(f"q{rnd.randrange(50000)}" for _ in range(QUERY_TOKENS - 2)) for _ in range(batch)]
    targets = [" ".join(f"a{rnd.randrange(50000)}" for _ in range(TARGET_LEN - 1)) for _ in range(batch)]
    return queries, targets


def parity_check(index, q_local, dev, world, rank):
    """Before timing, at every N: the (distributed) search against the reference computation recomputed with torch on
    every shard - `torch.matmul(allqueries.half(), embeddings)` + `torch.topk` (src/index.py:117-118), per-shard lists
    merged with a second top-k (src/index.py:144-151).  Checks: returned scores == merged reference scores (<= 1 fp16
    ulp: cuBLAS and tcgen05 accumulate fp32 in different orders on Gaussian inputs), sorted descending, and every
    returned id's own score recomputed by its OWNER shard equals the returned score (<= 1 ulp).  Returns a dict."""
    import torch
    import torch.distributed as dist

    k = TOPK
    B = q_local.shape[0]
    scores, gids = index.search_device(q_local, k)
    q16 = q_local.half()
    if world > 1:
        allq = torch.empty(world * B, DIM, dtype=torch.float16, device=dev)
        dist.all_gather_into_tensor(allq, q16.contiguous())
    else:
        allq = q16
    S = torch.matmul(allq, index._bank.t())                                  # [W*B, N_local] fp16, the reference's product
    ref_s, _ = torch.topk(S, k, dim=1)
    if world > 1:
        ref_all = torch.empty(world, world * B, k, dtype=torch.float16, device=dev)
        dist.all_gather_into_tensor(ref_all, ref_s.contiguous())
        merged = torch.topk(ref_all.permute(1, 0, 2).reshape(world * B, world * k).float(), k, dim=1)[0]
        g_all = torch.empty(world, B, k, dtype=torch.int64, device=dev)
        s_all = torch.empty(world, B, k, dtype=torch.float16, device=dev)
        dist.all_gather_into_tensor(g_all, gids.contiguous())
        dist.all_gather_into_tensor(s_all, scores.contiguous())
    else:
        merged = ref_s.float()
        g_all, s_all = gids[None], scores[None]
    mine = merged[rank * B:(rank + 1) * B]
    got = scores.float()
    ulp = torch.maximum(mine.abs(), got.abs()).clamp_min(2.0 ** -14) * 2.0 ** -10
    bad_scores = int(((got - mine).abs() > ulp).sum())
    bad_sorted = int((got[:, 1:] > got[:, :-1]).sum())
    # owner check of the ids: rank r owns gid with gid % W == r at local row gid // W
    own = (g_all % world) == rank
    rows = torch.where(own, g_all // world, torch.zeros_like(g_all))
    qidx = (torch.arange(world, device=dev)[:, None, None] * B + torch.arange(B, device=dev)[None, :, None]).expand_as(g_all)
    mine_s = S[qidx, rows].float()
    ret_s = s_all.float()
    ulp2 = torch.maximum(mine_s.abs(), ret_s.abs()).clamp_min(2.0 ** -14) * 2.0 ** -10
    bad_ids = ((mine_s - ret_s).abs() > ulp2) & own
    dup = int(sum(len(set(r)) != k for r in gids.tolist()))
    fails = torch.tensor([bad_scores, bad_sorted, int(bad_ids.sum()), dup], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(fails)
    f = fails.tolist()
    del S
    return {"status": "ok" if sum(f) == 0 else "FAIL", "queries": world * B, "topk": k,
            "score_mismatches": f[0], "unsorted": f[1], "id_score_mismatches": f[2], "rows_with_duplicate_ids": f[3],
            "method": "scores vs torch.matmul(q.half(), E)+topk per shard merged by a second topk (src/index.py:117-151), "
                      "<= 1 fp16 ulp; every returned id re-scored by its owner shard"}


def gpu_reference_leg(args, bank, dev, steps=3, warmup=1):
    """The UNMODIFIED reference modules on cuda:0 (oracle/ref_runner.py over oracle/_ref/src): reference Contriever-base
    + `DistributedIndex` in `--index_mode flat` (matmul + topk, src/index.py:113-157) + eager FiD-base, bf16 parameters
    (`--precision bf16`, src/model_io.py:94-98), the same 8-query step on the same bank.  This is the comparator of
    north_star's ">= 10x the reference's GPU path"; FAISS is absent from the image, so next to it the fp32
    `matmul` + `topk` over an fp32 copy of the bank is timed as the stand-in for faiss GpuIndexFlatIP (labelled)."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_runner

    if ref_runner.reference_root() is None:
        return {"unavailable": "reference sources not staged (oracle/make_ref.py)"}
    B = args.batch
    ref = ref_runner.ReferenceStep(args.rows, dev, torch.bfloat16, N_DOCS, TEXT_LEN, bank=bank)
    inputs = make_step_inputs(B, 0)
    for _ in range(warmup):
        ref.step(*inputs, TOPK)
    torch.cuda.synchronize()
    times, phases = [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        loss, _, ph = ref.step(*inputs, TOPK)          # ends with float(loss): synchronised
        times.append(time.perf_counter() - t0)
        phases.append(ph)
    assert loss == loss, "non-finite reference loss"
    ms = 1e3 * sum(times) / len(times)
    ph = [1e3 * sum(p[i] for p in phases) / len(phases) for i in range(3)]
    out = {"value": B / (ms * 1e-3), "unit": "queries/s", "ms_per_step": ms, "steps": steps, "queries_per_step": B,
           "phases_ms": {"contriever": ph[0], "search_knn": ph[1], "fid_forward_loss": ph[2]},
           "what": "unmodified reference (oracle/_ref/src) on cuda:0, bf16 eager PyTorch + cuBLAS, --index_mode flat; "
                   "host token ids in, loss out (wall clock, synchronised)"}
    # search alone at the MIPS batch: reference flat index (fp16 matmul + topk) and the FAISS-flat stand-in (fp32)
    q = make_queries().to(dev)
    E = ref.index.embeddings

    def timed(fn, n=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    with torch.no_grad():
        ms_flat = timed(lambda: ref.index._compute_scores_and_indices(q, TOPK))
        out["search_256q_flat_fp16"] = {"ms": ms_flat, "queries_per_s": NQ / (ms_flat * 1e-3),
                                        "what": "reference DistributedIndex._compute_scores_and_indices, 256 queries"}
        try:
            chunk = 1 << 20
            E32 = E[:, :chunk].float()

            def faiss_standin():
                best = None
                for _ in range(args.rows // chunk):        # same fp32 block re-used: arithmetic and traffic of a full sweep
                    s_, i_ = torch.topk(torch.matmul(q, E32), TOPK, dim=1)
                    best = s_ if best is None else torch.maximum(best, s_)
                return best

            ms32 = timed(faiss_standin, 3)
            out["search_256q_fp32_standin"] = {"ms": ms32, "queries_per_s": NQ / (ms32 * 1e-3),
                                               "what": "STAND-IN for faiss GpuIndexFlatIP (faiss absent): fp32 matmul + "
                                                       "topk over 1 Mi-column fp32 blocks, full-bank arithmetic"}
        except Exception as e:
            out["search_256q_fp32_standin"] = {"error": repr(e)[:200]}
    del ref
    torch.cuda.empty_cache()
    return out


DUMP_LOGITS_BYTES = 48 << 20     # --dump-outputs: the logits in full up to this size, else a fixed sample of their rows
DUMP_ENC_ROWS = 2048             # ... and a fixed sample of the encoder-state rows (6 MB), 64 MB in all


def _sample_rows(t, n, seed):
    """`t` [rows, width] -> (t[rows], rows): a fixed seeded sample of `n` rows in ascending order."""
    import torch

    rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return t[rows.to(t.device)], rows


def dump_outputs(out_dir, out, gids, scores):
    """--dump-outputs: what one timed step returned, as out_dir/<name>.npy - the FiD loss and logits, a row sample of
    the encoder states, and the retrieved global passage ids (float64, exact) with their scores.  16-bit values are
    widened to float32."""
    import numpy as np

    loss, logits, enc = out
    arrays = {"loss": loss.float(), "passage_ids": gids.double(), "passage_scores": scores.float()}
    flat = logits.reshape(-1, logits.shape[-1])
    keep = DUMP_LOGITS_BYTES // (flat.shape[1] * 4)
    if flat.shape[0] <= keep:
        arrays["logits"] = logits.float()
    else:                           # the *_rows arrays index the rows of the tensor flattened to [-1, last dimension]
        sample, rows = _sample_rows(flat, keep, 1)
        arrays["logits_sample"], arrays["logits_sample_rows"] = sample.float(), rows.double()
    enc = enc.reshape(-1, enc.shape[-1])
    sample, rows = _sample_rows(enc, min(DUMP_ENC_ROWS, enc.shape[0]), 2)
    arrays["encoder_states_sample"], arrays["encoder_states_sample_rows"] = sample.float(), rows.double()
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def run_ours(args):
    import ctypes

    import torch
    import torch.distributed as dist

    from atlas_b200 import ops
    from atlas_b200._lib import lib
    from atlas_b200.atlas import Atlas
    from atlas_b200.fid import FiD, T5ConfigLite
    from atlas_b200.index import DistributedIndex
    from atlas_b200.retrievers import BertConfigLite, Contriever, DualEncoderRetriever

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl")
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    L = lib()
    B = args.batch
    index = DistributedIndex()
    index._bank = make_bank(args.rows, dev, 1234 + rank)
    index.doc_map = LazyDocs(args.rows, rank, world)
    index._id_base, index._id_stride = rank, world
    index.max_queries_per_rank = B          # every rank searches B queries per step: no size exchange, no host sync

    class _SyntheticStore:  # passage text by global id, generated on the fly (no 32M python dicts)
        def lookup(self, owners_locals):
            return [{"id": str(l * world + r), "title": f"t{l * world + r}", "text": f"passage {l * world + r}"}
                    for r, l in owners_locals]

        def close(self):
            pass

    index._store = _SyntheticStore()
    torch.manual_seed(0)          # identical weights on every rank
    contriever = Contriever(BertConfigLite()).to(torch.bfloat16).to(dev).eval()
    reader = FiD(T5ConfigLite()).to(torch.bfloat16).to(dev).eval()
    reader.encoder.config.n_context, reader.encoder.config.bsz = N_DOCS, B
    opt = bench_opt(B)
    atlas = Atlas(opt, reader, DualEncoderRetriever(opt, contriever), HashTokenizer("t5", 32128),
                  HashTokenizer("bert", 30522)).eval()
    bank_tokens = make_token_bank(args.rows * world, dev)
    atlas.set_token_bank(bank_tokens)

    def barrier_sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident step inputs (the `value` loop) -------------------------------------------
    queries, targets = make_query_strings(B, rank)
    q_enc = atlas.retriever_tokenize(queries)                                   # [B, 384] ids / mask on the device
    labels, dec = atlas.reader_tokenize(queries, targets, None)
    rq_ids, rq_lens = bank_tokens.query_tokens(atlas.reader_tokenizer, queries, dev)
    status_acc = torch.zeros((), dtype=torch.int64, device=dev)

    def step_device():
        """One retrieve-then-read step of this rank's B queries, inputs resident, NO host synchronisation:
        Contriever -> sharded scan + (at N > 1) 2 all-gathers + merge -> token-bank splice -> FiD forward + loss."""
        with torch.no_grad():
            q_emb = contriever(input_ids=q_enc["input_ids"], attention_mask=q_enc["attention_mask"])
            scores, gids, status = index.search_device(q_emb, TOPK, return_status=True)
            status_acc.copy_(torch.maximum(status_acc, status))
            tok = bank_tokens.splice(gids, TEXT_LEN, rq_ids, rq_lens)
            out = reader(input_ids=tok["input_ids"].view(B, -1), attention_mask=tok["attention_mask"].view(B, -1),
                         decoder_input_ids=dec, labels=labels)
        return out, gids, scores

    def step_api():
        """The same step through the module surface train.py / evaluate.py call, HOST inputs and outputs: query strings
        -> Atlas.retriever_tokenize / reader_tokenize (host tokenisation + H2D) -> Atlas.retrieve (query embedding,
        DistributedIndex.search_knn: ids + scores D2H, passage dicts from the store) -> Atlas.reader_passage_tokens
        (device token bank) -> Atlas.compute_reader_loss_and_logits (loss D2H)."""
        enc = atlas.retriever_tokenize(queries)
        lab, dec_ids = atlas.reader_tokenize(queries, targets, None)
        passages, scores = atlas.retrieve(index, TOPK, queries, enc["input_ids"], enc["attention_mask"])
        tok = atlas.reader_passage_tokens(queries, passages)
        loss, _ = atlas.compute_reader_loss_and_logits(tok, dec_ids, lab)
        return loss, passages, scores

    # ---------------- parity of the (distributed) search against the reference computation, before timing ----------
    with torch.no_grad():
        q_par = contriever(input_ids=q_enc["input_ids"], attention_mask=q_enc["attention_mask"])
        parity = parity_check(index, q_par, dev, world, rank)
    assert parity["status"] == "ok", f"search parity check failed: {parity}"

    # the interpreter's cyclic GC is kept out of the timed regions of BOTH arms of this process (a generation-2 pass over the
    # millions of objects transformers / torch import costs 10 - 30 ms, i.e. a whole step, whenever it happens to trigger)
    import gc

    gc.collect()
    gc.freeze()
    # ---------------- value: device-resident inputs -----------------------------------------
    n_warm = max(args.warmup, 3 if world == 1 else 10)     # NCCL connections / graph capture settle before timing
    for _ in range(n_warm):
        step_device()
    launches0 = L.atlas_b200_launch_count()
    barrier_sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        torch.cuda.nvtx.range_push("atlas_b200_timed")
        e0.record()
        for _ in range(args.steps):
            last = None             # drop the previous step's logits / encoder states before the next step allocates
            last = step_device()
        e1.record()
        barrier_sync()
        torch.cuda.nvtx.range_pop()
    loss = last[0][0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    del last
    if args.profile_step:
        if world > 1:
            dist.destroy_process_group()
        return
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    launches_eager = None
    ms_per_step = total_ms / args.steps
    value = B * world / (ms_per_step * 1e-3)
    assert bool(torch.isfinite(loss.float())), "non-finite loss in the benchmark step"
    assert int(status_acc.item()) == 0, "the fast search path overflowed during the timed steps (exhaustive path needed)"

    # ---------------- e2e: host inputs / host results through the Atlas module surface --------------------------
    for _ in range(3):
        step_api()
    barrier_sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loss_host, passages, _ = step_api()
    barrier_sync()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    assert loss_host == loss_host and len(passages) == B and len(passages[0]) == TOPK
    # where the e2e step spends its time (untimed diagnostic pass: a device synchronisation after every phase)
    phase_samples = {}
    for _ in range(7):
        marks = [time.perf_counter()]

        def mark(name):
            torch.cuda.synchronize()
            marks.append(time.perf_counter())
            phase_samples.setdefault(name, []).append((marks[-1] - marks[-2]) * 1e3)

        enc = atlas.retriever_tokenize(queries)
        lab, dec_ids = atlas.reader_tokenize(queries, targets, None)
        mark("tokenize_queries_and_targets_h2d")
        psg, _ = atlas.retrieve(index, TOPK, queries, enc["input_ids"], enc["attention_mask"])
        mark("retrieve_contriever_search_knn_passage_dicts")
        tok = atlas.reader_passage_tokens(queries, psg)
        mark("reader_passage_tokens_device_bank")
        atlas.compute_reader_loss_and_logits(tok, dec_ids, lab)
        mark("reader_forward_loss_item")
    e2e_phases = {k: sorted(v)[len(v) // 2] for k, v in phase_samples.items()}      # median of 7 passes
    h2d = (sum(t.numel() * t.element_size() for t in q_enc.values()) + labels.numel() * 8 + dec.numel() * 8
           + rq_ids.numel() * 8 + rq_lens.numel() * 4 + B * N_DOCS * 8) * world
    d2h = (4 + B * TOPK * (8 + 4) + 8) * world

    # ---------------- the same device-resident step with the encoder on every padded position (for the record) ---------
    from atlas_b200 import ops as _ops

    padded_encoder = None
    if _ops._ENC_PACKED:
        _ops._ENC_PACKED = False
        try:
            for _ in range(3):
                step_device()
            barrier_sync()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            for _ in range(args.steps):
                step_device()
            p1.record()
            barrier_sync()
            pms = max_over_ranks(p0.elapsed_time(p1)) / args.steps
            padded_encoder = {"value": B * world / (pms * 1e-3), "unit": "queries/s", "ms_per_step": pms,
                              "what": "ATLAS_B200_ENC_PACKED=0: embedding, projections and norms of the FiD encoder on all "
                                      f"{N_DOCS} x {TEXT_LEN} padded positions per query like the reference (all-padding key "
                                      "blocks still skipped by the attention kernels)"}
        finally:
            _ops._ENC_PACKED = True
        step_device()

    # ---------------- per-kernel time of the step (eager launches bracketed with CUDA events in the library) -------
    reader.cuda_graphs = False
    prof = {}
    gemm_launches = []
    for kind, name in ((2, "gemm"), (3, "attention")):
        step_device()
        torch.cuda.synchronize()
        l0 = L.atlas_b200_launch_count()
        L.atlas_b200_profile_enable(kind)
        step_device()
        torch.cuda.synchronize()
        work = L.atlas_b200_profile_work()
        if name == "gemm":      # per-launch records: the encoder-sized launches are a different instantiation of the kernel
            cap = 1024
            lms, lwk = (ctypes.c_double * cap)(), (ctypes.c_double * cap)()
            ln = L.atlas_b200_profile_launches(lms, lwk, cap)
            gemm_launches = [(lms[i], lwk[i]) for i in range(ln)]
        kms, kn = ctypes.c_double(0), ctypes.c_int32(0)
        L.atlas_b200_profile_collect(ctypes.byref(kms), ctypes.byref(kn))
        L.atlas_b200_profile_enable(0)
        prof[name] = (kms.value, kn.value, work)
        launches_eager = L.atlas_b200_launch_count() - l0
    reader.cuda_graphs = True

    # ---------------- the retrieval kernel alone at its BASELINE batch (256 queries) -------------
    index.max_queries_per_rank = NQ // world
    mips = mips_leg(args, index, dev, world, rank, L, barrier_sync, max_over_ranks)
    index.max_queries_per_rank = B

    # ---------------- greedy generation with the KV-cached decode path (supplementary) -----------------------------
    try:
        generate = generate_leg(args, atlas, bank_tokens, index, q_enc, rq_ids, rq_lens, dev, world, L, barrier_sync,
                                max_over_ranks)
    except Exception as e:
        generate = {"error": repr(e)[:300]}

    # ---------------- the reader's TRAINING step (forward + backward kernels), BASELINE configs[3] shapes -------------
    try:
        train = train_leg(args, reader, dev, world, L, barrier_sync, max_over_ranks)
    except Exception as e:   # the headline line must survive a failure of this supplementary leg
        train = {"error": repr(e)[:300]}

    # ---------------- BASELINE configs[4]: Atlas-xl retrieve + forward + backward + distillation loss ----------------
    if args.no_xl:
        xl = {"skipped": "--no-xl"}
    else:
        try:
            xl = xl_train_leg(args, atlas, index, bank_tokens, dev, world, rank, L, barrier_sync, max_over_ranks)
        except Exception as e:
            xl = {"error": repr(e)[:300]}
        index.max_queries_per_rank = B

    # ---------------- index refresh in place (BASELINE configs[2]: re-embed the local shard), one embedder batch -------
    try:
        refresh = refresh_leg(args, contriever, index, dev, world, L, barrier_sync, max_over_ranks)
    except Exception as e:
        refresh = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peak, peak_src = peaks("tensor")
    gemm_traffic, gemm_traffic_note = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_gemm_traffic.json")
    if os.path.exists(tpath):     # dram bytes of ONE representative launch from the committed `ncu --set full` capture
        with open(tpath) as f:
            tj = json.load(f)
        gemm_traffic = tj.get("dram_bytes_per_launch")
        gemm_traffic_note = f"{tj.get('launch')}: algorithmic {tj.get('algorithmic_bytes_per_launch')} B; {tj.get('source')}"
    g_ms, g_n, g_flops = prof["gemm"]
    a_ms, a_n, a_flops = prof["attention"]
    all_gemm = {"ms_per_step": g_ms, "launches_per_step": g_n, "flops_per_step": g_flops,
                "achieved_tflops": g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0}
    all_gemm["frac"] = all_gemm["achieved_tflops"] / peak if peak else None
    # the dominant kernel: gemm_kernel<bf16, 256, pair> - the launches of the encoder blocks and the cross K | V projections
    # (>= 20 GFLOP each; the decoder's 256-row launches run the 128-wide single-CTA instantiation and are latency-bound)
    big = [(m, w) for m, w in gemm_launches if w >= 2e10]
    if big:
        g_ms, g_n, g_flops = sum(m for m, _ in big), len(big), sum(w for _, w in big)
    achieved = g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    a_tflops = a_flops / (a_ms * 1e-3) / 1e12 if a_ms > 0 else None
    line = {
        "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": n_warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                     "frac": achieved / peak if peak else None, "traffic": gemm_traffic, "traffic_note": gemm_traffic_note,
                     "peak_source": peak_src,
                     "kernel": "gemm_kernel<bf16, 256, pair> (tcgen05 2-CTA tiles: the linear layers of the FiD-base encoder blocks "
                               "and the cross K | V projections, fused epilogues; launches >= 20 GFLOP, rows counted as computed)",
                     "all_gemm_launches": all_gemm,
                     "kernel_ms_per_step": g_ms, "kernel_launches_per_step": g_n, "algorithmic_flops_per_step": g_flops,
                     "kernel_share_of_step": g_ms / ms_per_step if ms_per_step else None,
                     "attention_kernel": {"ms_per_step": a_ms, "launches_per_step": a_n, "achieved_tflops": a_tflops,
                                          "work_note": "dense-equivalent FLOPs (4 B H Lq Lk 64 of the padded shapes): all-padding "
                                                       "key blocks / query tiles are skipped, the tensor-pipe rate is lower",
                                          "frac_of_tensor_peak": a_tflops / peak if (a_tflops and peak) else None,
                                          "share_of_step": a_ms / ms_per_step if ms_per_step else None},
                     "mips_scan": mips.get("roofline"),
                     "model_flops_utilisation": FID_FLOPS_PER_QUERY * B / (ms_per_step * 1e-3) / 1e12 / peak,
                     "model_flops_utilisation_note": "dense-model FLOPs (every padded position counted) over the step time; "
                                                     "`achieved` / `frac` above count only the rows the GEMMs computed"},
        "encoder": "padding-compacted: each passage keeps its 64-row tiles up to its last real token "
                   "(FiD._encode_rows, DESIGN.md 3.10); `padded_encoder` = the same step with ATLAS_B200_ENC_PACKED=0"
                   if _ops._ENC_PACKED else "every padded position (ATLAS_B200_ENC_PACKED=0)",
        "padded_encoder": padded_encoder,
        "e2e": {"value": B * world / (e2e_ms * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
                "phases_ms_synchronised": {k: round(v, 3) for k, v in e2e_phases.items()},
                "call": "query strings -> Atlas.retriever_tokenize / reader_tokenize -> Atlas.retrieve (Contriever.forward + "
                        "DistributedIndex.search_knn incl. passage dicts) -> Atlas.reader_passage_tokens (device token "
                        "bank) -> Atlas.compute_reader_loss_and_logits (loss.item())"},
        "parity_check": parity,
        "gpu_launches": int(launches_eager) * args.steps if launches_eager else 0,
        "gpu_launches_note": "kernels per step counted on an eager step; the timed steps replay the reader's launches "
                             "from a CUDA graph",
        "clocks": clocks.summary(),
        "mips": mips,
        "generate": generate,
        "train": train,
        "train_xl": xl,
        "refresh": refresh,
    }
    if not args.no_gpu_reference and world == 1:
        try:
            gref = gpu_reference_leg(args, index._bank, dev)
            if "value" in gref:
                gref["ours_over_reference_e2e"] = line["e2e"]["value"] / gref["value"]
                m = gref.get("search_256q_flat_fp16")
                if m and mips.get("value"):
                    m["ours_over_reference"] = mips["value"] / m["queries_per_s"]
            line["gpu_reference"] = gref
        except Exception as e:
            line["gpu_reference"] = {"error": repr(e)[:300]}
    if not args.no_cpu_baseline and world == 1:
        del index._bank
        torch.cuda.empty_cache()
        leg = cpu_reference_leg(args.rows, budget_s=30.0, max_steps=1, warmup=0)
        line["cpu_baseline"] = {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")}
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def generate_leg(args, atlas, bank_tokens, index, q_enc, rq_ids, rq_lens, dev, world, L, barrier_sync, max_over_ranks,
                 reps=3):
    """Greedy generation (`Atlas.generate` path, src/atlas.py:592-619) with the KV-cached decode (csrc/decode.cu): per GPU
    `batch` queries x 40 retrieved passages, `TARGET_LEN` tokens (min_length = max_length so every run decodes the same
    number of steps).  Reports generated tokens/s over all ranks, the time of one decode step (graph replay) and the
    cross-attention decode kernel against the HBM roofline: bytes = batch * 15 360 keys * (K + V) 2 * 768 * 2 B * 12 layers
    per step, every byte read once."""
    import ctypes

    import torch

    B = args.batch
    reader = atlas.reader
    with torch.no_grad():
        q_emb = atlas.retriever(q_enc["input_ids"], q_enc["attention_mask"], is_passages=False)
        _, gids, _ = index.search_device(q_emb, TOPK, return_status=True)
        tok = bank_tokens.splice(gids, TEXT_LEN, rq_ids, rq_lens)
    ids, mask = tok["input_ids"].view(B, -1), tok["attention_mask"].view(B, -1)
    reader.encoder.config.n_context, reader.encoder.config.bsz = N_DOCS, B

    def run(n_tokens):
        return reader.generate(input_ids=ids, attention_mask=mask, max_length=n_tokens, min_length=n_tokens)

    def timed(n_tokens):
        run(n_tokens)
        barrier_sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            seq = run(n_tokens)
        e1.record()
        barrier_sync()
        return max_over_ranks(e0.elapsed_time(e1)) / reps, seq

    ms_full, seq = timed(TARGET_LEN)
    ms_short, _ = timed(2)
    assert seq.shape == (B, TARGET_LEN)
    step_ms = (ms_full - ms_short) / (TARGET_LEN - 2)
    # the cross-attention decode kernel alone (eager steps bracketed with CUDA events inside the library)
    reader.cuda_graphs = False
    try:
        run(4)
        torch.cuda.synchronize()
        L.atlas_b200_profile_enable(5)
        run(4)
        torch.cuda.synchronize()
        kms, kn = ctypes.c_double(0), ctypes.c_int32(0)
        L.atlas_b200_profile_collect(ctypes.byref(kms), ctypes.byref(kn))
        L.atlas_b200_profile_enable(0)
    finally:
        reader.cuda_graphs = True
    peak, peak_src = peaks("hbm")
    c = reader.config
    from atlas_b200 import ops as _ops

    # the decode steps skip 64-key tiles of padding only (exact zeros of the softmax): bytes actually read = the live tiles'
    live = _ops.key_block_live((1.0 - mask.float()) * -1e9)
    live_frac = float(live.float().mean()) if live is not None else 1.0
    bytes_dense = B * N_DOCS * TEXT_LEN * 2 * c.num_heads * 64 * 2
    bytes_per_launch = int(bytes_dense * live_frac)
    k_ms = kms.value / max(1, kn.value)
    achieved = bytes_per_launch / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    return {"metric": "greedy generation tokens/sec (FiD-base, n_docs 40, KV-cached decode, encoder + cross K|V once)",
            "value": B * world * (TARGET_LEN - 1) / (ms_full * 1e-3), "unit": "tokens/s", "ms_per_generate": ms_full,
            "queries_per_generate": B * world, "tokens_per_query": TARGET_LEN - 1, "ms_encoder_and_first_step": ms_short,
            "ms_per_decode_step": step_ms, "decode_steps_per_s": 1e3 / step_ms if step_ms > 0 else None,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "peak_source": peak_src,
                         "kernel": "decode_cross_attention_kernel (one new token against the cached cross K|V)",
                         "kernel_ms_per_launch": k_ms, "launches_timed": kn.value,
                         "algorithmic_bytes_per_launch": bytes_per_launch,
                         "bytes_note": f"K | V rows of the live 64-key tiles ({live_frac:.3f} of all tiles; the others hold padding "
                                       f"only and are skipped): dense K | V = {bytes_dense} B per launch",
                         "dense_equivalent_GBps": bytes_dense / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None,
                         "step_bytes_all_layers": bytes_per_launch * c.num_decoder_layers,
                         "step_level_GBps": bytes_per_launch * c.num_decoder_layers / (step_ms * 1e-3) / 1e9 if step_ms > 0 else None}}


def xl_train_leg(args, atlas_base, index, bank_tokens, dev, world, rank, L, barrier_sync, max_over_ranks, steps=2, warmup=1):
    """BASELINE configs[4]: Atlas-xl (T5-v1.1-xl dims: d 2048, 32 heads, d_ff 5120, 24 + 24 layers, n_docs 40, text_maxlength
    384) retrieve + reader forward + backward + retriever distillation (`Atlas.forward(train_retriever=True)`,
    gold_score_mode ppmean, src/atlas.py:399-550, dropout 0), per GPU 1 query per step, gradient checkpointing on both
    models, followed at N > 1 by one NCCL all-reduce of the flattened gradients (what DDP does in train.py).  Reader input
    tokens/s (B * n_docs * text_maxlength per step, SURVEY.md §8d C5's unit) over all ranks."""
    import ctypes

    import torch
    import torch.distributed as dist

    from atlas_b200.atlas import Atlas
    from atlas_b200.fid import FiD, T5ConfigLite
    from atlas_b200.retrievers import BertConfigLite, Contriever, DualEncoderRetriever

    torch.manual_seed(1)
    with torch.device(dev):
        reader = FiD(T5ConfigLite(d_model=2048, d_ff=5120, num_layers=24, num_decoder_layers=24, num_heads=32))
        contriever = Contriever(BertConfigLite())
    reader = reader.to(torch.bfloat16).train()
    contriever = contriever.to(torch.bfloat16).train()
    opt = bench_opt(1)
    opt.use_gradient_checkpoint_reader = True
    opt.use_gradient_checkpoint_retriever = True
    atlas = Atlas(opt, reader, DualEncoderRetriever(opt, contriever), atlas_base.reader_tokenizer,
                  atlas_base.retriever_tokenizer).train()
    atlas.set_token_bank(bank_tokens)
    index.max_queries_per_rank = 1
    queries, targets = make_query_strings(1, 100 + rank)
    params = [p for p in atlas.parameters() if p.requires_grad]

    def step():
        for p in params:
            p.grad = None
        reader_loss, retriever_loss = atlas(index, queries, targets, train_retriever=True, iter_stats={})
        (reader_loss + retriever_loss).backward()
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in params if p.grad is not None])
            dist.all_reduce(flat)
        return reader_loss, retriever_loss

    try:
        for _ in range(warmup):
            rl, tl = step()
        barrier_sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            rl, tl = step()
        e1.record()
        barrier_sync()
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        assert bool(torch.isfinite(rl.float())) and bool(torch.isfinite(tl.float())), "non-finite xl training losses"
        shares = {}
        for kind, name in ((2, "gemm"), (3, "attention_fwd"), (4, "attention_bwd")):
            L.atlas_b200_profile_enable(kind)
            step()
            torch.cuda.synchronize()
            work = L.atlas_b200_profile_work()
            kms, kn = ctypes.c_double(0), ctypes.c_int32(0)
            L.atlas_b200_profile_collect(ctypes.byref(kms), ctypes.byref(kn))
            L.atlas_b200_profile_enable(0)
            shares[name] = {"ms_per_step": kms.value, "launches_per_step": kn.value,
                            "achieved_tflops": work / (kms.value * 1e-3) / 1e12 if kms.value > 0 else None,
                            "share_of_step": kms.value / ms if ms else None}
        peak_mem = torch.cuda.max_memory_allocated() / 2 ** 30
    finally:
        for p in params:
            p.grad = None
        del atlas, reader, contriever, params
        torch.cuda.empty_cache()
    tokens = N_DOCS * TEXT_LEN * world
    n_reader = 2849.8e6
    return {"metric": "Atlas-xl training tokens/sec (retrieve + T5-xl FiD forward + backward + ppmean retriever distillation, "
                      "bf16, dropout 0, checkpointing on)",
            "value": tokens / (ms * 1e-3), "unit": "tokens/s", "ms_per_step": ms, "steps": steps, "queries_per_step": world,
            "reader_tokens_per_step": tokens, "reader_loss": float(rl), "retriever_loss": float(tl),
            "reader_parameters": n_reader, "peak_memory_GiB": peak_mem,
            "gradient_allreduce": "one NCCL all-reduce of the flattened bf16 gradients" if world > 1 else "none (1 GPU)",
            "kernels": shares}


def refresh_leg(args, retriever, index, dev, world, L, barrier_sync, max_over_ranks, steps=5, warmup=2):
    """Index refresh (`Atlas.build_index`, src/atlas.py:61-88): one embedder batch of 512 synthetic passages (lengths
    U[64, 192] tokens, padded to the longest like the reference's tokenizer call) through Contriever-base with fp16
    weight copies, pooled rows written straight into bank rows (`Contriever.embed_into`).  Passages/s over all ranks (no
    communication: every rank rewrites its own shard) and the tensor-roofline fraction with SURVEY.md §8(d)'s FLOPs per
    token (169.9 MFLOP + 36 864 L).  Runs last: it overwrites the first 512 rows of the synthetic bank."""
    import torch

    nb, lmax = 512, 192
    g = torch.Generator().manual_seed(4242)
    lens = torch.randint(64, lmax + 1, (nb,), generator=g)
    lens[0] = lmax
    ids = torch.randint(1000, 30000, (nb, lmax), generator=g)
    mask = (torch.arange(lmax)[None, :] < lens[:, None]).to(torch.int64)
    ids = (ids * mask).to(dev)
    mask = mask.to(dev)
    rows = index._bank[:nb]

    def step():
        retriever.embed_into(ids, mask, rows, dtype=torch.float16)

    for _ in range(warmup):
        step()
    barrier_sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier_sync()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    assert bool(torch.isfinite(rows.float()).all()), "non-finite embeddings in the refresh leg"
    flops_dense = nb * lmax * (169.9e6 + 36864.0 * lmax)
    # the encoder runs on each passage's 64-row tiles up to its last real token (DESIGN.md 3.10): FLOPs of the rows computed
    from atlas_b200 import ops as _ops

    flops = flops_dense
    if _ops._ENC_PACKED and _ops._BERT_PACKED and lmax % 64 == 0:
        kept_rows = ((lens + 63) // 64 * 64).double()
        flops = float((kept_rows * 169.9e6 + 36864.0 * kept_rows * kept_rows).sum())
    peak, peak_src = peaks("tensor")
    achieved = flops / (ms * 1e-3) / 1e12
    return {"metric": "index refresh passages/sec (Contriever-base fp16 embed of 512-passage batches into bank rows)",
            "value": nb * world / (ms * 1e-3), "unit": "passages/s", "ms_per_batch": ms, "steps": steps,
            "passages_per_batch": nb, "padded_tokens": lmax, "tokens_per_s": nb * lmax * world / (ms * 1e-3),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak if peak else None, "peak_source": peak_src,
                         "algorithmic_flops_per_batch": flops, "flops_of_all_padded_positions": flops_dense,
                         "flops_note": "rows computed: every passage's 64-row tiles up to its last real token"
                                       if flops != flops_dense else "every padded position"},
            "shard_refresh_estimate_s": args.rows / (nb / (ms * 1e-3))}


def train_leg(args, reader, dev, world, L, barrier_sync, max_over_ranks, steps=3, warmup=2):
    """FiD-base forward + backward (`loss.backward()` through grad_ops.py's kernels; at N > 1 followed by one NCCL
    all-reduce of the flattened gradients, what DDP does in train.py) on `train_batch` queries x 40 passages x 384 tokens
    per GPU: reader tokens/s (B * n_docs * text_maxlength per step, SURVEY.md §8d C5's unit) and the share of the GEMM /
    attention-backward kernels.  Supplementary to the headline metric (which is the forward step)."""
    import ctypes

    import torch
    import torch.distributed as dist

    tb = min(args.batch, 2)
    reader.train()
    cfg = reader.encoder.config
    old = (cfg.n_context, cfg.bsz)
    cfg.n_context, cfg.bsz = N_DOCS, tb
    g = torch.Generator().manual_seed(99)
    ids = torch.randint(2, 32000, (tb, N_DOCS * TEXT_LEN), generator=g).to(dev)
    mask = torch.ones(tb, N_DOCS * TEXT_LEN, dtype=torch.bool, device=dev)
    labels = torch.randint(2, 32000, (tb, TARGET_LEN), generator=g).to(dev)
    # the supplementary `padded` figure: passages of the forward step's length distribution (query + U[128, 256] passage tokens,
    # padded to text_maxlength like src/atlas.py:261-270 pads) - the attention kernels skip all-padding key blocks
    plen = QUERY_TOKENS + torch.randint(PASSAGE_TOKENS // 2, PASSAGE_TOKENS + 1, (tb, N_DOCS), generator=g)
    mask_padded = (torch.arange(TEXT_LEN)[None, None, :] < plen[..., None]).reshape(tb, N_DOCS * TEXT_LEN).to(dev)
    ids_padded = ids * mask_padded

    def step(padded=False):
        reader.zero_grad(set_to_none=True)
        out = reader(input_ids=ids_padded if padded else ids, attention_mask=mask_padded if padded else mask, labels=labels)
        out[0].backward()
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in reader.parameters() if p.grad is not None])
            dist.all_reduce(flat)
        return out[0]

    try:
        for _ in range(warmup):
            loss = step()
        barrier_sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = step()
        e1.record()
        barrier_sync()
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        assert bool(torch.isfinite(loss.float())), "non-finite training loss"
        shares = {}
        for kind, name in ((2, "gemm"), (4, "attention_bwd")):
            L.atlas_b200_profile_enable(kind)
            step()
            torch.cuda.synchronize()
            work = L.atlas_b200_profile_work()
            kms, kn = ctypes.c_double(0), ctypes.c_int32(0)
            L.atlas_b200_profile_collect(ctypes.byref(kms), ctypes.byref(kn))
            L.atlas_b200_profile_enable(0)
            shares[name] = {"ms_per_step": kms.value, "launches_per_step": kn.value,
                            "achieved_tflops": work / (kms.value * 1e-3) / 1e12 if kms.value > 0 else None,
                            "share_of_step": kms.value / ms if ms else None}
        for _ in range(warmup):
            loss_p = step(True)
        barrier_sync()
        e0.record()
        for _ in range(steps):
            loss_p = step(True)
        e1.record()
        barrier_sync()
        ms_padded = max_over_ranks(e0.elapsed_time(e1)) / steps
        assert bool(torch.isfinite(loss_p.float())), "non-finite training loss (padded passages)"
    finally:
        reader.zero_grad(set_to_none=True)
        reader.eval()
        cfg.n_context, cfg.bsz = old
    tokens = tb * N_DOCS * TEXT_LEN * world
    return {"metric": "reader training tokens/sec (FiD-base forward + backward, bf16, dropout 0)",
            "value": tokens / (ms * 1e-3), "unit": "tokens/s", "ms_per_step": ms, "steps": steps,
            "queries_per_step": tb * world, "reader_tokens_per_step": tokens,
            "gradient_allreduce": "one NCCL all-reduce of the flattened bf16 gradients" if world > 1 else "none (1 GPU)",
            "kernels": shares,
            "mask": "every position real (no padding: the dense worst case)",
            "padded_passages": {"value": tokens / (ms_padded * 1e-3), "unit": "tokens/s (padded positions counted)",
                                "ms_per_step": ms_padded,
                                "what": f"the same step on passages of the forward step's length distribution (query + "
                                        f"U[{PASSAGE_TOKENS // 2}, {PASSAGE_TOKENS}] passage tokens padded to {TEXT_LEN}): "
                                        "all-padding key blocks are skipped by the attention kernels, forward and backward"}}


def mips_leg(args, index, dev, world, rank, L, barrier_sync, max_over_ranks):
    """search_knn alone: 256 queries / top-40 over the sharded bank (BASELINE configs[1] at N=1, configs[2] at N=8)."""
    import ctypes

    import torch

    from atlas_b200 import ops

    steps, warmup = max(20, args.steps), 5
    q_host = make_queries().pin_memory()
    per = NQ // world
    q_host_local = q_host[rank * per:(rank + 1) * per].contiguous().pin_memory() if world > 1 else q_host
    q_dev_local = q_host_local.to(dev)
    for _ in range(warmup):
        index.search_device(q_dev_local, TOPK, return_status=True)
    L.atlas_b200_profile_enable(1)
    barrier_sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        _, _, st = index.search_device(q_dev_local, TOPK, return_status=True)     # no host synchronisation
    e1.record()
    barrier_sync()
    assert int(st.item()) == 0, "fast search path overflowed in the MIPS leg"
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    kms, kn = ctypes.c_double(0), ctypes.c_int32(0)
    L.atlas_b200_profile_collect(ctypes.byref(kms), ctypes.byref(kn))
    L.atlas_b200_profile_enable(0)
    ms_per_step = total_ms / steps

    def e2e_step():
        if world == 1:
            return ops.search_host(index._bank, q_host_local, TOPK, workspace=index._workspace)
        return index.search_knn(q_host_local.to(dev, non_blocking=True), TOPK)

    for _ in range(3):
        e2e_step()
    barrier_sync()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    barrier_sync()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / steps
    peak, peak_src = peaks("hbm")
    kernel_ms = kms.value / steps
    alg_bytes = args.rows * DIM * 2
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r01_mips_scan_traffic.json")
    if os.path.exists(tpath):     # dram bytes of the sweep from the committed `ncu --set full` capture (see profiles/)
        with open(tpath) as f:
            traffic = json.load(f).get("dram_bytes_per_search")
    return {
        "metric": "retrieve queries/sec (exact top-40 search_knn, 256-query batches)", "value": NQ / (ms_per_step * 1e-3),
        "unit": "queries/s", "ms_per_step": ms_per_step, "steps": steps, "queries_per_step": NQ,
        "e2e": {"value": NQ / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": q_host_local.numel() * 4 * world,
                "d2h_bytes_per_step": NQ * TOPK * (2 + 8) if world > 1 else NQ * TOPK * (4 + 8),
                "call": "atlas_b200_search_host (C ABI, host buffers)" if world == 1 else
                        "DistributedIndex.search_knn (pinned host queries -> passage dicts + scores)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak if peak else None, "traffic": traffic, "peak_source": peak_src,
                     "kernel": "mips_scan_ts_kernel (bank sweep; one search = %d launches covering the bank once)"
                               % max(1, kn.value // steps),
                     "kernel_ms_per_search": kernel_ms, "kernel_launches_timed": kn.value,
                     "algorithmic_bytes_per_search": alg_bytes,
                     "kernel_share_of_step": kernel_ms / ms_per_step if ms_per_step else None},
        "aggregate_bank_GBps": world * alg_bytes / (ms_per_step * 1e-3) / 1e9,
    }


_JSON_FD = None


def emit(line):
    """The ONE JSON line of the contract goes to the process's original stdout; everything else that writes to fd 1
    during the run (NCCL prints its version there when NCCL_DEBUG=VERSION) has been pointed at stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    args = parse()
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
