"""GPU parity tests for the MIPS + top-k path (csrc/mips.cu) through the C ABI.

Bars: bit-exact scores AND ids against the oracle / the reference goldens on exact-grid inputs;
<= 1 fp16 ulp + tie-aware ids on realistic (gauss) inputs; size-independent properties at
BASELINE.json's full size (4 Mi x 768)."""
import numpy as np
import pytest
import torch

import mips_oracle
import synth
from conftest import golden_inputs, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from atlas_b200._lib import lib

    lib()  # fail loudly if the CUDA library is missing
    return torch.device("cuda:0")


def _run(bank_np, q_np, k, dev, **kw):
    from atlas_b200 import ops

    s, i = ops.search_shard(torch.from_numpy(bank_np).to(dev), torch.from_numpy(q_np).to(dev), k, **kw)
    return s.cpu().numpy(), i.cpu().numpy()


@pytest.mark.parametrize("name", ["c1_grid", "c1_grid_k80", "ragged_k5", "k_equals_n"])
def test_golden_bit_exact(name, dev):
    g = load_golden(name)
    bank, q, _ = golden_inputs(g)
    s, i = _run(bank, q, int(g["k"]), dev)
    assert np.array_equal(s.view(np.uint16), g["ref_scores"].view(np.uint16))  # reference values, tie-free
    assert np.array_equal(i, g["canon_ids"])                                   # canonical tie rule
    for r in range(s.shape[0]):                                                # reference's own pick
        assert mips_oracle.ids_match_tie_aware(g["ref_scores"][r], g["ref_ids"][r], i[r])


def test_golden_gauss_tolerance(dev):
    g = load_golden("c1_gauss")
    bank, q, _ = golden_inputs(g)
    s, i = _run(bank, q, int(g["k"]), dev)
    ref = g["ref_scores"].astype(np.float32)
    ulp = np.spacing(np.abs(g["ref_scores"])).astype(np.float32)
    assert np.all(np.abs(s.astype(np.float32) - ref) <= ulp), "scores differ by more than 1 fp16 ulp"
    # ids: identical wherever the reference score is separated from its neighbours by > 2 ulp
    for r in range(s.shape[0]):
        for p in range(s.shape[1]):
            lo = ref[r, p + 1] if p + 1 < s.shape[1] else -np.inf
            hi = ref[r, p - 1] if p > 0 else np.inf
            if p + 1 < s.shape[1] and ref[r, p] - lo > 2 * ulp[r, p] and hi - ref[r, p] > 2 * ulp[r, p]:
                assert i[r, p] == g["canon_ids"][r, p]


@pytest.mark.parametrize("n,nq,k", [(128, 1, 1), (129, 7, 129), (1000, 130, 33), (5000, 300, 40), (40000, 256, 128),
                                    (3000, 5, 1024)])
def test_oracle_bit_exact_shapes(n, nq, k, dev):
    bank = synth.make_bank(n, seed=n)
    q = synth.make_queries(nq, seed=nq)
    want_v, want_i = mips_oracle.canonical_topk(mips_oracle.scores_fp16(q, bank), k)
    s, i = _run(bank, q, k, dev)
    assert np.array_equal(s.view(np.uint16), want_v.view(np.uint16))
    assert np.array_equal(i, want_i)


def test_sampled_path_and_exhaustive_agree(dev):
    from atlas_b200 import ops

    n, nq, k = 300000, 200, 40  # n > candidate capacity -> threshold-from-sample path
    bank = synth.make_bank(n, seed=77)
    q = synth.make_queries(nq, seed=78)
    b, qt = torch.from_numpy(bank).to(dev), torch.from_numpy(q).to(dev)
    s1, i1, st = ops.mips_topk(b, qt, k)
    assert int(st.item()) == 0
    s2, i2, _ = ops.mips_topk(b, qt, k, exhaustive=True)
    assert torch.equal(s1, s2) and torch.equal(i1, i2)
    want_v, want_i = mips_oracle.canonical_topk(mips_oracle.scores_fp16(q, bank), k)
    assert np.array_equal(i1.cpu().numpy(), want_i)
    assert np.array_equal(s1.cpu().numpy().view(np.uint16), want_v.view(np.uint16))


def test_global_id_mapping(dev):
    bank = synth.make_bank(999, seed=1)
    q = synth.make_queries(3, seed=2)
    _, i0 = _run(bank, q, 9, dev)
    _, i1 = _run(bank, q, 9, dev, id_base=5, id_stride=8)
    assert np.array_equal(i1, 5 + 8 * i0)


def test_all_ties_overflow_falls_back(dev):
    """A zero bank (what init_embeddings leaves before build_index, src/index.py:51) ties every score:
    the candidate lists overflow, status is raised, and the exhaustive path returns the k lowest ids."""
    from atlas_b200 import ops

    n, k = 70000, 40
    bank = torch.zeros(n, 768, dtype=torch.float16, device=dev)
    q = torch.from_numpy(synth.make_queries(4, seed=3)).to(dev)
    _, _, st = ops.mips_topk(bank, q, k)
    assert int(st.item()) == 1
    s, i = ops.search_shard(bank, q, k)
    assert torch.all(s == 0)
    assert torch.equal(i.cpu(), torch.arange(k).repeat(4, 1))


def test_adversarial_order(dev):
    """Scores increasing with the row index (worst case for any running threshold)."""
    n, k = 200000, 40
    base = synth.make_queries(1, seed=9)[0].astype(np.float16)
    scale = (np.arange(n, dtype=np.float32) / n).astype(np.float16)
    bank = (scale[:, None] * np.sign(base)[None, :] * 0.5).astype(np.float16)
    q = np.sign(base)[None, :].astype(np.float32)
    want_v, want_i = mips_oracle.canonical_topk(mips_oracle.scores_fp16(q, bank), k)
    s, i = _run(bank, q, k, dev)
    assert np.array_equal(s.view(np.uint16), want_v.view(np.uint16))
    assert np.array_equal(i, want_i)


def test_argument_errors(dev):
    from atlas_b200 import ops
    from atlas_b200._lib import AtlasB200Error

    bank = torch.zeros(64, 768, dtype=torch.float16, device=dev)
    q = torch.zeros(2, 768, device=dev)
    with pytest.raises(AtlasB200Error, match="k out of range"):   # torch.topk raises in the reference
        ops.mips_topk(bank, q, 65)
    with pytest.raises(AtlasB200Error):
        ops.mips_topk(bank, q, 2000)
    s, i, _ = ops.mips_topk(bank, q[:0], 5)                         # zero queries is legal
    assert s.shape == (0, 5) and i.shape == (0, 5)


def test_search_host_equals_device_path(dev):
    from atlas_b200 import ops

    bank = synth.make_bank(30000, seed=21)
    q = synth.make_queries(64, seed=22, dist="gauss")
    b = torch.from_numpy(bank).to(dev)
    s_d, i_d = ops.search_shard(b, torch.from_numpy(q).to(dev), 40)
    s_h, i_h = ops.search_host(b, torch.from_numpy(q).pin_memory(), 40)
    assert torch.equal(i_h, i_d.cpu())
    assert torch.equal(s_h, s_d.float().cpu())


def test_merge_kernel_matches_oracle(dev):
    from atlas_b200 import ops

    world, n, k = 4, 4000, 40
    bank = synth.make_bank(n, seed=31)
    qs = [synth.make_queries(m, seed=40 + r) for r, m in enumerate([3, 0, 5, 2])]
    want = mips_oracle.search_knn_oracle(bank, qs, k)
    allq = np.concatenate(qs)
    shard_s, shard_i = [], []
    for r in range(world):
        rows = mips_oracle.shard_rows(n, r, world)
        s, i = _run(bank[rows], allq, k, dev, id_base=r, id_stride=world)
        shard_s.append(torch.from_numpy(s))
        shard_i.append(torch.from_numpy(i))
    S = torch.stack(shard_s).to(dev)
    I = torch.stack(shard_i).to(dev)
    off = np.cumsum([0] + [len(x) for x in qs])
    for r in range(world):
        ms, mi = ops.topk_merge(S, I, world, allq.shape[0], k, int(off[r]), len(qs[r]))
        assert np.array_equal(mi.cpu().numpy(), want[r][1])
        assert np.array_equal(ms.cpu().numpy().view(np.uint16), want[r][0].view(np.uint16))


def test_index_module_drop_in(dev, tmp_path):
    """The reference-shaped surface (SURVEY.md §8b): slice-assign into `embeddings`, search, save/load."""
    from atlas_b200.index import DistributedIndex

    g = load_golden("c1_grid")
    bank, q, _ = golden_inputs(g)
    k = int(g["k"])
    index = DistributedIndex()
    index.init_embeddings(synth.make_passages(bank.shape[0]))
    assert index.embeddings.shape == (768, bank.shape[0]) and index.embeddings.dtype == torch.float16
    step = 512  # build_index writes 512-passage batches: index.embeddings[:, a:b] = emb.T (src/atlas.py:79)
    for a in range(0, bank.shape[0], step):
        emb = torch.from_numpy(bank[a:a + step]).to(dev)
        index.embeddings[:, a:a + len(emb)] = emb.T
    docs, scores = index.search_knn(torch.from_numpy(q).to(dev), k)
    ids = np.array([[int(d["id"]) for d in row] for row in docs])
    assert np.array_equal(ids, g["canon_ids"])
    assert np.array_equal(np.array(scores, dtype=np.float32).astype(np.float16).view(np.uint16),
                          g["ref_scores"].view(np.uint16))
    docs0, scores0 = index.search_knn(torch.empty(0, 768, device=dev), k)
    assert docs0 == [] and scores0 == []
    index.save_index(str(tmp_path), 4)
    emb0 = torch.load(str(tmp_path / "embeddings.0.pt"))
    assert emb0.shape == (768, 2500) and emb0.dtype == torch.float16 and emb0.is_contiguous()
    index2 = DistributedIndex()
    index2.load_index(str(tmp_path), 4)
    assert torch.equal(index2.embeddings, index.embeddings)
    docs2, scores2 = index2.search_knn(torch.from_numpy(q).to(dev), k)
    assert scores2 == scores and [[d["id"] for d in r] for r in docs2] == [[d["id"] for d in r] for r in docs]


def test_bf16_bank_variant(dev):
    from atlas_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(5)
    bank = (torch.randint(-16, 17, (20000, 768), generator=g).float() / 8).to(torch.bfloat16).to(dev)
    q = (torch.randint(-16, 17, (17, 768), generator=g).float() / 8).to(dev)
    s, i = ops.search_shard(bank, q, 40)
    full = (q.to(torch.bfloat16).float() @ bank.float().T).to(torch.bfloat16)  # exact products/sums on this grid
    v, ix = torch.sort(full.float(), dim=1, descending=True, stable=True)
    assert torch.equal(s.float(), v[:, :40])
    assert torch.equal(i, ix[:, :40])


def test_full_size_properties(dev):
    """BASELINE.json configs[1]: 4 Mi x 768 fp16 bank, 256 queries, top-40.  Exact-grid bank so that
    cuBLAS and tcgen05 accumulation agree bit-for-bit; checked against torch on the GPU in chunks."""
    from atlas_b200 import ops

    n, nq, k = 4 * 1024 * 1024, 256, 40
    gen = torch.Generator(device=dev).manual_seed(11)
    bank = torch.empty(n, 768, dtype=torch.float16, device=dev)
    for s0 in range(0, n, 1 << 18):
        x = torch.randn(1 << 18, 768, device=dev, generator=gen)
        bank[s0:s0 + (1 << 18)] = (torch.clamp(torch.round(x * 8) / 8, -4, 4)).half()
    x = torch.randn(nq, 768, device=dev, generator=gen)
    q = torch.clamp(torch.round(x * 8) / 8, -4, 4)
    s, i, st = ops.mips_topk(bank, q, k)
    assert int(st.item()) == 0
    # property 1: sorted descending, ids in range and distinct per row
    assert torch.all(s[:, :-1] >= s[:, 1:])
    assert int(i.min()) >= 0 and int(i.max()) < n
    assert all(len(set(r)) == k for r in i[:8].tolist())
    # property 2: returned scores are the exact fp16 dot products of the returned rows
    rows = bank[i[:16].reshape(-1)].float().view(16, k, 768)
    dots = torch.einsum("qkd,qd->qk", rows, q[:16].half().float()).half()
    assert torch.equal(dots, s[:16])
    # property 3: equals the reference computation (matmul + canonical top-k) on a query subset
    sub = slice(0, 32)
    full = torch.matmul(q[sub].half(), bank.T)                       # [32, 4Mi] fp16, src/index.py:117
    v, ix = torch.sort(full.float(), dim=1, descending=True, stable=True)
    assert torch.equal(s[sub].float(), v[:, :k])
    assert torch.equal(i[sub], ix[:, :k])
    # property 4: nothing outside the result beats the k-th score
    assert torch.all((full > s[sub, -1:]).sum(dim=1) <= k - 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_distributed_search_nccl(tmp_path):
    """NCCL world of 2: sharded bank, query all-gather, packed result all-gather, merge kernel."""
    import subprocess
    import sys

    from conftest import ROOT

    script = ROOT + "/tests/_nccl_worker.py"
    res = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
         "127.0.0.1", "--master-port", "29877", script],
        capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]


def test_streamed_index_load(dev, tmp_path):
    """`load_index` streams the reference-format shard files ([768, n] fp16, src/index.py:75-87) through pinned chunks and a
    GPU transpose: any chunk width (even / odd tails, wider than a shard) reproduces the bank bit for bit."""
    from atlas_b200.index import DistributedIndex

    g = torch.Generator().manual_seed(77)
    shards = [torch.randn(768, n, generator=g).half() for n in (2501, 64, 1999)]
    files = []
    for i, t in enumerate(shards):
        f = str(tmp_path / f"embeddings.{i}.pt")
        torch.save(t, f)
        files.append(f)
    want = torch.cat([t.t() for t in shards], 0).contiguous()
    for width in (262144, 1000, 333, 8):
        bank = DistributedIndex._load_bank_streamed(files, dev, chunk_cols=width)
        assert bank.shape == want.shape and bank.is_contiguous()
        assert torch.equal(bank.cpu(), want), width
