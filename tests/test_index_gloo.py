"""CPU, world_size 2 and 4 over gloo: the HOST logic of `atlas_b200.index.DistributedIndex.search_knn`
(query exchange, global-id mapping, packed result exchange, merge bookkeeping, passage lookup through
the node-shared store, save/load round trip) against the golden outputs of the reference index.

The CUDA scan/merge are replaced IN THIS TEST ONLY by the numpy oracle (the product classes have no
CPU path and raise without a GPU); the NCCL + kernel version of the same flow is covered by
tests/test_search_gpu.py under `-m gpu`.
"""
import os
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from conftest import ROOT, golden_inputs, load_golden


def _make_cpu_index_class():
    import mips_oracle
    from atlas_b200.index import DistributedIndex

    class OracleBackedIndex(DistributedIndex):
        """Host logic of the product class; device kernels swapped for the oracle (test only)."""

        @staticmethod
        def _device():
            return torch.device("cpu")

        def _local_search(self, allqueries, topk, exhaustive=False):
            bank = self._bank.numpy()
            s = mips_oracle.scores_fp16(allqueries.float().numpy(), bank)
            v, local = mips_oracle.canonical_topk(s, topk)
            status = torch.zeros(1, dtype=torch.int32)     # the device overflow flag of the fast path (never set here)
            return torch.from_numpy(v), torch.from_numpy(self._id_base + self._id_stride * local), status

        def _merge(self, blob_all, ids_off, world, nq_total, topk, q_begin, nq_out):
            nb = nq_total * topk
            vs = torch.stack([blob_all[w, : nb * 2].view(torch.float16).view(nq_total, topk) for w in range(world)])
            ids = torch.stack([blob_all[w, ids_off:ids_off + nb * 8].view(torch.int64).view(nq_total, topk)
                               for w in range(world)])
            out_v = np.empty((nq_out, topk), np.float16)
            out_i = np.empty((nq_out, topk), np.int64)
            for j in range(nq_out):
                cv = vs[:, q_begin + j].reshape(-1).numpy()
                ci = ids[:, q_begin + j].reshape(-1).numpy()
                order = np.lexsort((ci, -(cv.astype(np.float32) + 0.0)))[:topk]
                out_v[j], out_i[j] = cv[order], ci[order]
            return torch.from_numpy(out_v), torch.from_numpy(out_i)

    return OracleBackedIndex


def _worker(rank, world, name, rendezvous, tmpdir, store_mode, capacity=None):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import synth
    import mips_oracle

    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), ATLAS_B200_PASSAGE_STORE=store_mode)
    torch.distributed.init_process_group("gloo", init_method=f"file://{rendezvous}", rank=rank, world_size=world)
    try:
        g = load_golden(name)
        bank, q, nq_per_rank = golden_inputs(g)
        k = int(g["k"])
        n = bank.shape[0]
        off = np.cumsum([0] + nq_per_rank)
        Index = _make_cpu_index_class()
        index = Index()
        index.max_queries_per_rank = capacity        # fixed per-rank capacity: no size exchange in front of the gather
        index.init_embeddings(synth.make_passages(n, rank, world))
        rows = mips_oracle.shard_rows(n, rank, world)
        # the reference's write pattern: index.embeddings[:, a:b] = emb.T   (src/atlas.py:79)
        index.embeddings[:, : len(rows)] = torch.from_numpy(bank[rows]).T
        docs, scores = index.search_knn(torch.from_numpy(q[off[rank]:off[rank + 1]]), k)
        want_ids = g["canon_ids"][off[rank]:off[rank + 1]]
        want_scores = g["ref_scores"][off[rank]:off[rank + 1]]
        got_ids = np.array([[int(d["id"]) for d in row] for row in docs], dtype=np.int64).reshape(-1, k)
        got_scores = np.array(scores, dtype=np.float32).reshape(-1, k).astype(np.float16)
        assert len(docs) == nq_per_rank[rank]
        assert np.array_equal(got_ids, want_ids), (rank, got_ids[:1], want_ids[:1])
        assert np.array_equal(got_scores.view(np.uint16), want_scores.view(np.uint16))
        for row in docs:
            for d in row:
                assert d["title"] == f"t{d['id']}"
        # save / load round trip in the reference's on-disk format (src/index.py:61-111)
        index.save_index(tmpdir, 2 * world)
        torch.distributed.barrier()
        index2 = Index()
        index2.load_index(tmpdir, 2 * world)
        assert index2.embeddings.shape == (768, len(rows))
        assert torch.equal(index2.embeddings, index.embeddings)
        docs2, scores2 = index2.search_knn(torch.from_numpy(q[off[rank]:off[rank + 1]]), k)
        assert scores2 == scores
        # after load the global numbering is contiguous per rank, not round-robin: same passages as long
        # as no tie straddles (ids order inside a tie may differ) -> compare as sets per row on unique scores
        for a, b, srow in zip(docs, docs2, scores):
            ida = [int(d["id"]) for d in a]
            idb = [int(d["id"]) for d in b]
            for p in range(k):
                if srow.count(srow[p]) == 1 and srow[p] != srow[-1]:
                    assert ida[p] == idb[p]
        index._reset_store()
        index2._reset_store()
    finally:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


@pytest.mark.parametrize("name,world,store,capacity", [("w2_grid", 2, "shm", None), ("w4_grid_empty_rank", 4, "shm", None),
                                                       ("w2_grid", 2, "exchange", None),
                                                       ("w4_grid_empty_rank", 4, "shm", 64), ("w2_grid", 2, "shm", 64)])
def test_search_knn_host_logic_gloo(name, world, store, capacity):
    # rendezvous through a file of a private directory: no fixed TCP port that a concurrent run on the same host could hold
    with tempfile.TemporaryDirectory() as tmp, tempfile.TemporaryDirectory() as rdzv:
        mp.spawn(_worker, args=(world, name, os.path.join(rdzv, "store"), tmp, store, capacity), nprocs=world, join=True)


def test_capacity_overflow_raises():
    """More local queries than `max_queries_per_rank` is a configuration error, not a silent truncation."""
    from atlas_b200._lib import AtlasB200Error

    Index = _make_cpu_index_class()
    index = Index()
    index.max_queries_per_rank = 2
    index._bank = torch.zeros(8, 768, dtype=torch.float16)
    import atlas_b200.dist_utils as du

    old = du.get_world_size
    du.get_world_size = lambda: 2
    try:
        with pytest.raises(AtlasB200Error):
            index.search_device(torch.zeros(3, 768), 4)
    finally:
        du.get_world_size = old


def test_single_rank_host_logic():
    """world_size 1 path (no process group) with the golden C1 case."""
    import mips_oracle
    import synth

    g = load_golden("c1_grid")
    bank, q, _ = golden_inputs(g)
    Index = _make_cpu_index_class()
    index = Index()
    index.init_embeddings(synth.make_passages(bank.shape[0]))
    index.embeddings[:, :] = torch.from_numpy(bank).T
    docs, scores = index.search_knn(torch.from_numpy(q), int(g["k"]))
    ids = np.array([[int(d["id"]) for d in row] for row in docs])
    assert np.array_equal(ids, g["canon_ids"])
    assert np.array_equal(np.array(scores, dtype=np.float32).astype(np.float16).view(np.uint16),
                          g["ref_scores"].view(np.uint16))
    with pytest.raises(RuntimeError):
        index.search_knn(torch.from_numpy(q), bank.shape[0] + 1)


def test_product_index_has_no_cpu_path():
    from atlas_b200._lib import AtlasB200Error
    from atlas_b200.index import DistributedFAISSIndex, DistributedIndex

    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(AtlasB200Error):
        DistributedIndex().init_embeddings([{"id": "0"}])
    with pytest.raises(AtlasB200Error):
        DistributedFAISSIndex("ivfpq", 64)
