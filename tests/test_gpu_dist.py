"""GPU: the multi-GPU stage kernels.  Virtual ranks (threads sharing one GPU, exchanges by
tensor slicing) always run; the real NCCL run needs >= 2 GPUs."""
import subprocess
import sys
import threading

import numpy as np
import pytest

from conftest import ROOT, corpus_text

pytestmark = pytest.mark.gpu


EXCHANGES = ("peer", "collective")


def run_virtual(stb, world, leaves_np, S, cut, exchange="peer"):
    import torch
    from genome_compression_b200.dist import CudaStages, DistBuilder, ShardPlan, ThreadComm

    n = len(leaves_np)
    shared = ThreadComm.Shared(world)
    plan = ShardPlan(n, world, cut)
    results, errors = [None] * world, []

    def work(rank):
        try:
            torch.cuda.set_device(0)
            lo, hi = plan.level_range(rank, 0)
            local = torch.from_numpy(leaves_np[lo:hi].view(np.int64).copy()).cuda()
            builder = DistBuilder(CudaStages(stb, S, 0), comm=ThreadComm(shared, rank), cut=cut, exchange=exchange)
            tree = builder.build_from_leaves(local, n)
            results[rank] = builder.gather(tree)
            builder.close()
        except Exception as e:  # noqa: BLE001
            errors.append(e)
            shared.barrier.abort()

    threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    if errors:
        raise errors[0]
    return results[0]


@pytest.mark.parametrize("exchange", EXCHANGES)
@pytest.mark.parametrize("world,cut", [(1, 1 << 16), (2, 64), (4, 1), (8, 1024)])
def test_virtual_ranks_match_single_gpu(stb, oracle, world, cut, exchange):
    text = corpus_text("merged")
    leaves = oracle.fasta_to_leaves(text, 12)
    full = run_virtual(stb, world, leaves, 12, cut, exchange)
    single = stb.SharedTree(12).build_from_leaves(leaves)
    assert full.layer_counts() == single.layer_counts()
    assert full.serialize() == single.serialize() == oracle.build(leaves, 12).serialize()
    full.sort()
    single.sort()
    assert full.serialize() == single.serialize()
    assert np.array_equal(full.decode(), leaves)


@pytest.mark.parametrize("S,n", [(16, 30000), (5, 70001), (12, 1), (12, 3)])
def test_virtual_ranks_iupac_and_edges(stb, oracle, S, n):
    rng = np.random.default_rng(S * 1000 + n)
    codes = np.array([1, 2, 4, 8, 3, 12, 7, 14, 0, 9, 5, 11, 13, 10, 6, 15], dtype=np.uint64)
    nib = codes[rng.integers(0, 16, size=(n, S))]
    leaves = (nib << (4 * np.arange(S, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
    if n > 100:
        leaves[n // 2:n // 2 + n // 4] = leaves[:n // 4]
        if S == 16:
            leaves[[3, 99, n - 1]] = np.uint64(0xFFFFFFFFFFFFFFFF)
    want = oracle.build(leaves, S)
    for world, exchange in ((2, "peer"), (3, "peer"), (3, "collective")):
        full = run_virtual(stb, world, leaves, S, cut=16, exchange=exchange)
        assert full.serialize() == want.serialize(), (S, n, world, exchange)


def test_virtual_ranks_synthetic_large(stb):
    import torch
    n_bases = 48_000_000
    buf = torch.empty(n_bases, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n_bases, seed=3, repeat_permille=500)
    single = stb.SharedTree(12).build_from_body(buf)
    leaves = stb.SharedTree(12).pack_fasta(buf)
    for exchange in EXCHANGES:
        full = run_virtual(stb, 4, leaves, 12, cut=1 << 14, exchange=exchange)
        assert full.layer_counts() == single.layer_counts()
        assert full.serialize() == single.serialize()


def test_rank_index_past_1024_blocks(stb):
    """More than 1024 blocks of 1024 words: the scan of the block sums carries across its
    1024-element rounds."""
    import torch
    from genome_compression_b200.dist import CudaStages

    n_words = (1 << 21) + 777
    bitmap = np.random.default_rng(21).integers(0, 1 << 32, size=n_words, dtype=np.uint64).astype(np.uint32)
    stages = CudaStages(stb, 12, 0)
    bitmap_dev = torch.from_numpy(bitmap.view(np.int32)).cuda()
    word_prefix = torch.empty(n_words + 1, dtype=torch.int32, device="cuda")
    scratch = torch.empty(-(-n_words // 1024) + 1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    stages.rank_index(bitmap_dev, n_words, word_prefix, scratch)
    torch.cuda.synchronize()
    popcount = np.unpackbits(bitmap.view(np.uint8)).reshape(n_words, 32).sum(axis=1)
    want = np.concatenate([[0], np.cumsum(popcount)]).astype(np.uint32)
    assert np.array_equal(word_prefix.cpu().numpy().view(np.uint32), want)


def test_nccl_two_ranks(stb):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (run with gpurun --gpus 2)")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29531", str(ROOT / "tests" / "dist_gpu_check.py"), "60000000"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "dist_gpu_check ok" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


def test_virtual_ranks_from_text_direct_leaf_table(stb, oracle):
    """Text entry point: replicated direct-addressed leaf table + all-reduce(MIN); an IUPAC
    symbol anywhere makes every rank fall back to the record exchange."""
    import torch
    from genome_compression_b200.dist import CudaStages, DistBuilder, ShardPlan, ThreadComm

    for text, S, world in ((corpus_text("merged").upper(), 12, 4), (corpus_text("humhbb").upper(), 5, 3),
                           (corpus_text("humhbb").upper().replace(b"ACGT", b"ACNT", 3), 12, 2)):
        n = len(text) // S
        shared = ThreadComm.Shared(world)
        plan = ShardPlan(n, world, cut=64)
        out, errors = [None] * world, []

        def work(rank):
            try:
                torch.cuda.set_device(0)
                lo, hi = plan.level_range(rank, 0)
                body = torch.frombuffer(bytearray(text[lo * S:hi * S] + b"A" * 16), dtype=torch.uint8).cuda()
                builder = DistBuilder(CudaStages(stb, S, 0), comm=ThreadComm(shared, rank), cut=64)
                out[rank] = builder.gather(builder.build_from_body(body, n * S))
                builder.close()
            except Exception as e:  # noqa: BLE001
                errors.append(e)
                shared.barrier.abort()

        threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        assert not errors, errors
        want = oracle.build(oracle.fasta_to_leaves(text, S), S)
        assert out[0].serialize() == want.serialize(), (S, world)
