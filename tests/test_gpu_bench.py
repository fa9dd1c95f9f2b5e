"""GPU: bench.py --dump-outputs writes the tree of the last timed build, the same tables a direct build of the
same seeded input returns."""
import json

import numpy as np
import pytest

from test_bench_contract import run_bench

pytestmark = pytest.mark.gpu


def test_dump_outputs_hold_the_timed_build(stb, tmp_path):
    import torch
    n, seed = 24_000_000, 5
    res = run_bench("--steps", "2", "--warmup", "1", "--bases", str(n), "--seed", str(seed), "--no-cpu-baseline", "--no-e2e",
                    "--no-pipeline", "--dump-outputs", str(tmp_path))
    assert res.returncode == 0, res.stderr[-2000:]
    assert json.loads(res.stdout)["steps"] == 2
    paths = sorted(tmp_path.glob("*.npy"))
    assert [p.stem for p in paths] == ["counts", "layer_counts", "leaves", "nodes"]
    assert sum(p.stat().st_size for p in paths) <= 64_000_000
    got = {p.stem: np.load(p) for p in paths}
    assert all(a.dtype == np.float64 for a in got.values())

    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=seed, repeat_permille=500)
    tree = stb.SharedTree(12).build_from_body(buf)
    assert got["counts"].tolist() == [tree.width(), tree.depth(), tree.leaf_count(), tree.node_count(), tree.root()]
    assert got["layer_counts"].tolist() == tree.layer_counts()
    leaves = got["leaves"].astype(np.uint64)
    assert len(leaves) == min(tree.leaf_count(), 1 << 20)
    assert np.array_equal(leaves[:, 1], tree.leaves()[leaves[:, 0].astype(np.int64)])
    nodes = got["nodes"].astype(np.int64)
    for k in range(tree.depth() - 1):
        rows = nodes[nodes[:, 0] == k]
        assert len(rows) > 0 and np.array_equal(rows[:, 2:].astype(np.uint32), tree.layer(k)[rows[:, 1]]), k
