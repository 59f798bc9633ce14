"""bench.py --dump-outputs: the last timed step's forest, written as .npy arrays, is the same for any --steps / --warmup and
is the forest the oracle builds from the same seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir, steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(steps), "--warmup", str(warmup),
           "--no-e2e", "--no-writer-e2e", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    names = sorted(os.listdir(out_dir))
    arrays = {f[:-4]: np.load(os.path.join(out_dir, f)) for f in names}
    assert all(f.endswith(".npy") for f in names)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in names) <= bench.DUMP_LIMIT_BYTES
    return arrays


def test_dumped_forest_is_reproducible_and_equals_the_oracle_forest(tmp_path):
    a = _bench_dump(tmp_path / "a", steps=2, warmup=1)
    b = _bench_dump(tmp_path / "b", steps=1, warmup=0)
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), k
    wl = bench.WORKLOADS["c1"]
    n, d, T = wl["n"], wl["d"], wl["n_trees"]
    db = oracle.Db(wl["metric"], d)
    db.set_items(np.arange(n, dtype=np.uint32), oracle.synth_rows(bench.SEED, d, 0, n, wl["centre"]))
    db.build(oracle.StdRng(bench.SEED), n_trees=T, threads=4)
    nodes = {k: oracle.decode_node(v, oracle.EUCLIDEAN, d) for k, v in db.nodes().items()}
    assert a["node_counts"].sum() == len(nodes)
    splits = {int(r[0]): r for r in a["split_nodes"]}
    desc = {int(i): int(c) for i, c in a["descendants"]}
    assert len(splits) + len(desc) == len(nodes)
    for k, nd in nodes.items():
        if nd["kind"] == "descendants":
            assert desc[k] == len(nd["descendants"]), k
        else:
            assert (splits[k][1], splits[k][2]) == (nd["left"], nd["right"]), k
            if nd["normal"] is not None:
                assert np.float32(splits[k][3]) == nd["header"][0], k
    for i, v in zip(a["split_normal_ids"], a["split_normals"]):
        want = nodes[int(i)]["normal"]
        assert np.isnan(v).all() if want is None else v.tobytes() == want.tobytes()
    leaf = a["leaf_of_sampled_items"]
    assert leaf.shape == (T, len(a["sampled_items"]))
    for t in range(T):
        for j in range(0, leaf.shape[1], 101):
            assert int(a["sampled_items"][j]) in nodes[int(leaf[t, j])]["descendants"]
