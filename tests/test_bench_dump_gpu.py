"""bench.py --dump-outputs end to end on the device: the file holds the sketch of the seeded
input block that the timed step computed (shrunken workloads; rows sampled as in srht_c3)."""
import json
import os
import sys

import numpy as np
import pytest
import torch

from test_bench_contract import _load_bench


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gauss_c2", "srht_c1"])
def test_dump_outputs_is_the_sketch_of_the_timed_step(tmp_path, monkeypatch, capsys, name):
    import rla4mor_b200 as rb
    from rla4mor_b200 import dense
    bench = _load_bench()
    kind = bench.WORKLOADS[name]["kind"]
    m, logn, k, keep = 40, 12, 100, 16
    monkeypatch.setitem(bench.WORKLOADS, name, dict(kind=kind, m=m, logn=logn, k=k, config="shrunk"))
    monkeypatch.setattr(bench, "DUMP_BYTES_PER_OUTPUT", keep * k * 8)        # keep 16 of the 40 rows
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("LOCAL_RANK", raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--workload", name, "--steps", "2", "--no-secondary", "--no-e2e",
                                      "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "dump")])
    bench.run_ours(bench.parse())
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == 2 and len(line["roofline"]["step_ms"]) == 2
    assert os.listdir(tmp_path / "dump") == [name + ".npy"]
    got = np.load(tmp_path / "dump" / (name + ".npy"))

    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(1234)                    # bench.py's block of rank 0
    U = torch.empty((m, 2 ** logn), dtype=torch.float64, device=dev)
    for lo in range(0, m, 32):
        U[lo:lo + 32].normal_(generator=gen)
    if kind == "gauss":
        want = dense.embed_apply_rng(0, dense.KIND_NORMAL, 1.0 / np.sqrt(k), k, U)
    else:
        emb = rb.SrhtEmbedding(source=rb.DeviceVectorSpace(2 ** logn), options={"range_dim": k}, _seed=0)
        want = emb._plan(torch.float64, dev).apply(U)
    rows = np.sort(np.random.RandomState(0).choice(m, keep, replace=False))
    assert got.dtype == np.float64 and got.shape == (keep, k)
    assert np.array_equal(got, want.cpu().numpy()[rows])
