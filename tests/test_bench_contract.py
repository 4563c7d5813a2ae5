"""bench.py contract (CPU only): defaults, workload table, and the JSON line of the reference arm
on a shrunken workload (the real sizes are BASELINE.json's; here only the keys are checked)."""
import importlib.util
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_defaults_and_workloads(monkeypatch):
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    args = bench.parse()
    assert args.gpus == 1 and args.steps >= 1 and args.warmup >= 3 and args.impl == "ours"
    assert args.workload == "gauss_c2"                                   # BASELINE.json configs[1]
    wl = bench.WORKLOADS
    assert wl["gauss_c2"] == dict(kind="gauss", m=512, logn=22, k=2000, config="configs[1]")
    assert wl["srht_c3"]["m"] == 1024 and wl["srht_c3"]["logn"] == 24 and wl["srht_c3"]["k"] == 4000
    assert wl["srht_c1"]["m"] == 200 and wl["srht_c1"]["logn"] == 16 and wl["srht_c1"]["k"] == 1000


def test_reference_arm_json_line(monkeypatch, capsys):
    bench = _load_bench()
    for name, kind in (("gauss_c2", "gauss"), ("srht_c3", "srht")):
        monkeypatch.setitem(bench.WORKLOADS, name, dict(kind=kind, m=8, logn=12, k=100, config="shrunk"))
        monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
                                          "--workload", name])
        monkeypatch.setenv("RANK", "0")
        bench.run_reference(bench.parse())
        line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
        assert line["impl"] == "reference" and line["unit"] == "GB/s" and line["higher_is_better"] is True
        assert line["value"] > 0 and line["gpu_launches"] == 0 and line["vs_baseline"] is None
        assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
        assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        assert line["config"]["workload"] == name
        # the config object is the one our arm prints for the same workload and N (driver: same_config)
        assert line["config"] == bench.workload_config(name, 1)
        assert set(line["config"]) >= {"workload", "baseline_config", "embedding", "m_total", "m_per_gpu", "n", "k",
                                        "partition", "scaling", "l2"}
    # ranks other than 0 print nothing
    monkeypatch.setenv("RANK", "1")
    bench.run_reference(bench.parse())
    assert capsys.readouterr().out == ""


def test_dump_outputs_option_and_sample(monkeypatch):
    import numpy as np
    import torch
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    assert bench.parse().dump_outputs is None
    monkeypatch.setattr(sys, "argv", ["bench.py", "--dump-outputs", "d", "--steps", "2"])
    args = bench.parse()
    assert args.dump_outputs == "d" and args.steps == 2
    small = torch.randn(512, 2000, dtype=torch.float64)                 # gauss_c2: 8 MB, kept whole
    assert np.array_equal(bench.dump_sample(small), small.numpy())
    big = torch.randn(1024, 4000, dtype=torch.float64)                  # srht_c3: 33 MB, a fixed sample of rows
    a = bench.dump_sample(big)
    assert a.dtype == np.float64 and a.shape == (500, 4000) and 4 * a.nbytes <= 64e6
    rows = np.sort(np.random.RandomState(0).choice(1024, 500, replace=False))
    assert np.array_equal(a, big.numpy()[rows]) and rows[-1] >= 500    # the seeded rows, not the first 500


def test_reference_arm_lifts_the_thread_limit_torchrun_sets(monkeypatch):
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must still use every host core."""
    bench = _load_bench()
    monkeypatch.setenv("OMP_NUM_THREADS", "1")
    cores = bench.all_host_threads()
    assert cores == (os.cpu_count() or 1) and os.environ["OMP_NUM_THREADS"] == str(cores)
    if cores > 1:
        assert bench.blas_threads() > 1
