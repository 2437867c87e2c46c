"""bench.py contract pieces that can be checked without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=120):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          env=e, timeout=timeout, cwd=ROOT)


def test_reference_arm_on_nonzero_rank_exits_silently():
    """Under torchrun (N > 1) rank 0 alone runs the CPU reference arm; the other ranks exit 0 without work."""
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0
    assert r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: the b200 arm refuses to run without a CUDA device instead of measuring something else."""
    r = _run(["--steps", "1", "--warmup", "1", "--skip-cpu-baseline", "--skip-e2e"])
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)


def test_algorithmic_bytes_formula_matches_survey_8d():
    """SURVEY.md §8(d): B = sum_l E_l (8 + 4 D) + 4 V H + 4 sum(weights) + 4 L V  ->  cfg2 = 21.68 GB per layer."""
    sys.path.insert(0, ROOT)
    import bench
    wl = bench.WORKLOADS["cfg2"]
    V, H, E = wl["V"], wl["H"], wl["E"]
    L, M = len(E), sum(E)
    cls_params = {"normalize_by_num_incoming": True}
    got = bench.algorithmic_bytes("rgcn", V, E, H, H, cls_params)
    expect = M * (8 + 4 * H) + 4 * V * H + 4 * L * H * H + 4 * L * V
    assert got == expect
    assert abs(got - 21.68e9) < 0.01e9
    line_keys = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                 "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"}
    with open(os.path.join(ROOT, "profiles", "bench_r1_final_full.json")) as f:
        line = json.load(f)
    assert line_keys <= set(line)
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])


def test_traffic_is_labelled_static_with_its_source():
    """roofline.traffic is never measured inside the timed run (ncu replays kernels): it is a static figure with the ncu
    capture it came from, or None with the reason."""
    sys.path.insert(0, ROOT)
    import bench
    val, src = bench.load_traffic("cfg2", "auto")
    assert (val is None) or (isinstance(val, int) and val > 1e9)
    assert isinstance(src, str) and ("static" in src or "no ncu" in src)
    val2, src2 = bench.load_traffic("no_such_workload", "auto")
    assert val2 is None and "no ncu" in src2


def test_bench_names_a_kernel_per_workload_kind():
    sys.path.insert(0, ROOT)
    import bench
    kinds = {w["kind"] for w in bench.WORKLOADS.values()}
    assert kinds <= set(bench.KERNEL_OF)
    assert bench.WORKLOADS["cfg5"]["V"] == 16_000_000 and sum(bench.WORKLOADS["cfg5"]["E"]) > 255_000_000


def test_dumped_rows_are_fixed_and_fit_the_limit():
    """--dump-outputs: the same rows in every run, all rows of a small output, and a default run (cfg2 + h320 + cfg1) within
    the size limit."""
    sys.path.insert(0, ROOT)
    import bench
    rows = bench.dump_rows(1_000_000, 256)
    assert np.array_equal(rows, bench.dump_rows(1_000_000, 256))
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < 1_000_000
    assert rows.size * 256 * 4 == bench.DUMP_ARRAY_BYTES
    assert np.array_equal(bench.dump_rows(8000, 320), np.arange(8000))
    total = sum(bench.dump_rows(w["V"], w["H"]).size * w["H"] * 4
                for w in (bench.WORKLOADS[n] for n in ("cfg2", "h320", "cfg1")))
    assert total <= bench.DUMP_TOTAL_BYTES


def test_dump_outputs_refuses_more_than_the_limit(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    with pytest.raises(SystemExit):
        bench.write_outputs(str(tmp_path / "d"), {"a": np.zeros(bench.DUMP_TOTAL_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "d").exists()
    bench.write_outputs(str(tmp_path / "d"), {"a": np.ones((3, 2), np.float32)})
    assert np.array_equal(np.load(tmp_path / "d" / "a.npy"), np.ones((3, 2), np.float32))


def test_dropout_stream_offsets_are_disjoint():
    from tf2_gnn_b200.layers.node_ops import DropoutState
    st = DropoutState(seed=3)
    a = st.take(10)        # 3 Philox counters (4 values each)
    b = st.take(1)
    c = st.take(8)
    assert (a, b, c) == (0, 3, 4) and st.offset == 6
