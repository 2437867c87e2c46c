"""bench.py on the device: --steps sets the number of timed layer calls, and --dump-outputs writes what the timed path
computed on the seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu


def _bench(steps, dump_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", str(steps),
                        "--warmup", "3", "--skip-cpu-baseline", "--no-clock-sampler", "--dump-outputs", str(dump_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_steps_and_dumped_outputs(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import bench
    from tf2_gnn_b200.layers import MessagePassingInput
    from tf2_gnn_b200.runtime import PreparedBatch
    one, three = _bench(1, tmp_path / "one"), _bench(3, tmp_path / "three")
    assert (one["steps"], three["steps"]) == (1, 3)
    assert (one["e2e"]["steps"], three["e2e"]["steps"]) == (1, 3)
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]
    assert sorted(os.listdir(tmp_path / "one")) == ["tiny.npy"]
    got = np.load(tmp_path / "one" / "tiny.npy")
    assert got.dtype == np.float32
    assert np.array_equal(got, np.load(tmp_path / "three" / "tiny.npy"))
    # the same layer call in this process, on the inputs bench.py generates
    wl = bench.WORKLOADS["tiny"]
    h, adjs, w = bench.make_inputs(wl, seed=0)
    layer, _ = bench.build_layer(wl, 0)
    layer.set_weights_from_oracle_dict({"edge_mlps": [[x] for x in w]})
    adj_dev = tuple(torch.from_numpy(a).cuda() for a in adjs)
    out = layer(MessagePassingInput(torch.from_numpy(h).cuda(), adj_dev), prepared=PreparedBatch(adj_dev, wl["V"]))
    rows = bench.dump_rows(wl["V"], wl["H"])
    assert np.array_equal(got, out.cpu().numpy()[rows])
