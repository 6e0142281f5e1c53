"""bench.py's contract pieces that do not need a GPU: the reference arm runs on the host cores and prints the same
`config` object as the b200 arm would (the driver compares them), for every --config."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line_and_shared_config():
    sys.path.insert(0, ROOT)
    import bench

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "evals/s" and line["higher_is_better"]
    assert line["e2e"] == {"value": line["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1

    class A:
        pass

    for cfg, c in bench.CONFIGS.items():
        a = A()
        a.config, a.batch, a.channels, a.blocks, a.batches_per_step, a.slots = cfg, c["batch"], c["channels"], c["blocks"], c["batches_per_step"], 4
        conf = bench.make_config(a)
        assert conf["batch"] == c["batch"] and conf["batches_per_step"] == c["batches_per_step"] and "workload" in conf
        if cfg == 2:
            assert conf == line["config"]          # the two arms of one --config print the same object
            assert line["metric"] == bench.metric_name(256) == "nn_leaf_evals_per_sec_batch256"


@pytest.mark.gpu
def test_dump_outputs_are_reproducible_and_hold_the_last_timed_batches(nb, synth, tmp_path):
    """--dump-outputs: two runs with the same arguments write the same results of the last timed step, bit for bit, all
    float32; and they are the results of the last timed batches themselves: every dumped batch is evaluated again here
    from bench.Workload's inputs (the same seeds) through nsb_eval_decode_async and must agree."""
    K, W, bps = 2, 3, 6
    args = ["--steps", str(K), "--warmup", str(W), "--batches-per-step", str(bps), "--no-cpu-baseline", "--no-selfplay",
            "--no-latency-leg"]
    got = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == K and line["warmup"] == W and line["gpu_launches"] == K * bps
        got.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("legal_probs", "win", "draw", "nan_flag")})
    a, b = got
    assert all(x.dtype == np.float32 for x in a.values())
    for n in a:
        assert np.array_equal(a[n].view(np.uint32), b[n].view(np.uint32)), n

    sys.path.insert(0, ROOT)
    import bench

    c = bench.CONFIGS[2]
    B = c["batch"]
    assert line["config"]["batch"] == B and a["win"].shape == a["draw"].shape == a["nan_flag"].shape == (bps, B)
    desc = nb.net_desc(c["channels"], c["blocks"])
    with nb.Context(desc, batch_max=B, slots=4, blob=nb.random_blob(desc, c["seed"])) as ctx:
        wl = bench.Workload(nb, synth, ctx, B, 0)
        assert a["legal_probs"].shape == (bps, wl.n_moves)
        end = (W + K) * bps                    # launches of the warm-up and the timed steps, the dump holds the last bps
        for k, i in enumerate(range(end - bps, end)):
            legal = np.zeros(wl.n_moves, dtype=np.float32)
            win, draw, flag = np.zeros(B, dtype=np.float32), np.zeros(B, dtype=np.float32), np.zeros(B, dtype=np.uint8)
            ctx.eval_decode_async(0, np.ascontiguousarray(wl.host_pool[i % wl.pool]), B, wl.off, wl.idx, nb.DECODE_PROBS,
                                  legal, win, draw, flag)
            ctx.await_(0)
            assert np.allclose(a["legal_probs"][k], legal, rtol=1e-5, atol=1e-6), k
            assert np.allclose(a["win"][k], win, rtol=1e-5, atol=1e-6) and np.allclose(a["draw"][k], draw, rtol=1e-5, atol=1e-6), k
            assert np.array_equal(a["nan_flag"][k], flag.astype(np.float32)), k
        wl.free()
    sums = np.add.reduceat(a["legal_probs"].astype(np.float64), wl.off[:-1].astype(np.int64), axis=1)
    assert np.allclose(sums, 1.0, atol=1e-4) and not a["nan_flag"].any()
