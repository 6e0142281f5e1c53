"""192-channel nets: the width runs on the CTA-pair trunk (trunk_pair_kernel<192>), whose Cout halves of 96 channels
are padded to the 128 rows of the MMA while the K side stays exact (3 blocks of 64).

The reference for the kernel is the unchanged 256-channel kernel on the same net zero-padded to 256 channels
(weights_io.pad_channels): every output element accumulates the same K sequence there, the padded kernel only adds
exact zeros from its fourth K block, so the two agree bit for bit.  Around that: the depth tolerances of
test_depth_parity.py against the oracle, batch invariance at the benchmark's shape, the paths that touch the
kernel's work list and I/O, and a trained-looking net through the ONNX loaders."""
import ctypes
import json
import os
import subprocess
import warnings

import numpy as np
import pytest

import helpers
import test_depth_parity as depth
import test_evalcache
import test_gpu_parity as parity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "nshogi-engine_b200", "host")

# weight seeds whose value head is alive at 192 channels (win spread of the fp32 oracle > 0.1 on the positions below)
SEED_10x192 = 3
SEED_20x192 = 3


def _u32(a):
    return a.view(np.uint32)


def _eval(nb, ctx, fb, n, slot=0):
    policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
    win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    ctx.eval_async(slot, fb, n, policy, win, draw)
    ctx.await_(slot)
    return policy, win, draw


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_create_accepts_192_and_rejects_other_widths(nb):
    l = nb.lib()
    h = ctypes.c_void_p()
    for bad in (64, 96, 160, 320):
        desc = nb.net_desc(bad, 1)
        assert l.nsb_create(ctypes.byref(h), 0, 8, 1, ctypes.byref(desc)) == -1, bad
        assert b"128|192|256" in l.nsb_last_error()
    desc = nb.net_desc(192, 1)
    rc = l.nsb_create(ctypes.byref(h), 0, 8, 1, ctypes.byref(desc))
    if nb.device_count() > 0:
        assert rc == 0, l.nsb_last_error()
        l.nsb_destroy(h)
    else:
        assert rc == -3 and b"no CPU fallback" in l.nsb_last_error()


@pytest.mark.parametrize("narrow,wide", [(192, 256), (128, 192)])
def test_pad_channels_keeps_the_function(pkg, nb, orc, synth, narrow, wide):
    """The padded blob has the wider net's size and computes the same outputs through the oracle (fp32 and
    bf16-emulating): the added channels are zero in every layer."""
    wio = pkg.weights_io
    desc, wdesc = nb.net_desc(narrow, 2), nb.net_desc(wide, 2)
    blob = nb.random_blob(desc, 5)
    padded = wio.pad_channels(blob, desc, wide)
    assert padded.dtype == np.float32 and padded.size == nb.random_blob(wdesc, 5).size
    w = helpers.split_blob(wdesc, padded)
    assert not w["stem_w"][narrow:].any() and not w["blocks"][0][0][:, narrow:].any() and not w["pol_w"][:, narrow:].any()
    n = 6
    planes = orc.expand(orc.pack(synth.random_positions(n, seed=4)), n)
    for bf16 in (False, True):
        a = orc.forward(desc, blob, planes, emulate_bf16=bf16)
        b = orc.forward(wdesc, padded, planes, emulate_bf16=bf16)
        for x, y in zip(a, b):
            assert np.array_equal(_u32(x), _u32(y)), bf16
    with pytest.raises(ValueError):
        wio.pad_channels(padded, wdesc, narrow)


# ---- GPU: the kernel ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 5, 64, 512])
def test_bit_exact_against_padded_256_kernel(pkg, nb, orc, synth, monkeypatch, n):
    monkeypatch.delenv("NSB_TRUNK256", raising=False)
    desc, wdesc = nb.net_desc(192, 10), nb.net_desc(256, 10)
    blob = nb.random_blob(desc, SEED_10x192)
    padded = pkg.weights_io.pad_channels(blob, desc, 256)
    fb = orc.pack(synth.random_positions(n, seed=100 + n))
    with nb.Context(desc, batch_max=n, blob=blob) as ctx:
        assert ctx.trunk_kernel_name().startswith("trunk_pair_kernel (192 ch")
        got = _eval(nb, ctx, fb, n)
    with nb.Context(wdesc, batch_max=n, blob=padded) as ctx:
        assert ctx.trunk_kernel_name().startswith("trunk_pair_kernel (256 ch")
        want = _eval(nb, ctx, fb, n)
    for g, w in zip(got, want):
        assert np.array_equal(_u32(g), _u32(w))
    assert np.all(np.isfinite(got[0])) and got[1].min() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("blocks,seed,n,slots", [(10, SEED_10x192, 5, 1), (10, SEED_10x192, 64, 2), (20, SEED_20x192, 64, 3)])
def test_depth_parity_vs_oracle_192(nb, orc, synth, monkeypatch, blocks, seed, n, slots):
    """test_depth_parity.py's metrics and tolerances (helpers.drift_metrics) at 192 channels."""
    monkeypatch.delenv("NSB_TRUNK256", raising=False)
    desc = nb.net_desc(192, blocks)
    blob = nb.random_blob(desc, seed)
    pos = synth.random_positions(n, seed=2024)
    fb = orc.pack(pos)
    off, idx = synth.random_legal_moves(n, seed=3, edge_rows=False)
    legal = np.zeros(int(off[-1]), dtype=np.float32)
    w2, d2 = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
        assert ctx.trunk_kernel_name().startswith("trunk_pair_kernel (192 ch")
        policy, win, draw = _eval(nb, ctx, fb, n)
        ctx.eval_positions_decode_async(slots - 1, pos, n, off, idx, nb.DECODE_PROBS, legal, w2, d2, None)
        ctx.await_(slots - 1)
    m = helpers.drift_metrics(nb, orc, desc, blob, fb, n, (policy, win, draw), off, idx)
    assert m["win_spread_fp32"] > 1e-2, ("dead value head: pick another seed", m)
    depth._check(m, f"{blocks}x192@{n}")
    want, _ = orc.decode(policy, win, draw, off, idx, nb.DECODE_PROBS)
    assert np.allclose(legal, want, rtol=1e-6, atol=1e-9) and np.array_equal(w2, win) and np.array_equal(d2, draw)


@pytest.mark.gpu
def test_batch_invariance_at_bench_shape(nb, orc, synth, monkeypatch):
    """B = 512 on a 4-slot context (the benchmark's shape, 20 x 192): every row equals, bit for bit, the same position
    evaluated alone in a batch of one - whichever pair, pass and CTA rank computed it."""
    monkeypatch.delenv("NSB_TRUNK256", raising=False)
    desc = nb.net_desc(192, 20)
    blob = nb.random_blob(desc, SEED_20x192)
    base, batch = 24, 512
    fb = orc.pack(synth.random_positions(base, seed=2024)).reshape(base, 86)
    perm = np.random.default_rng(1).integers(0, base, size=batch)
    perm[:base] = np.arange(base)
    big = np.ascontiguousarray(fb[perm].reshape(-1))
    with nb.Context(desc, batch_max=batch, slots=4, blob=blob) as ctx:
        p_big, w_big, d_big = _eval(nb, ctx, big, batch, slot=3)
        singles = [_eval(nb, ctx, np.ascontiguousarray(fb[i]), 1, slot=i % 4) for i in range(base)]
    p1 = np.concatenate([s[0] for s in singles])
    w1 = np.concatenate([s[1] for s in singles])
    d1 = np.concatenate([s[2] for s in singles])
    assert np.array_equal(_u32(p_big), _u32(p1[perm]))
    assert np.array_equal(w_big, w1[perm]) and np.array_equal(d_big, d1[perm])


# ---- GPU: the paths that touch the kernel's work list and I/O, as test_gpu_parity.py / test_evalcache.py run them --
@pytest.mark.gpu
def test_packed_positions_equal_bitboards_192(nb, orc, synth, monkeypatch):
    parity.test_stage1_fused_into_trunk_prologue(nb, orc, synth, monkeypatch, 192, 1)


@pytest.mark.gpu
def test_direct_io_equals_staged_192(nb, orc, synth, monkeypatch):
    parity.test_direct_io_equals_staged(nb, orc, synth, monkeypatch, 192, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("direct", [False, True])
def test_cached_path_192(nb, orc, synth, direct):
    test_evalcache.test_eval_cached_serves_hits_and_evaluates_misses(nb, orc, synth, 192, direct)


@pytest.mark.gpu
def test_rank_order_of_decoded_rows_192(nb, orc, synth, monkeypatch):
    parity.test_rank_order_of_decoded_rows(nb, orc, synth, monkeypatch, 192, 1)


@pytest.mark.gpu
def test_custom_features_v1_93_channels_192(nb, orc, synth, monkeypatch):
    parity.test_custom_features_v1_93_channels(nb, orc, synth, monkeypatch, 192, 1)


# ---- GPU: a trained-looking net through both ONNX loaders --------------------------------------------------------
@pytest.mark.gpu
def test_ten_block_batchnorm_192_net_through_onnx_load(nb, orc, synth, tmp_path):
    """10 x 192 with batch-norm -> torch.onnx.export -> onnx_import.h (nsb_host_unit --onnx-blob) -> the executor,
    against the PyTorch model's fp32 forward; then the same file through infer::B200::load (nsb_host_bench)."""
    import torch
    from torch.onnx._internal.torchscript_exporter import onnx_proto_utils

    C, blocks, n = 192, 10, 64
    net = depth._trained_like_net(C, blocks, seed=3)
    onnx_path = str(tmp_path / "net10x192.onnx")

    class Wrap(torch.nn.Module):
        def __init__(self, inner):
            super().__init__()
            self.inner = inner

        def forward(self, x):
            p, w, d = self.inner(x)
            return p, w.reshape(-1, 1), d.reshape(-1, 1)

    onnx_proto_utils._add_onnxscript_fn = lambda proto, custom_opsets: proto   # needs the absent `onnx` package
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        torch.onnx.export(Wrap(net).eval(), (torch.zeros(2, 86, 9, 9),), onnx_path, dynamo=False, input_names=["input"],
                          output_names=["policy", "value", "draw"], opset_version=17,
                          dynamic_axes={"input": {0: "batch"}, "policy": {0: "batch"}, "value": {0: "batch"}, "draw": {0: "batch"}})
    subprocess.check_call(["make", "-C", HOST, "-s", "all"])
    raw = str(tmp_path / "net10x192.blob")
    out = subprocess.run([os.path.join(HOST, "nsb_host_unit"), "--onnx-blob", onnx_path, raw], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.startswith("ok 86 192 10 256"), out.stdout + out.stderr
    blob = np.fromfile(raw, dtype=np.float32, offset=16)
    desc = nb.net_desc(C, blocks)
    fb = orc.pack(synth.random_positions(n, seed=77))
    planes = orc.expand(fb, n)
    with torch.no_grad():
        tp, tw, td = (t.numpy() for t in net(torch.from_numpy(planes).reshape(-1, 86, 9, 9)))
    assert np.ptp(tw) > 1e-2, "dead value head: pick another seed"
    with nb.Context(desc, batch_max=n, slots=2, blob=blob) as ctx:
        policy, win, draw = _eval(nb, ctx, fb, n)
    off, idx = synth.random_legal_moves(n, seed=2, edge_rows=False)
    pg, _ = orc.decode(policy, win, draw, off, idx, nb.DECODE_PROBS)
    pt, _ = orc.decode(tp, tw, td, off, idx, nb.DECODE_PROBS)
    m = {"layers": 22, "n": n, "prob_vs_fp32": float(np.max(np.abs(pg - pt))), "win_vs_fp32": float(np.max(np.abs(win - tw))),
         "draw_vs_fp32": float(np.max(np.abs(draw - td))), "logit_vs_fp32": float(np.max(np.abs(policy - tp))),
         "logit_rms_fp32": float(np.sqrt(np.mean(tp.astype(np.float64) ** 2))), "win_spread_fp32": float(np.ptp(tw)),
         "reference": "PyTorch fp32 forward of the batch-norm model (weights NOT bf16-exact: includes weight rounding)"}
    depth._record("10x192-batchnorm-onnx@64", m)
    assert m["prob_vs_fp32"] <= depth.TOL_PROB_VS_FP32, m
    assert m["win_vs_fp32"] <= depth.TOL_VALUE_VS_FP32 and m["draw_vs_fp32"] <= depth.TOL_VALUE_VS_FP32, m
    out = subprocess.run([os.path.join(HOST, "nsb_host_bench"), "--selfcheck", "--repeat", "10", "--batch", "64", "--weights", onnx_path],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["ok"] and line["net"] == "10x192"
