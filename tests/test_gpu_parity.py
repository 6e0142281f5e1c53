"""GPU suite (-m gpu): parity of the CUDA path, called through the C ABI, against the CPU oracle,
the committed golden vectors and the reference's own extractbit.cu compiled in place."""
import os

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu

# Tolerances (stated here, justified in DESIGN.md §7):
TOL_LOGIT_VS_BF16_ORACLE = 1e-2   # same bf16 rounding points; fp32 accumulation order differs, so a
                                  # value on a rounding boundary can flip by one bf16 ulp (2^-8 relative)
TOL_VALUE_VS_BF16_ORACLE = 2e-3
TOL_PROB_VS_FP32 = 2e-2           # SURVEY.md §8c: policy probabilities max-abs-diff, bf16 in / fp32 acc
TOL_VALUE_VS_FP32 = 1e-2
TOL_DECODE_REL = 1e-6


@pytest.fixture(scope="module")
def ctx128(nb):
    desc = nb.net_desc(128, 2)
    blob = nb.random_blob(desc, 1234)
    c = nb.Context(desc, batch_max=512, slots=2, blob=blob)
    yield c, desc, blob
    c.close()


def run_eval(nb, ctx, fb, n, slot=0):
    policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
    win = np.zeros(n, dtype=np.float32)
    draw = np.zeros(n, dtype=np.float32)
    ctx.eval_async(slot, fb, n, policy, win, draw)
    ctx.await_(slot)
    return policy, win, draw


# ---- tcgen05 building block -----------------------------------------------------------------------------------
@pytest.mark.parametrize("n_cols,k,shift", [(192, 64, 0), (192, 64, 11), (96, 128, 1), (192, 128, 22), (96, 16, 5)])
def test_umma_descriptor_and_epilogue_selftest(nb, n_cols, k, shift):
    assert nb.umma_selftest(n_cols, k, shift) == (0.0, 0.0)


# ---- stage 2: extract == reference extractBits<> ----------------------------------------------------------------
@pytest.mark.parametrize("n,channels", [(1, 86), (3, 86), (256, 86), (37, 93), (5, 1), (4096, 86)])
@pytest.mark.parametrize("channels_first", [True, False])
def test_extract_bit_exact(nb, orc, synth, ctx128, n, channels, channels_first):
    ctx = ctx128[0]
    fb = synth.random_feature_bitboards(n * channels, seed=n + channels)
    d_fb = nb.DeviceBuffer.from_host(fb)
    d_out = nb.DeviceBuffer(n * channels * 81 * 4)
    d_out.fill(0xFF)
    ctx.extract_device(0, d_fb.ptr, n, channels, channels_first, d_out.ptr)
    ctx.await_(0)
    shape = (n, channels, 81) if channels_first else (n, 81, channels)
    got = d_out.to_host(shape, np.uint32)
    want = orc.expand(fb, n, channels, channels_first).view(np.uint32)
    assert np.array_equal(got, want)
    if orc.have_ref_extract() and n <= 256:   # the reference's own kernels, compiled from /root/reference
        d_ref = nb.DeviceBuffer(n * channels * 81 * 4)
        d_ref.fill(0xFF)
        assert orc.ref_extract_device(d_ref.ptr, d_fb.ptr, n, channels, channels_first) == 0
        assert np.array_equal(d_ref.to_host(shape, np.uint32), want)
        d_ref.free()
    d_fb.free()
    d_out.free()


def test_extract_golden_and_empty(nb, ctx128, golden_dir):
    ctx = ctx128[0]
    g = np.load(os.path.join(golden_dir, "expand_kat.npz"))
    fb = np.zeros(96, dtype=nb.FEATURE_BITBOARD)
    fb["lo"], fb["hi"] = g["lo"], g["hi"]
    d_fb = nb.DeviceBuffer.from_host(fb)
    d_out = nb.DeviceBuffer(96 * 81 * 4)
    for cf, key, shape in ((True, "nchw", (2, 48, 81)), (False, "nhwc", (2, 81, 48))):
        ctx.extract_device(0, d_fb.ptr, 2, 48, cf, d_out.ptr)
        ctx.await_(0)
        assert np.array_equal(d_out.to_host(shape, np.uint32), g[key])
    ctx.extract_device(0, d_fb.ptr, 0, 86, True, d_out.ptr)  # empty batch is a no-op
    ctx.await_(0)
    d_fb.free()
    d_out.free()


# ---- stage 1: pack ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 5, 256, 1000])
def test_pack_bit_exact(nb, orc, synth, ctx128, n):
    ctx = ctx128[0]
    pos = synth.random_positions(n, seed=n)
    d_pos = nb.DeviceBuffer.from_host(pos)
    d_fb = nb.DeviceBuffer(n * 86 * 16)
    ctx.pack_positions_device(0, d_pos.ptr, n, d_fb.ptr)
    ctx.await_(0)
    got = d_fb.to_host((n * 86,), nb.FEATURE_BITBOARD)
    want = orc.pack(pos)
    assert np.array_equal(got["lo"], want["lo"]) and np.array_equal(got["hi"], want["hi"])
    d_pos.free()
    d_fb.free()


# ---- decode ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 64, 1000])
@pytest.mark.parametrize("kind", [0, 1, 2])
@pytest.mark.parametrize("fallback", [False, True])
def test_decode_matches_oracle(nb, orc, synth, ctx128, n, kind, fallback):
    """Standalone decode kernel vs the oracle for every mode (PROBS = feedworker.cc:100-136, LOGITS / BOTH =
    frame.cc:93-118), with and without the NaN fallback (feedResult<true> / the reference's default <false>), Gumbel
    root rows (softmax skipped) and raw logits beside the probabilities.  synth.random_logits plants an all-NaN
    logit row (5), a partly-NaN one (6), -inf logits (7), a NaN win rate (8) and a NaN draw rate (9)."""
    ctx = ctx128[0]
    mode = kind | (nb.DECODE_NAN_FALLBACK if fallback else 0)
    policy, win, draw = synth.random_logits(n, seed=n)
    off, idx = synth.random_legal_moves(n, seed=n)
    rf = (np.arange(n) % 5 == 2).astype(np.uint8) * nb.ROW_SKIP_SOFTMAX
    total = int(off[-1])
    d = [nb.DeviceBuffer.from_host(a) for a in (policy, win, draw, off, idx, rf)]
    d_out, d_log, d_flag = nb.DeviceBuffer(max(total, 1) * 4), nb.DeviceBuffer(max(total, 1) * 4), nb.DeviceBuffer(n)
    d_log.fill(0)
    ctx.decode_device_ex(0, d[0].ptr, d[1].ptr, d[2].ptr, n, d[3].ptr, d[4].ptr, mode, d[5].ptr, d_out.ptr, d_log.ptr, d_flag.ptr)
    ctx.await_(0)
    got, got_log, flag = d_out.to_host((total,), np.float32), d_log.to_host((total,), np.float32), d_flag.to_host((n,), np.uint8)
    want, want_log, wflag = orc.decode_ex(policy, win, draw, off, idx, mode, row_flags=rf, want_logits=True)
    assert np.array_equal(flag, wflag)
    if n >= 64:
        assert list(np.nonzero(flag)[0]) == ([5, 6, 8, 9] if fallback else [])
    if kind == nb.DECODE_LOGITS:
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    else:
        assert np.array_equal(np.isnan(got), np.isnan(want))          # NaN rows: the same rows, whatever the payload
        assert np.allclose(got, want, rtol=TOL_DECODE_REL, atol=1e-9, equal_nan=True)
        if kind == nb.DECODE_BOTH:
            assert np.array_equal(got_log.view(np.uint32), want_log.view(np.uint32))
            for i in np.nonzero(rf)[0]:                                # Gumbel root: the raw logits, bit for bit
                assert np.array_equal(got[off[i]:off[i + 1]].view(np.uint32), want_log[off[i]:off[i + 1]].view(np.uint32))
    for b_ in d + [d_out, d_log, d_flag]:
        b_.free()


# ---- forward ----------------------------------------------------------------------------------------------------
def test_forward_golden_small_net(nb, orc, golden_dir):
    g = np.load(os.path.join(golden_dir, "forward_small.npz"))
    desc = nb.net_desc(128, 1)
    blob = nb.random_blob(desc, int(g["blob_seed"]))
    pos = np.frombuffer(g["positions"].tobytes(), dtype=nb.POSITION)
    n = len(pos)
    policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
    win = np.zeros(n, dtype=np.float32)
    draw = np.zeros(n, dtype=np.float32)
    with nb.Context(desc, batch_max=4, blob=blob) as ctx:
        ctx.eval_positions_async(0, pos, n, policy, win, draw)
        ctx.await_(0)
    assert np.max(np.abs(policy - g["policy_bf16"])) < TOL_LOGIT_VS_BF16_ORACLE
    assert np.max(np.abs(win - g["win_bf16"])) < TOL_VALUE_VS_BF16_ORACLE
    assert np.max(np.abs(draw - g["draw_bf16"])) < TOL_VALUE_VS_BF16_ORACLE
    assert np.max(np.abs(win - g["win_fp32"])) < TOL_VALUE_VS_FP32


@pytest.mark.parametrize("n", [1, 2, 3, 37])
def test_forward_matches_oracle_128(nb, orc, synth, ctx128, n):
    ctx, desc, blob = ctx128
    pos = synth.random_positions(n, seed=100 + n)
    fb = orc.pack(pos)
    policy, win, draw = run_eval(nb, ctx, fb, n)
    planes = orc.expand(fb, n)
    op, ow, od = orc.forward(desc, blob, planes, emulate_bf16=True)
    assert np.max(np.abs(policy - op)) < TOL_LOGIT_VS_BF16_ORACLE
    assert np.max(np.abs(win - ow)) < TOL_VALUE_VS_BF16_ORACLE and np.max(np.abs(draw - od)) < TOL_VALUE_VS_BF16_ORACLE
    fp, fw, fd = orc.forward(desc, blob, planes, emulate_bf16=False)
    off, idx = synth.random_legal_moves(n, seed=n, edge_rows=False)
    pg, _ = orc.decode(policy, win, draw, off, idx, nb.DECODE_PROBS)
    pf, _ = orc.decode(fp, fw, fd, off, idx, nb.DECODE_PROBS)
    assert np.max(np.abs(pg - pf)) < TOL_PROB_VS_FP32
    assert np.max(np.abs(win - fw)) < TOL_VALUE_VS_FP32 and np.max(np.abs(draw - fd)) < TOL_VALUE_VS_FP32


def test_forward_fuzzed_feature_values(nb, orc, synth, ctx128):
    """Arbitrary FeatureBitboards (random masks, rotate, fractional values, garbage bits): the
    in-kernel expansion must follow extractbit.cu for any input, not just packed positions."""
    ctx, desc, blob = ctx128
    n = 9
    fb = synth.random_feature_bitboards(n * 86, seed=77)
    policy, win, draw = run_eval(nb, ctx, fb, n)
    op, ow, od = orc.forward(desc, blob, orc.expand(fb, n), emulate_bf16=True)
    assert np.max(np.abs(policy - op)) < 4 * TOL_LOGIT_VS_BF16_ORACLE  # denser inputs, larger activations
    assert np.max(np.abs(win - ow)) < 4 * TOL_VALUE_VS_BF16_ORACLE


@pytest.mark.parametrize("n", [1, 2, 5])
def test_forward_matches_oracle_256(nb, orc, synth, n):
    """256 channels run on the CTA-pair kernel (cta_group::2 MMAs, DSMEM exchange of half of every
    layer's output and of the skip rows); n = 1 and 5 leave the second CTA of the last pair without
    a position."""
    desc = nb.net_desc(256, 2)
    blob = nb.random_blob(desc, 99)
    pos = synth.random_positions(n, seed=256)
    fb = orc.pack(pos)
    with nb.Context(desc, batch_max=8, blob=blob) as ctx:
        policy, win, draw = run_eval(nb, ctx, fb, n)
    op, ow, od = orc.forward(desc, blob, orc.expand(fb, n), emulate_bf16=True)
    assert np.max(np.abs(policy - op)) < TOL_LOGIT_VS_BF16_ORACLE
    assert np.max(np.abs(win - ow)) < TOL_VALUE_VS_BF16_ORACLE and np.max(np.abs(draw - od)) < TOL_VALUE_VS_BF16_ORACLE


def test_pair_kernel_equals_single_cta_kernel(nb, orc, synth, monkeypatch):
    """The CTA-pair kernel accumulates every output element in the same K order as the one-CTA
    kernel, so the two must agree bit for bit - at a size where the pairs run several passes
    (513 positions -> 257 groups over 74 pairs) and with the fused decode on."""
    desc = nb.net_desc(256, 3)
    blob = nb.random_blob(desc, 7)
    n, base = 513, 24
    pos = synth.random_positions(base, seed=11)
    fb = orc.pack(pos).reshape(base, 86)
    perm = np.random.default_rng(2).integers(0, base, size=n)
    perm[:base] = np.arange(base)
    big = np.ascontiguousarray(fb[perm].reshape(-1))
    off, idx = synth.random_legal_moves(n, seed=5, edge_rows=False)

    def run(single):
        if single:
            monkeypatch.setenv("NSB_TRUNK256", "single")
        else:
            monkeypatch.delenv("NSB_TRUNK256", raising=False)
        policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
        win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
        legal = np.zeros(int(off[-1]), dtype=np.float32)
        flag = np.zeros(n, dtype=np.uint8)
        with nb.Context(desc, batch_max=n, blob=blob, diag=single) as ctx:   # the one-CTA kernel: libnsb_diag.so
            ctx.eval_async(0, big, n, policy, win, draw)
            ctx.await_(0)
            ctx.eval_decode_async(0, big, n, off, idx, nb.DECODE_PROBS, legal, win, draw, flag)
            ctx.await_(0)
        return policy, win, draw, legal

    p1, w1, d1, l1 = run(single=True)
    p2, w2, d2, l2 = run(single=False)
    assert np.array_equal(p1.view(np.uint32), p2.view(np.uint32))
    assert np.array_equal(w1, w2) and np.array_equal(d1, d2) and np.array_equal(l1.view(np.uint32), l2.view(np.uint32))
    # batch-index invariance across pairs / passes / CTA rank
    assert np.array_equal(p2.view(np.uint32), p2[:base][perm].view(np.uint32))


def test_fused_decode_equals_separate_decode(nb, orc, synth, ctx128):
    """(c): gather + softmax fused into the trunk epilogue == decode of the same launch's logits."""
    ctx, desc, blob = ctx128
    n = 45
    pos = synth.random_positions(n, seed=5)
    fb = orc.pack(pos)
    off, idx = synth.random_legal_moves(n, seed=5)
    policy, win, draw = run_eval(nb, ctx, fb, n)
    for mode in (nb.DECODE_PROBS, nb.DECODE_LOGITS):
        legal = np.zeros(int(off[-1]), dtype=np.float32)
        w2 = np.zeros(n, dtype=np.float32)
        d2 = np.zeros(n, dtype=np.float32)
        flag = np.ones(n, dtype=np.uint8)
        ctx.eval_decode_async(1, fb, n, off, idx, mode, legal, w2, d2, flag)
        ctx.await_(1)
        want, wflag = orc.decode(policy, win, draw, off, idx, mode)
        assert np.array_equal(w2, win) and np.array_equal(d2, draw) and np.array_equal(flag, wflag)
        if mode == nb.DECODE_LOGITS:
            assert np.array_equal(legal.view(np.uint32), want.view(np.uint32))
        else:
            assert np.allclose(legal, want, rtol=TOL_DECODE_REL, atol=1e-9)
    # positions-in variant (stage 1 on device too)
    legal2 = np.zeros(int(off[-1]), dtype=np.float32)
    ctx.eval_positions_decode_async(0, pos, n, off, idx, nb.DECODE_LOGITS, legal2, w2, d2, flag)
    ctx.await_(0)
    assert np.array_equal(legal2.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("batch,kernel", [(256, "classic"), (4096, "classic"), (256, "duo"), (4096, "duo"), (4096, None)])
def test_full_size_batch_invariance(nb, orc, synth, monkeypatch, batch, kernel):
    """BASELINE sizes: every position's result is independent of its batch index, of the batch
    size and of which CTA / accumulator column evaluates it (bit-exact), and equals the oracle on
    the distinct positions.  10 x 128 net == config 2.  Bit-exactness holds per trunk kernel; a one-slot context
    left to itself (kernel None) switches from trunk_fused.cu to trunk_duo_kernel with the batch size, and the two
    differ by float rounding (another K order), so that case is held to the oracle tolerance instead."""
    if kernel:
        monkeypatch.setenv("NSB_TRUNK128", kernel)
    else:
        monkeypatch.delenv("NSB_TRUNK128", raising=False)
    desc = nb.net_desc(128, 10)
    blob = nb.random_blob(desc, 1234)
    base = 16
    pos = synth.random_positions(base, seed=2024)
    fb = orc.pack(pos).reshape(base, 86)
    rng = np.random.default_rng(1)
    perm = rng.integers(0, base, size=batch)
    perm[:base] = np.arange(base)
    big = np.ascontiguousarray(fb[perm].reshape(-1))
    with nb.Context(desc, batch_max=batch, blob=blob) as ctx:
        p_small, w_small, d_small = run_eval(nb, ctx, np.ascontiguousarray(fb.reshape(-1)), base)
        p_big, w_big, d_big = run_eval(nb, ctx, big, batch)
    if kernel:
        assert np.array_equal(p_big.view(np.uint32), p_small[perm].view(np.uint32))
        assert np.array_equal(w_big, w_small[perm]) and np.array_equal(d_big, d_small[perm])
    else:  # 16 positions ran on trunk_fused.cu, 4,096 on trunk_duo_kernel
        assert np.array_equal(p_big[base:].view(np.uint32), p_big[perm[base:]].view(np.uint32))   # invariance inside the batch
        assert np.max(np.abs(p_big - p_small[perm])) < 2 * TOL_LOGIT_VS_BF16_ORACLE
        assert np.max(np.abs(w_big - w_small[perm])) < 2 * TOL_VALUE_VS_BF16_ORACLE
    op, ow, od = orc.forward(desc, blob, orc.expand(fb.reshape(-1), base), emulate_bf16=True)
    assert np.max(np.abs(p_small - op)) < 3 * TOL_LOGIT_VS_BF16_ORACLE   # 21 layers deep
    assert np.max(np.abs(w_small - ow)) < 3 * TOL_VALUE_VS_BF16_ORACLE


# ---- the Infer contract ------------------------------------------------------------------------------------------
def test_infer_interface_contract(pkg, nb, orc, synth):
    """Reads like the reference's use of Infer/Evaluator (src/bench/batchsize.cc:47-70)."""
    B = 128
    desc = nb.net_desc(128, 2)
    blob = nb.random_blob(desc, 1234)
    infer = pkg.infer.B200(0, B, 86, desc, blob=blob)
    infer.resetGPU()
    ev = pkg.infer.Evaluator(B, infer)
    fb = orc.pack(synth.startpos(B))
    ev.getFeatureBitboards()[:] = fb
    assert not ev.isComputing()
    ev.computeNonBlocking(B)
    ev.await_()
    assert not ev.isComputing()
    first = ev.getPolicy().copy()
    ev.computeBlocking(B)
    assert np.array_equal(first, ev.getPolicy())
    pol = first.reshape(B, nb.POLICY_SIZE)
    assert np.array_equal(pol[0], pol[B - 1])          # startpos x B -> identical rows
    assert np.all((ev.getWinRate() > 0) & (ev.getWinRate() < 1)) and np.all((ev.getDrawRate() > 0) & (ev.getDrawRate() < 1))
    op, ow, od = orc.forward(desc, blob, orc.expand(fb[:86], 1), emulate_bf16=True)
    assert np.max(np.abs(pol[0] - op[0])) < TOL_LOGIT_VS_BF16_ORACLE
    with pytest.raises(nb.NsbError):                   # BatchSize <= BatchSizeMax (trt.cc:237)
        infer.ctx.eval_async(0, fb, B + 1, ev.getPolicy(), ev.getWinRate(), ev.getDrawRate())
    ev.close()
    infer.close()


def test_errors_are_reported_not_swallowed(nb):
    desc = nb.net_desc(128, 1)
    with nb.Context(desc, batch_max=4) as ctx:           # no weights loaded
        z = np.zeros(4 * 86, dtype=nb.FEATURE_BITBOARD)
        with pytest.raises(nb.NsbError) as e:
            ctx.eval_async(0, z, 4, np.zeros((4, 2187), np.float32), np.zeros(4, np.float32), np.zeros(4, np.float32))
        assert "weights not loaded" in str(e.value)
        with pytest.raises(nb.NsbError):
            ctx.load_weights(np.zeros(10, dtype=np.float32))
        with pytest.raises(nb.NsbError):
            ctx.await_(3)


# ---- edge cases ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,channels", [(2, 2), (7, 64), (1, 128), (33, 31)])
def test_extract_other_channel_counts(nb, orc, synth, ctx128, n, channels):
    """extractBits<> is generic in the channel count (src/cuda/extractbit.cu:76-96): even counts take the
    8-byte NHWC path, odd ones the scalar path, and the NCHW blocks end in a ragged tail."""
    ctx = ctx128[0]
    fb = synth.random_feature_bitboards(n * channels, seed=1000 + channels)
    fb["hi"][::3] |= np.uint64(1 << 24)                    # plenty of rotated planes
    d_fb = nb.DeviceBuffer.from_host(fb)
    d_out = nb.DeviceBuffer(n * channels * 81 * 4)
    for cf in (True, False):
        d_out.fill(0xAB)
        ctx.extract_device(0, d_fb.ptr, n, channels, cf, d_out.ptr)
        ctx.await_(0)
        shape = (n, channels, 81) if cf else (n, 81, channels)
        assert np.array_equal(d_out.to_host(shape, np.uint32), orc.expand(fb, n, channels, cf).view(np.uint32))
    d_fb.free()
    d_out.free()


def test_empty_batch_and_empty_rows(nb, orc, synth, ctx128):
    """n = 0 is a no-op on every entry point; a position without legal moves (an empty CSR row) produces
    no output and does not disturb its neighbours."""
    ctx, desc, blob = ctx128
    z = np.zeros(1, dtype=np.float32)
    ctx.eval_async(0, np.zeros(1, dtype=nb.FEATURE_BITBOARD), 0, z, z, z)
    ctx.eval_decode_async(0, np.zeros(1, dtype=nb.FEATURE_BITBOARD), 0, np.zeros(1, dtype=np.uint32),
                          np.zeros(1, dtype=np.uint16), nb.DECODE_PROBS, z, z, z, None)
    ctx.await_(0)
    n = 6
    pos = synth.random_positions(n, seed=5)
    fb = orc.pack(pos)
    cnt = np.array([3, 0, 1, 0, 40, 2], dtype=np.uint32)
    off = np.zeros(n + 1, dtype=np.uint32)
    off[1:] = np.cumsum(cnt)
    idx = np.random.default_rng(1).choice(nb.POLICY_SIZE, size=int(off[-1]), replace=False).astype(np.uint16)
    legal = np.full(int(off[-1]), -7.0, dtype=np.float32)
    win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    flag = np.zeros(n, dtype=np.uint8)
    ctx.eval_decode_async(0, fb, n, off, idx, nb.DECODE_PROBS, legal, win, draw, flag)
    ctx.await_(0)
    policy, w2, d2 = run_eval(nb, ctx, fb, n)
    want, wflag = orc.decode(policy, w2, d2, off, idx, nb.DECODE_PROBS)
    assert np.allclose(legal, want, rtol=1e-5, atol=1e-7) and np.array_equal(flag, wflag)
    assert np.array_equal(win, w2) and legal[off[2]] == 1.0          # 1-move row (feedworker.cc:101-103)
    for i in range(n):
        if cnt[i] > 1:
            assert abs(legal[off[i]:off[i + 1]].sum() - 1.0) < 1e-5


def test_pair_kernel_stress_over_streams():
    """Race hunt (tools/pair_stress.py): 32 launches of a 41-layer 256-channel net on 777 positions over
    4 concurrent streams, every result bit-identical to the one-CTA kernel's."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools",
                                                       "pair_stress.py"), "8"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "mismatching launches: 0" in out.stdout


def test_duo_kernel_selected_for_multi_slot_contexts_and_matches(nb, orc, synth, monkeypatch):
    """A 128-channel ctx with >= 2 slots launches trunk_duo_kernel (two CTAs per SM, weights through tensor
    memory), a one-slot ctx trunk_fused.cu; both agree with the oracle, and with each other within float
    noise (different K order).  1,000 positions: 500 groups over 296 co-resident CTAs, two passes."""
    monkeypatch.delenv("NSB_TRUNK128", raising=False)
    desc = nb.net_desc(128, 3)
    blob = nb.random_blob(desc, 21)
    n = 1000
    pos = synth.random_positions(n, seed=4)
    fb = orc.pack(pos)
    off, idx = synth.random_legal_moves(n, seed=8, edge_rows=False)

    def run(slots, force=None):
        policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
        win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
        legal = np.zeros(int(off[-1]), dtype=np.float32)
        if force:
            monkeypatch.setenv("NSB_TRUNK128", force)
        else:
            monkeypatch.delenv("NSB_TRUNK128", raising=False)
        with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
            name = ctx.trunk_kernel_name()
            ctx.eval_async(0, fb, n, policy, win, draw)
            ctx.await_(0)
            ctx.eval_decode_async(slots - 1, fb, n, off, idx, nb.DECODE_PROBS, legal, win, draw, None)
            ctx.await_(slots - 1)
        return name, policy, win, legal

    n1, p1, w1, l1 = run(1, "classic")
    n2, p2, w2, l2 = run(2)
    assert n1 == "trunk_fused_kernel<128>" and n2.startswith("trunk_duo_kernel") and "2 CTAs per SM" in n2
    # a one-slot context left to itself holds both kernels and picks by batch size: 1,000 positions = 500 position pairs
    # are faster as two waves of co-resident CTA pairs (trunk_duo_kernel) than as four waves of one CTA per SM
    n0, p0, w0, l0 = run(1)
    assert n0.startswith("trunk_fused_kernel<128>") and "trunk_duo_kernel" in n0
    assert np.array_equal(p0.view(np.uint32), p2.view(np.uint32)) and np.array_equal(l0.view(np.uint32), l2.view(np.uint32))
    monkeypatch.delenv("NSB_TRUNK128", raising=False)
    op, ow, od = orc.forward(desc, blob, orc.expand(fb[:24 * 86], 24), emulate_bf16=True)
    for p, w in ((p1, w1), (p2, w2)):
        assert np.max(np.abs(p[:24] - op)) < 2 * TOL_LOGIT_VS_BF16_ORACLE and np.max(np.abs(w[:24] - ow)) < 2 * TOL_VALUE_VS_BF16_ORACLE
    assert np.max(np.abs(l1 - l2)) < 5e-3 and np.max(np.abs(w1 - w2)) < 2e-3
    # batch-index invariance inside the duo kernel: identical positions give identical bits
    same = np.random.default_rng(0).integers(0, 8, size=n)
    fb8 = np.ascontiguousarray(fb.reshape(n, 86)[same].reshape(-1))
    policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
    win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    with nb.Context(desc, batch_max=n, slots=2, blob=blob) as ctx:
        ctx.eval_async(0, fb8, n, policy, win, draw)
        ctx.await_(0)
    first = {int(k): int(np.argmax(same == k)) for k in np.unique(same)}
    ref_rows = np.array([first[int(k)] for k in same])
    assert np.array_equal(policy.view(np.uint32), policy[ref_rows].view(np.uint32)) and np.array_equal(win, win[ref_rows])


@pytest.mark.parametrize("channels,slots", [(128, 1), (128, 2), (256, 1)])
def test_stage1_fused_into_trunk_prologue(nb, orc, synth, monkeypatch, channels, slots):
    """SURVEY.md §8 f2: packed positions -> stem operand inside the trunk kernel (no bitboards in HBM).  For
    each trunk kernel (classic, duo, pair) the positions-in calls must give the bits of the bitboards-in
    calls fed with the oracle's stage 1, for dense logits, fused decode (odd n: a padded position in the
    last group) and the separate pack kernel (NSB_FUSE_PACK=0)."""
    monkeypatch.delenv("NSB_TRUNK128", raising=False)
    monkeypatch.delenv("NSB_TRUNK256", raising=False)
    desc = nb.net_desc(channels, 2)
    blob = nb.random_blob(desc, 77)
    n = 301
    pos = synth.random_positions(n, seed=31)
    pos["max_ply"][7] = 0  # guarded division (SURVEY App. A.2)
    fb = orc.pack(pos)
    off, idx = synth.random_legal_moves(n, seed=3)

    def run(fused):
        if fused:
            monkeypatch.delenv("NSB_FUSE_PACK", raising=False)
        else:
            monkeypatch.setenv("NSB_FUSE_PACK", "0")
        out = {}
        with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
            for name, src in (("bb", fb), ("pos", pos)):
                policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
                win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
                legal = np.zeros(int(off[-1]), dtype=np.float32)
                w2, d2 = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
                flag = np.ones(n, dtype=np.uint8)
                launches0 = ctx.launch_count()
                if name == "bb":
                    ctx.eval_async(0, src, n, policy, win, draw)
                    ctx.await_(0)
                    ctx.eval_decode_async(slots - 1, src, n, off, idx, nb.DECODE_LOGITS, legal, w2, d2, flag)
                else:
                    ctx.eval_positions_async(0, src, n, policy, win, draw)
                    ctx.await_(0)
                    ctx.eval_positions_decode_async(slots - 1, src, n, off, idx, nb.DECODE_LOGITS, legal, w2, d2, flag)
                ctx.await_(slots - 1)
                out[name] = (policy, win, draw, legal, w2, d2, flag, ctx.launch_count() - launches0)
        return out

    for fused in (True, False):
        o = run(fused)
        for a, b in zip(o["bb"][:7], o["pos"][:7]):
            assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b)
        # one kernel per call when fused, two (pack + trunk) otherwise
        assert o["bb"][7] == 2 and o["pos"][7] == (2 if fused else 4)


@pytest.mark.parametrize("channels,slots", [(128, 1), (128, 2), (256, 1)])
def test_direct_io_equals_staged(nb, orc, synth, monkeypatch, channels, slots):
    """NSB_IO_DIRECT: the trunk launch reads and writes the caller's mapped page-locked buffers itself (no copy
    nodes).  Same bits as the staged path for every host-buffer entry point; pageable buffers in direct mode
    silently take the staged path; a one-slot ctx defaults to direct, a pipeline to staged."""
    monkeypatch.delenv("NSB_IO", raising=False)
    monkeypatch.delenv("NSB_FUSE_PACK", raising=False)
    desc = nb.net_desc(channels, 2)
    blob = nb.random_blob(desc, 5)
    n = 203
    pos = synth.random_positions(n, seed=8)
    fb = orc.pack(pos)
    off, idx = synth.random_legal_moves(n, seed=9)
    total = int(off[-1])
    P = nb.PinnedArray
    h_fb, h_pos = P((n * 86,), nb.FEATURE_BITBOARD), P((n,), nb.POSITION)
    h_fb.array[:] = fb
    h_pos.array[:] = pos
    h_off, h_idx = P((n + 1,), np.uint32), P((total,), np.uint16)
    h_off.array[:] = off
    h_idx.array[:] = idx
    h_policy, h_win, h_draw = P((n, nb.POLICY_SIZE), np.float32), P((n,), np.float32), P((n,), np.float32)
    h_legal, h_flag = P((total,), np.float32), P((n,), np.uint8)

    def calls(ctx):
        out = []
        for src, dense, dec in ((h_fb, ctx.eval_async, ctx.eval_decode_async),
                                (h_pos, ctx.eval_positions_async, ctx.eval_positions_decode_async)):
            for a in (h_policy, h_win, h_draw, h_legal):
                a.array[...] = -7.0
            h_flag.array[:] = 9
            l0 = ctx.launch_count()
            dense(0, src.array, n, h_policy.array, h_win.array, h_draw.array)
            ctx.await_(0)
            out += [h_policy.array.copy(), h_win.array.copy(), h_draw.array.copy()]
            h_win.array[:] = -7.0
            dec(slots - 1, src.array, n, h_off.array, h_idx.array, nb.DECODE_PROBS, h_legal.array, h_win.array, h_draw.array,
                h_flag.array)
            ctx.await_(slots - 1)
            out += [h_legal.array.copy(), h_win.array.copy(), h_draw.array.copy(), h_flag.array.copy()]
            assert ctx.launch_count() - l0 == 2
        return out

    with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
        assert ctx.io_mode() == ("direct" if slots == 1 else "staged")
        ctx.set_io_mode(False)
        staged = calls(ctx)
        ctx.set_io_mode(True)
        assert ctx.io_mode() == "direct"
        direct = calls(ctx)
        # the caller refills the SAME buffers between batches (evaluationworker.cc:124-154): a launch must see the
        # new contents, not lines cached from the previous launch's reads of host memory
        h_fb.array[:] = fb.reshape(n, 86)[::-1].reshape(-1)
        h_pos.array[:] = pos[::-1]
        rev = calls(ctx)
        ctx.set_io_mode(False)
        rev_staged = calls(ctx)
        ctx.set_io_mode(True)
        h_fb.array[:] = fb
        h_pos.array[:] = pos
        # pageable numpy arrays in direct mode: staged fallback, same results
        policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
        win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
        ctx.eval_async(0, fb, n, policy, win, draw)
        ctx.await_(0)
    assert np.all(staged[0] != -7.0) and np.all(staged[3] != -7.0)
    for a, b in zip(staged, direct):
        assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b)
    assert np.array_equal(policy.view(np.uint32), staged[0].view(np.uint32)) and np.array_equal(win, staged[1])
    for a, b in zip(rev_staged, rev):
        assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b)
    assert np.array_equal(rev[0].view(np.uint32), staged[0][::-1].view(np.uint32)) and not np.array_equal(rev[1], staged[1])
    for a in (h_fb, h_pos, h_off, h_idx, h_policy, h_win, h_draw, h_legal, h_flag):
        a.free()


def test_direct_io_on_caller_registered_buffers(nb, orc, synth, monkeypatch):
    """The Infer contract with buffers the caller owns and pins (reference src/evaluate/evaluator.cc:95-106):
    nsb_host_register makes them eligible for direct I/O - one stream operation per computeNonBlocking."""
    monkeypatch.delenv("NSB_IO", raising=False)
    desc = nb.net_desc(128, 1)
    blob = nb.random_blob(desc, 3)
    n = 64
    fb = orc.pack(synth.random_positions(n, seed=2))
    feat = np.zeros(n * 86 + 256, dtype=nb.FEATURE_BITBOARD)[:n * 86]
    feat[:] = fb
    policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
    win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    with nb.Context(desc, batch_max=n, blob=blob) as ctx:
        assert ctx.io_mode() == "direct"
        ctx.eval_async(0, feat, n, policy, win, draw)   # pageable: staged fallback
        ctx.await_(0)
        want = (policy.copy(), win.copy(), draw.copy())
        bufs = (feat, policy, win, draw)
        for a in bufs:
            nb.host_register(a)
        try:
            for a in bufs[1:]:
                a[...] = 0
            ctx.eval_async(0, feat, n, policy, win, draw)
            ctx.await_(0)
        finally:
            for a in bufs:
                nb.host_unregister(a)
    for a, b in zip(want, (policy, win, draw)):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_adopted_host_ranges_are_revalidated_and_forgotten(nb, orc, synth, monkeypatch):
    """ADVICE r1 (medium): the reference's Evaluator pins its arrays itself (cudaHostRegister, evaluator.cc:95-106) and
    unpins + frees them BEFORE the executor is destroyed.  An adopted range must not survive that: (1) while the caller's
    registration stands, nsb_host_register adopts it and direct I/O works on it; (2) after the caller has unregistered
    it, registering the same address again must not trust the stale entry - the library locks the range itself;
    (3) nsb_host_unregister forgets an adopted range without unlocking it, and leaves nsb_host_alloc memory alone."""
    import torch
    monkeypatch.delenv("NSB_IO", raising=False)
    rt = torch.cuda.cudart()
    desc = nb.net_desc(128, 1)
    blob = nb.random_blob(desc, 3)
    n = 32
    fb = orc.pack(synth.random_positions(n, seed=2))
    feat = np.zeros(n * 86 + 512, dtype=nb.FEATURE_BITBOARD)[:n * 86]
    feat[:] = fb
    policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
    win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    bufs = (feat, policy, win, draw)
    with nb.Context(desc, batch_max=n, blob=blob) as ctx:
        ctx.eval_async(0, feat, n, policy, win, draw)            # pageable: staged
        ctx.await_(0)
        want = policy.copy()
        for a in bufs:                                            # the caller pins (what Evaluator does)
            assert int(rt.cudaHostRegister(a.ctypes.data, a.nbytes, 0)) == 0
        assert [nb.host_register(a) for a in bufs] == [False] * 4     # adopted: NSB_HOST_ALREADY_LOCKED
        policy[...] = 0
        l0 = ctx.launch_count()
        ctx.eval_async(0, feat, n, policy, win, draw)            # direct I/O on the adopted ranges
        ctx.await_(0)
        assert ctx.launch_count() - l0 == 1 and np.array_equal(policy.view(np.uint32), want.view(np.uint32))
        for a in bufs:                                            # ~Evaluator: the caller unpins; the entries are stale now
            assert int(rt.cudaHostUnregister(a.ctypes.data)) == 0
        assert [nb.host_register(a) for a in bufs] == [True] * 4      # NOT trusted: re-validated, locked by the library
        policy[...] = 0
        ctx.eval_async(0, feat, n, policy, win, draw)
        ctx.await_(0)
        assert np.array_equal(policy.view(np.uint32), want.view(np.uint32))
        for a in bufs:
            nb.host_unregister(a)                                 # unlocks what the library locked
        for a in bufs:                                            # forgotten: pageable again -> staged path, same bits
            assert int(rt.cudaHostRegister(a.ctypes.data, a.nbytes, 0)) == 0
            assert int(rt.cudaHostUnregister(a.ctypes.data)) == 0
        policy[...] = 0
        ctx.eval_async(0, feat, n, policy, win, draw)
        ctx.await_(0)
        assert np.array_equal(policy.view(np.uint32), want.view(np.uint32))
        pinned = nb.PinnedArray((16,), np.float32)               # nsb_host_alloc memory is not nsb_host_unregister's to forget
        nb.host_unregister(pinned.array)
        assert nb.host_register(pinned.array) is False
        pinned.free()


@pytest.mark.parametrize("channels,slots", [(128, 1), (128, 2), (256, 1)])
def test_rank_order_of_decoded_rows(nb, orc, synth, monkeypatch, channels, slots):
    """order_out of nsb_eval_request_async: per position the permutation that sorts its decoded row by decreasing
    value (the reference's Node::sort(), src/mcts/node.h:163-168, called per leaf at feedworker.cc:129), ties by
    lower index.  Bit-exact against the oracle's restatement applied to the GPU's own rows, for every trunk
    kernel, both decode modes, edge rows (1, 164, 165, 593 moves), duplicated policy slots (exact ties), NaN rows
    (identity), staged and direct I/O; the other outputs are unchanged by asking for the order."""
    monkeypatch.delenv("NSB_IO", raising=False)
    desc = nb.net_desc(channels, 2)
    blob = nb.random_blob(desc, 17)
    n = 70
    pos = synth.random_positions(n, seed=6)
    off, idx = synth.random_legal_moves(n, seed=6)          # edge rows included
    idx = idx.copy()
    r = 5                                                   # exact ties: one row gathers the same slot many times
    idx[off[r]:off[r + 1]] = idx[off[r]]
    idx[off[r + 1]:off[r + 1] + 4] = idx[off[r + 1]]
    total = int(off[-1])
    P = nb.PinnedArray
    h_pos, h_off, h_idx = P((n,), nb.POSITION), P((n + 1,), np.uint32), P((total,), np.uint16)
    h_pos.array[:], h_off.array[:], h_idx.array[:] = pos, off, idx
    h_legal, h_order = P((total,), np.float32), P((total,), np.uint16)
    h_win, h_draw, h_flag = P((n,), np.float32), P((n,), np.float32), P((n,), np.uint8)
    with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
        for direct in (False, True):
            ctx.set_io_mode(direct)
            for mode in (nb.DECODE_PROBS, nb.DECODE_LOGITS):
                h_order.array[:] = 0xFFFF
                ctx.eval_request_async(0, n, h_off.array, h_idx.array, mode, h_legal.array, h_win.array, h_draw.array,
                                       positions=h_pos.array, order_out=h_order.array, nan_flag=h_flag.array)
                ctx.await_(0)
                legal, order, flag = h_legal.array.copy(), h_order.array.copy(), h_flag.array.copy()
                assert not flag.any()
                assert np.array_equal(order, orc.rank_rows(legal, off, flag))
                for b in range(n):
                    row, o = legal[off[b]:off[b + 1]], order[off[b]:off[b + 1]].astype(np.int64)
                    assert np.array_equal(np.sort(o), np.arange(len(row)))            # a permutation
                    assert np.all(np.diff(row[o]) <= 0)                               # sortedness
                assert np.array_equal(order[off[r]:off[r + 1]], np.arange(off[r + 1] - off[r]))   # all tied: identity
                # same call without the order: identical rows
                plain = np.zeros(total, dtype=np.float32)
                w2, d2 = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
                ctx.eval_positions_decode_async(slots - 1, pos, n, off, idx, mode, plain, w2, d2, None)
                ctx.await_(slots - 1)
                assert np.array_equal(plain.view(np.uint32), legal.view(np.uint32)) and np.array_equal(w2, h_win.array)
    for a in (h_pos, h_off, h_idx, h_legal, h_order, h_win, h_draw, h_flag):
        a.free()


def _nan_case_blobs(nb, desc, blob):
    """Three nets that produce NaNs in different places: the draw-rate bias (every position's draw rate is NaN, its
    logits are fine), the bias of policy plane 3 (a NaN logit in every row that gathers a slot of that plane, values
    fine), and both."""
    out = {}
    for name in ("draw", "logit", "both"):
        b = blob.copy()
        w = helpers.split_blob(desc, b)      # views into b
        if name in ("draw", "both"):
            w["fc2_b"][1] = np.nan
        if name in ("logit", "both"):
            w["pol_b"][3] = np.nan
        out[name] = b
    return out


@pytest.mark.parametrize("channels,slots", [(128, 1), (128, 2), (256, 1)])
def test_nan_semantics_follow_feedworker(nb, orc, synth, monkeypatch, channels, slots):
    """The four cases of FeedWorker::feedResult<NaNFallbackEnabled> (src/mcts/feedworker.cc:56-137) on every trunk
    kernel, fused decode with rank order:
      fallback on,  NaN draw rate  (:58-85)  -> nan_flag, the row keeps its ORDINARY softmax and rank order
      fallback on,  NaN logit      (:105-118)-> nan_flag, uniform row, identity order; 1-move rows untouched (:100-103)
      fallback off (reference default, src/context.h:103): nan_flag stays 0; NaN logits flow through the softmax
                    (the whole row is NaN, identity order); a NaN draw rate changes nothing
    and the reference's cache rule (:134: store iff !NaNFound): flagged rows are evaluated again, unflagged ones hit."""
    monkeypatch.delenv("NSB_TRUNK128", raising=False)
    monkeypatch.delenv("NSB_IO", raising=False)
    desc = nb.net_desc(channels, 1)
    blob = nb.random_blob(desc, 17)
    blobs = _nan_case_blobs(nb, desc, blob)
    n = 33
    pos = synth.random_positions(n, seed=9)
    off, idx = synth.random_legal_moves(n, seed=9)          # edge rows: 1, 164, 165, 593, 2 moves
    total = int(off[-1])
    hashes = np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(7)
    touches = np.array([np.any(idx[off[b]:off[b + 1]] // 81 == 3) for b in range(n)])   # rows that gather plane 3
    one_move = np.diff(off) == 1
    assert touches.sum() > 5 and (~touches).sum() >= 1 and one_move[0]

    def call(ctx, mode, use_cache=False):
        legal, order = np.zeros(total, dtype=np.float32), np.full(total, 0xFFFF, dtype=np.uint16)
        win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
        flag, hit = np.full(n, 9, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        ctx.eval_request_async(slots - 1, n, off, idx, mode, legal, win, draw, positions=pos, order_out=order,
                               nan_flag=flag, hashes=hashes if use_cache else None, hit_flag=hit if use_cache else None)
        ctx.await_(slots - 1)
        return legal, order, flag, hit, win, draw

    with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
        clean = call(ctx, nb.DECODE_PROBS)
    assert not clean[2].any() and np.array_equal(clean[1], orc.rank_rows(clean[0], off))
    F = nb.DECODE_NAN_FALLBACK
    for case, bl in blobs.items():
        with nb.Context(desc, batch_max=n, slots=slots, blob=bl) as ctx:
            dense = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
            dw, dd = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
            ctx.eval_positions_async(0, pos, n, dense, dw, dd)
            ctx.await_(0)
            assert np.isnan(dd).all() == (case != "logit") and np.isnan(dense[:, 3 * 81:4 * 81]).all() == (case != "draw")
            for mode in (nb.DECODE_PROBS | F, nb.DECODE_PROBS):
                legal, order, flag, _, win, draw = call(ctx, mode)
                want, wflag = orc.decode(dense, dw, dd, off, idx, mode)           # the oracle on the GPU's own logits
                assert np.array_equal(flag, wflag), (case, mode)
                assert np.array_equal(np.isnan(legal), np.isnan(want)), (case, mode)
                assert np.allclose(legal, want, rtol=TOL_DECODE_REL, atol=1e-9, equal_nan=True), (case, mode)
                assert np.array_equal(order, orc.rank_rows(legal, off)), (case, mode)
                assert np.array_equal(np.isnan(draw), np.isnan(dd)) and np.array_equal(win, dw)   # values come back as they are
                logit_rows = touches & ~one_move if case != "draw" else np.zeros(n, dtype=bool)
                if mode & F:
                    assert np.array_equal(flag.astype(bool), logit_rows if case == "logit" else np.ones(n, dtype=bool))
                else:
                    assert not flag.any()
                for b in range(n):
                    row, o = legal[off[b]:off[b + 1]], order[off[b]:off[b + 1]]
                    if logit_rows[b]:
                        assert np.array_equal(o, np.arange(len(row)))                      # uniform or all-NaN: identity
                        if mode & F:
                            assert np.allclose(row, 1.0 / len(row), rtol=1e-6)            # feedworker.cc:111-118
                        else:
                            assert np.isnan(row).all()
                    elif case == "draw":                                                   # policy untouched: the clean net's row
                        assert np.array_equal(row.view(np.uint32), clean[0][off[b]:off[b + 1]].view(np.uint32))
                        assert np.array_equal(o, clean[1][off[b]:off[b + 1]])
            # the cache follows NaNFound (feedworker.cc:134)
            for mode in (nb.DECODE_PROBS | F, nb.DECODE_PROBS):
                ctx.cache_create(4) if mode & F else ctx.cache_clear()
                first = call(ctx, mode, use_cache=True)
                again = call(ctx, mode, use_cache=True)
                cacheable = (np.diff(off) <= 164) & ~first[2].astype(bool)
                assert first[3].sum() == 0 and np.array_equal(again[3].astype(bool), cacheable), (case, mode)
                assert np.array_equal(np.isnan(again[0]), np.isnan(first[0]))
                assert np.array_equal(again[1], first[1])                                  # hits are ranked like evaluated rows


def test_selfplay_decode_in_one_launch(nb, orc, synth, monkeypatch):
    """NSB_DECODE_BOTH = Frame::setEvaluation<false> (src/selfplay/frame.cc:93-118) in one evaluation: the raw logits
    go to the device cache (:110-114), the caller receives probabilities (:116-118) - raw logits at Gumbel roots
    (NSB_ROW_SKIP_SOFTMAX) - and, if asked, the raw logits as well; rows served from the cache take the same route and
    give the same bits as evaluated ones.  Against the oracle's restatement on the GPU's own dense logits; the
    Dirichlet mix of the AlphaZero root (:121-133) is host code, checked in nsb_host_unit."""
    monkeypatch.delenv("NSB_IO", raising=False)
    for channels, slots in ((128, 1), (128, 2), (256, 1)):
        desc = nb.net_desc(channels, 2)
        blob = nb.random_blob(desc, 5)
        n = 61
        pos = synth.random_positions(n, seed=12)
        off, idx = synth.random_legal_moves(n, seed=12)
        total = int(off[-1])
        rf = (np.arange(n) % 7 == 1).astype(np.uint8) * nb.ROW_SKIP_SOFTMAX
        rf[1] = nb.ROW_SKIP_SOFTMAX                       # a cacheable 164-move row that is a Gumbel root
        hashes = np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(11)
        P = nb.PinnedArray
        hp = {k: P(a.shape, a.dtype) for k, a in dict(pos=pos, off=off, idx=idx, rf=rf, hashes=hashes).items()}
        for k, a in dict(pos=pos, off=off, idx=idx, rf=rf, hashes=hashes).items():
            hp[k].array[...] = a
        o = dict(legal=P((total,), np.float32), logits=P((total,), np.float32), order=P((total,), np.uint16),
                 win=P((n,), np.float32), draw=P((n,), np.float32), flag=P((n,), np.uint8), hit=P((n,), np.uint8))

        def call(ctx, direct, use_cache, row_flags=True, want_logits=True):
            for a in o.values():
                a.array[...] = 0
            ctx.set_io_mode(direct)
            ctx.eval_request_async(slots - 1, n, hp["off"].array, hp["idx"].array, nb.DECODE_BOTH, o["legal"].array, o["win"].array,
                                   o["draw"].array, positions=hp["pos"].array, order_out=o["order"].array, nan_flag=o["flag"].array,
                                   hashes=hp["hashes"].array if use_cache else None, hit_flag=o["hit"].array if use_cache else None,
                                   row_flags=hp["rf"].array if row_flags else None, logits_out=o["logits"].array if want_logits else None)
            ctx.await_(slots - 1)
            return {k: a.array.copy() for k, a in o.items()}

        with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
            dense = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
            dw, dd = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
            ctx.eval_positions_async(0, pos, n, dense, dw, dd)
            ctx.await_(0)
            want, want_log, _ = orc.decode_ex(dense, dw, dd, off, idx, nb.DECODE_BOTH, row_flags=rf, want_logits=True)
            ctx.cache_create(8)
            plain = call(ctx, False, False)
            assert np.array_equal(plain["logits"].view(np.uint32), want_log.view(np.uint32))      # gather: bit-exact
            assert np.allclose(plain["legal"], want, rtol=TOL_DECODE_REL, atol=1e-9)
            for b in np.nonzero(rf)[0]:
                assert np.array_equal(plain["legal"][off[b]:off[b + 1]].view(np.uint32), want_log[off[b]:off[b + 1]].view(np.uint32))
            assert np.array_equal(plain["order"], orc.rank_rows(plain["legal"], off)) and not plain["flag"].any()
            miss = call(ctx, True, True)                  # fills the cache with RAW LOGITS
            hit = call(ctx, False, True)                  # served from it: softmax of the stored logits
            hit_direct = call(ctx, True, True, want_logits=False)
            cacheable = np.diff(off) <= 164
            assert miss["hit"].sum() == 0 and np.array_equal(hit["hit"].astype(bool), cacheable)
            for r in (miss, hit, hit_direct):
                for k in ("legal", "win", "draw", "order"):
                    assert np.array_equal(r[k].view(np.uint32) if r[k].dtype == np.float32 else r[k],
                                          plain[k].view(np.uint32) if plain[k].dtype == np.float32 else plain[k]), k
            assert np.array_equal(hit["logits"].view(np.uint32), plain["logits"].view(np.uint32))
            # what the cache holds is the raw logits (frame.cc:110-114): a LOGITS-mode probe returns them unchanged
            for a in o.values():
                a.array[...] = 0
            ctx.eval_request_async(slots - 1, n, hp["off"].array, hp["idx"].array, nb.DECODE_LOGITS, o["legal"].array, o["win"].array,
                                   o["draw"].array, positions=hp["pos"].array, hashes=hp["hashes"].array, hit_flag=o["hit"].array)
            ctx.await_(slots - 1)
            assert np.array_equal(o["legal"].array.view(np.uint32), plain["logits"].view(np.uint32)) and o["hit"].array.sum() == cacheable.sum()
            # without row flags every row is softmaxed
            noflags = call(ctx, False, False, row_flags=False)
            want2, _, _ = orc.decode_ex(dense, dw, dd, off, idx, nb.DECODE_BOTH)
            assert np.allclose(noflags["legal"], want2, rtol=TOL_DECODE_REL, atol=1e-9)
        for a in list(hp.values()) + list(o.values()):
            a.free()


@pytest.mark.parametrize("channels,slots", [(128, 1), (128, 2), (256, 1)])
def test_custom_features_v1_93_channels(nb, orc, synth, monkeypatch, channels, slots):
    """preset::CustomFeaturesV1 (reference src/evaluate/preset.h:68-122): 93 planes, eleven of them (82..92) with
    arbitrary fp32 fill values.  The executor takes any feature count up to 96 as bitboards (the Infer contract); the
    stem then runs 8 K-steps per tap (93 + 11 twin channels).  Against the oracle on every trunk kernel; the fused
    expansion equals the standalone extract kernel's planes fed to the oracle; packed positions are refused (stage 1
    on the device builds SimpleFeatures)."""
    monkeypatch.delenv("NSB_TRUNK128", raising=False)
    monkeypatch.delenv("NSB_IO", raising=False)
    IN = 93
    desc = nb.net_desc(channels, 2, in_channels=IN)
    blob = nb.random_blob(desc, 31)
    n = 37
    fb = synth.random_feature_bitboards(n * IN, seed=93)
    # planes 0..81 are 0/1 planes in the real feature set: give them the fill value 1.0 (bits 32..63 of hi)
    hi = fb["hi"].reshape(n, IN)
    hi[:, :82] = (hi[:, :82] & np.uint64(0xFFFFFFFF)) | (np.uint64(0x3F800000) << np.uint64(32))
    fb["hi"] = hi.reshape(-1)
    off, idx = synth.random_legal_moves(n, seed=4)
    policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
    win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    legal = np.zeros(int(off[-1]), dtype=np.float32)
    w2, d2 = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
        ctx.eval_async(0, fb, n, policy, win, draw)
        ctx.await_(0)
        ctx.eval_decode_async(slots - 1, fb, n, off, idx, nb.DECODE_PROBS, legal, w2, d2, None)
        ctx.await_(slots - 1)
        with pytest.raises(nb.NsbError) as e:
            ctx.eval_positions_async(0, synth.random_positions(n, seed=1), n, policy.copy(), win.copy(), draw.copy())
        assert "SimpleFeatures" in str(e.value)
    planes = orc.expand(fb, n, IN)
    op, ow, od = orc.forward(desc, blob, planes, emulate_bf16=True)
    assert np.max(np.abs(policy - op)) < TOL_LOGIT_VS_BF16_ORACLE
    assert np.max(np.abs(win - ow)) < TOL_VALUE_VS_BF16_ORACLE and np.max(np.abs(draw - od)) < TOL_VALUE_VS_BF16_ORACLE
    fp, fw, fd = orc.forward(desc, blob, planes, emulate_bf16=False)
    pg, _ = orc.decode(policy, win, draw, off, idx, nb.DECODE_PROBS)
    pf, _ = orc.decode(fp, fw, fd, off, idx, nb.DECODE_PROBS)
    assert np.max(np.abs(pg - pf)) < TOL_PROB_VS_FP32 and np.max(np.abs(win - fw)) < TOL_VALUE_VS_FP32
    assert np.allclose(legal, pg, rtol=1e-6, atol=1e-9) and np.array_equal(w2, win)


def test_graft_entry_smoke():
    """The driver's smoke() entry point itself (it pins the launch count of the fused path)."""
    import __graft_entry__ as graft
    graft.smoke()


@pytest.mark.parametrize("channels,slots", [(128, 1), (128, 2), (256, 1)])
def test_maximum_batch_size(nb, orc, synth, monkeypatch, channels, slots):
    """batch_max = 65,535 (the reference's uint16_t BatchSizeMax, src/infer/trt.cc:52) in one call: 32,768 position
    pairs over 148 CTAs = 222 passes.  Checksum-of-rows property: every position is one of 16 base positions with
    one of 16 move lists, so every output row must equal, bit for bit, the row of its (position, list) pair from a
    16 x 16 reference batch; rank orders included.  All three trunk kernels (classic, duo, pair)."""
    monkeypatch.delenv("NSB_TRUNK256", raising=False)
    if channels == 128:   # bit-exact rows need ONE kernel for the 256-position reference batch and the big one
        monkeypatch.setenv("NSB_TRUNK128", "classic" if slots == 1 else "duo")
    desc = nb.net_desc(channels, 1)
    blob = nb.random_blob(desc, 3)
    n, base = 65535, 16
    pos16 = synth.random_positions(base, seed=77)
    off16, idx16 = synth.random_legal_moves(base, seed=77, edge_rows=False)
    rng = np.random.default_rng(5)

    def build(which_pos, which_list):
        cnt = np.diff(off16)[which_list].astype(np.int64)
        off = np.zeros(len(which_pos) + 1, dtype=np.uint32)
        off[1:] = np.cumsum(cnt)
        src = np.repeat(off16[:-1][which_list].astype(np.int64), cnt) + (np.arange(int(off[-1])) - np.repeat(off[:-1].astype(np.int64), cnt))
        return np.ascontiguousarray(pos16[which_pos]), off, np.ascontiguousarray(idx16[src])

    def run(ctx, p, off, idx):
        m = len(p)
        legal, order = np.zeros(int(off[-1]), dtype=np.float32), np.zeros(int(off[-1]), dtype=np.uint16)
        win, draw, flag = np.zeros(m, dtype=np.float32), np.zeros(m, dtype=np.float32), np.ones(m, dtype=np.uint8)
        ctx.eval_request_async(0, m, off, idx, nb.DECODE_PROBS, legal, win, draw, positions=p, order_out=order, nan_flag=flag)
        ctx.await_(0)
        return legal, order, win, draw, flag

    with nb.Context(desc, batch_max=n, slots=slots, blob=blob) as ctx:
        gp, gl = np.divmod(np.arange(base * base), base)
        ref_p, ref_off, ref_idx = build(gp, gl)
        r_legal, r_order, r_win, r_draw, _ = run(ctx, ref_p, ref_off, ref_idx)
        wp, wl = rng.integers(0, base, size=n), rng.integers(0, base, size=n)
        p, off, idx = build(wp, wl)
        legal, order, win, draw, flag = run(ctx, p, off, idx)
    assert not flag.any()
    pair = wp * base + wl
    assert np.array_equal(win, r_win[pair]) and np.array_equal(draw, r_draw[pair])
    cnt = np.diff(off).astype(np.int64)
    src = np.repeat(ref_off[:-1][pair].astype(np.int64), cnt) + (np.arange(int(off[-1])) - np.repeat(off[:-1].astype(np.int64), cnt))
    assert np.array_equal(legal.view(np.uint32), r_legal[src].view(np.uint32))
    assert np.array_equal(order, r_order[src])
    assert np.array_equal(r_order, orc.rank_rows(r_legal, ref_off))


def test_concurrent_contexts_soak_short():
    """tools/soak.py for 8 s: four host threads, four contexts (classic + shared cache, an executor attached to it, duo
    with 4 slots, the 256-channel pair kernel) on one GPU at once, every result bit-identical to its first."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "soak.py"), "8"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "soak ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_api_modes_differential_fuzz_short():
    """tools/fuzz_modes.py for 10 s: random nets / batch sizes / move lists (rows of 0, 1, 164, 165, 593 moves); bitboards in
    (staged) == packed positions in (direct, ranked) == through the cache (misses) == from the cache (hits), bit for bit,
    rank orders equal to the oracle's.  (2,708 configurations in a 150 s run while developing.)"""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "fuzz_modes.py"), "10", "7"], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0 and "fuzz ok" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]


def test_request_validation(nb, synth):
    """nsb_eval_request_async reports malformed requests instead of launching: both / neither input kind, a cache request
    without a cache, a bad decode mode, offsets that do not start at 0, decrease, or give a row more than 593 moves;
    a policy slot beyond 2186 (a caller's bug the reference would assert on) reads the last slot instead of faulting."""
    desc = nb.net_desc(128, 1)
    n = 4
    pos = synth.random_positions(n, seed=1)
    fb = np.zeros(n * 86, dtype=nb.FEATURE_BITBOARD)
    off, idx = synth.random_legal_moves(n, seed=1, edge_rows=False)
    legal = np.zeros(int(off[-1]), dtype=np.float32)
    win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    hashes = np.arange(n, dtype=np.uint64)
    with nb.Context(desc, batch_max=n, seed=1) as ctx:
        ok = dict(positions=pos)
        ctx.eval_request_async(0, n, off, idx, nb.DECODE_PROBS, legal, win, draw, **ok)
        ctx.await_(0)
        l0 = ctx.launch_count()
        for bad in (dict(positions=pos, features=fb), dict(), dict(positions=pos, hashes=hashes)):
            with pytest.raises(nb.NsbError):
                ctx.eval_request_async(0, n, off, idx, nb.DECODE_PROBS, legal, win, draw, **bad)
        with pytest.raises(nb.NsbError):
            ctx.eval_request_async(0, n, off, idx, 7, legal, win, draw, **ok)
        off_bad = off.copy()
        off_bad[0] = 1
        with pytest.raises(nb.NsbError):
            ctx.eval_request_async(0, n, off_bad, idx, nb.DECODE_PROBS, legal, win, draw, **ok)
        off_big = np.array([0, 594, 594, 594, 594], dtype=np.uint32) * np.uint32(n)   # > n * 593 moves in total
        with pytest.raises(nb.NsbError):
            ctx.eval_request_async(0, n, off_big, np.zeros(int(off_big[-1]), dtype=np.uint16), nb.DECODE_PROBS,
                                   np.zeros(int(off_big[-1]), dtype=np.float32), win, draw, **ok)
        off_dec = off.copy()
        off_dec[2] = off_dec[1] - 1                                                               # decreasing offsets
        with pytest.raises(nb.NsbError):
            ctx.eval_request_async(0, n, off_dec, idx, nb.DECODE_PROBS, legal, win, draw, **ok)
        off_row = np.array([0, 594, 595, 596, 597], dtype=np.uint32)                               # one row of 594 moves
        with pytest.raises(nb.NsbError):
            ctx.eval_request_async(0, n, off_row, np.zeros(597, dtype=np.uint16), nb.DECODE_PROBS, np.zeros(597, dtype=np.float32),
                                   win, draw, **ok)
        for bad_mode in (3, 0x200, nb.DECODE_NAN_FALLBACK | 3):
            with pytest.raises(nb.NsbError):
                ctx.eval_request_async(0, n, off, idx, bad_mode, legal, win, draw, **ok)
        with pytest.raises(nb.NsbError):
            ctx.eval_request_async(0, n + 1, off, idx, nb.DECODE_PROBS, legal, win, draw, **ok)    # > batch_max
        assert ctx.launch_count() == l0                                                            # nothing was launched
        ctx.eval_request_async(0, 0, off, idx, nb.DECODE_PROBS, legal, win, draw, **ok)            # n = 0 is a no-op
        assert ctx.launch_count() == l0
        idx_oob = idx.copy()
        idx_oob[:3] = [2187, 40000, 65535]                                                         # clamped to slot 2186
        idx_ref = idx.copy()
        idx_ref[:3] = 2186
        l_oob, l_ref = np.zeros_like(legal), np.zeros_like(legal)
        ctx.eval_request_async(0, n, off, idx_oob, nb.DECODE_LOGITS, l_oob, win, draw, **ok)
        ctx.await_(0)
        ctx.eval_request_async(0, n, off, idx_ref, nb.DECODE_LOGITS, l_ref, win, draw, **ok)
        ctx.await_(0)
        assert np.array_equal(l_oob.view(np.uint32), l_ref.view(np.uint32))
