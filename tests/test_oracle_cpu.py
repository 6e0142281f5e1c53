"""CPU suite (-m "not gpu"): pins the oracle against the reference's own compiled sources, known
answers and independent restatements; checks the C-ABI library exports; no GPU compute calls."""
import ctypes
import hashlib
import os
import re
import subprocess

import numpy as np
import pytest

import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- expand (reference src/cuda/extractbit.cu) ----------------------------------------------------
def test_expand_known_answers(orc, nb):
    """Hand-derived cases of extractbit.cu:20-37: lo/hi split at square 63, rotate, value bits,
    garbage bits 18..23 / 25..31 ignored, bit 63 of lo ignored."""
    one = np.uint64(0x3F800000) << np.uint64(32)
    fb = np.zeros(6, dtype=nb.FEATURE_BITBOARD)
    fb["lo"][0], fb["hi"][0] = 1, one                                  # square 0
    fb["lo"][1], fb["hi"][1] = 1 << 62, one                            # square 62 (last bit of lo)
    fb["lo"][2], fb["hi"][2] = 1 << 63, one | np.uint64(1)             # lo bit 63 ignored; square 63
    fb["lo"][3], fb["hi"][3] = 1, one | (np.uint64(1) << np.uint64(24))  # rotate: square 0 -> t = 80
    v = np.float32(0.375)
    fb["lo"][4] = (1 << 63) - 1
    fb["hi"][4] = np.uint64(0x3FFFF) | (np.uint64(v.view(np.uint32)) << np.uint64(32))  # all ones * value
    fb["lo"][5], fb["hi"][5] = 0, one | (np.uint64(0x3F) << np.uint64(18)) | (np.uint64(0x7F) << np.uint64(25)) \
        | (np.uint64(1) << np.uint64(17))                              # garbage + square 80
    out = orc.expand(fb, 1, 6, True)[0]
    exp = np.zeros((6, 81), dtype=np.float32)
    exp[0, 0] = 1
    exp[1, 62] = 1
    exp[2, 63] = 1
    exp[3, 80] = 1
    exp[4, :] = v
    exp[5, 80] = 1  # garbage bits 18..23 / 25..31 change nothing (bit 24 = rotate stays 0)
    assert np.array_equal(out.view(np.uint32), exp.view(np.uint32))


def test_expand_matches_numpy_restatement_and_golden(orc, nb, synth, golden_dir):
    g = np.load(os.path.join(golden_dir, "expand_kat.npz"))
    fb = np.zeros(96, dtype=nb.FEATURE_BITBOARD)
    fb["lo"], fb["hi"] = g["lo"], g["hi"]
    assert np.array_equal(orc.expand(fb, 2, 48, True).view(np.uint32), g["nchw"])
    assert np.array_equal(orc.expand(fb, 2, 48, False).view(np.uint32), g["nhwc"])
    fb = synth.random_feature_bitboards(7 * 86, seed=3)
    for cf in (True, False):
        assert np.array_equal(orc.expand(fb, 7, 86, cf).view(np.uint32),
                              helpers.expand_numpy(fb, 7, 86, cf).view(np.uint32))


def test_expand_empty(orc, nb):
    assert orc.expand(np.zeros(0, dtype=nb.FEATURE_BITBOARD), 0).shape == (0, 86, 81)


# ---- Random executor (reference src/infer/random.cc) --------------------------------------------------
def test_mt19937_64_known_answer(orc):
    """C++ standard [rand.predef]: the 10000th invocation of a default-constructed mt19937_64
    (seed 5489) is 9981545732273789042.  The oracle exposes floats, so check through the float
    conversion float(u)/2^64 of libstdc++'s generate_canonical<float,24> (one draw per float)."""
    l = orc.lib()
    r = l.nsb_oracle_rng_create(5489)
    n = 10000
    pol = np.empty((5, 2187), dtype=np.float32)
    w = np.empty(5, dtype=np.float32)
    d = np.empty(5, dtype=np.float32)
    l.nsb_oracle_random_fill(r, 5, pol.ctypes.data, w.ctypes.data, d.ctypes.data)  # 10945 draws
    l.nsb_oracle_rng_destroy(r)
    flat = np.concatenate([np.concatenate([pol[i], [w[i]], [d[i]]]) for i in range(5)])
    expect = np.float32(np.float32(9981545732273789042) / np.float32(18446744073709551616.0))
    assert flat[n - 1] == expect


def test_random_port_equals_reference_build_and_golden(orc, golden_dir):
    g = np.load(os.path.join(golden_dir, "random_ref.npz"))
    for seed in (0, 7):
        p, w, d = orc.random_fill(seed, 3)
        assert np.array_equal(p[:, :8], g[f"policy_head_{seed}"])
        assert np.array_equal(p[:, -4:], g[f"policy_tail_{seed}"])
        assert np.array_equal(w, g[f"win_{seed}"]) and np.array_equal(d, g[f"draw_{seed}"])
        sha = hashlib.sha256(p.tobytes() + w.tobytes() + d.tobytes()).digest()
        assert sha == g[f"sha256_{seed}"].tobytes()
        assert p.min() >= 0.0 and p.max() < 1.0
        if orc.have_ref_random():  # the reference's random.cc compiled in place (build container / GPU box)
            rp, rw, rd = orc.ref_random_fill(seed, 3)
            assert np.array_equal(p, rp) and np.array_equal(w, rw) and np.array_equal(d, rd)


# ---- pack (channel order src/evaluate/preset.h:20-66; semantics builder-defined) -------------------------
def test_pack_structure(orc, nb, synth):
    pos = synth.random_positions(32, seed=5)
    fb = orc.pack(pos).reshape(32, 86)
    planes = orc.expand(fb.reshape(-1), 32).reshape(32, 86, 81)
    for i in range(32):
        p = pos[i]
        me = int(p["side"])
        # every piece appears in exactly one of the 28 board planes, on its (possibly rotated) square
        occ = planes[i, :28].sum(axis=0)
        board = p["board"][::-1] if me == 1 else p["board"]
        assert np.array_equal(occ > 0, board > 0)
        assert occ.max() <= 1
        for s in range(81):
            code = int(board[s])
            if code:
                colour, pt = (code - 1) // 14, (code - 1) % 14
                ch = pt + (0 if colour == me else 14)
                assert planes[i, ch, s] == 1.0
        # stand planes are all-or-nothing thermometers
        k = 28
        for side in (me, 1 - me):
            for piece, mx in enumerate([6, 4, 4, 4, 4, 2, 2]):
                for j in range(1, mx + 1):
                    want = 1.0 if p["hands"][side][piece] >= j else 0.0
                    assert np.all(planes[i, k] == want)
                    k += 1
        assert np.all(planes[i, 80] == (1.0 if me == 0 else 0.0))
        assert np.all(planes[i, 81] == (1.0 if me == 1 else 0.0))
        assert np.all(planes[i, 82] == np.float32(p["ply"]) / np.float32(p["max_ply"]))
        assert np.all(planes[i, 83] == np.float32(1.0) / np.float32(p["max_ply"]))
        my_dv = p["black_draw_value"] if me == 0 else p["white_draw_value"]
        assert np.all(planes[i, 84] == my_dv)
        # rotate flag on every plane iff white to move
        assert np.all(((fb[i]["hi"] >> np.uint64(24)) & np.uint64(1)) == me)


def test_startpos_has_40_pieces(orc, synth):
    pos = synth.startpos(2)
    planes = orc.expand(orc.pack(pos), 2)
    assert planes[0, :28].sum() == 40 and planes[0, 28:80].sum() == 0


# ---- decode (reference src/mcts/feedworker.cc:56-136, src/selfplay/frame.cc:93-136) ------------------------
def test_decode_properties(orc, nb, synth):
    """synth.random_logits: row 5 all-NaN logits, row 6 some NaN logits, row 7 -inf logits, row 8 NaN win rate,
    row 9 NaN draw rate.  The four cases of FeedWorker::feedResult<NaNFallbackEnabled>:
      fallback on,  NaN logit (:105-118)  -> uniform row, NaNFound
      fallback on,  NaN win/draw (:58-85) -> NaNFound, the row keeps its normal softmax
      fallback off (the reference's default, context.h:103), NaN logit -> NaNs flow through softmax_, no flag
      fallback off, NaN win/draw          -> nothing happens to the row, no flag"""
    n = 64
    policy, win, draw = synth.random_logits(n, seed=1)
    off, idx = synth.random_legal_moves(n, seed=1)
    ref = helpers.softmax_rows(np.nan_to_num(policy, nan=0.0), off, idx)
    rows = lambda a, i: a[off[i]:off[i + 1]]
    for fallback in (True, False):
        mode = nb.DECODE_PROBS | (nb.DECODE_NAN_FALLBACK if fallback else 0)
        probs, flag = orc.decode(policy, win, draw, off, idx, mode)
        logits, flag2 = orc.decode(policy, win, draw, off, idx, nb.DECODE_LOGITS | (mode & nb.DECODE_NAN_FALLBACK))
        assert probs[off[0]] == 1.0 and off[1] - off[0] == 1      # 1-move shortcut (feedworker.cc:101-103)
        if fallback:
            assert list(np.nonzero(flag)[0]) == [5, 6, 8, 9] and np.array_equal(flag, flag2)
        else:
            assert not flag.any() and not flag2.any()
        for i in range(n):
            row, m = rows(probs, i), int(off[i + 1] - off[i])
            g = policy[i, idx[off[i]:off[i + 1]]]
            assert np.array_equal(rows(logits, i).view(np.uint32), g.view(np.uint32))   # raw gather
            if i in (5, 6) and m > 1:
                if fallback:     # NaN logit -> every legal logit := 1 -> uniform (feedworker.cc:111-118)
                    assert np.allclose(row, 1.0 / m, rtol=1e-6)
                elif np.isnan(g).any():
                    assert np.isnan(row).all()
                continue
            # rows 8 / 9 (NaN win / draw): the policy is the ordinary softmax either way
            assert abs(row.sum() - 1.0) < 1e-5
            if m > 1:
                assert np.allclose(row, rows(ref, i), rtol=2e-6, atol=1e-9)
    # a 1-move row never looks at its logit (:100-103), even when it is NaN and the fallback is on
    policy1 = policy.copy()
    policy1[0, :] = np.nan
    probs, flag = orc.decode(policy1, win, draw, off, idx, nb.DECODE_PROBS | nb.DECODE_NAN_FALLBACK)
    assert probs[off[0]] == 1.0 and flag[0] == 0


def test_decode_selfplay_flavour(orc, nb, synth):
    """Frame::setEvaluation<false> (frame.cc:93-136): raw logits (what the cache keeps) + softmax; no 1-move shortcut;
    the Gumbel root skips the softmax; no NaN handling unless the reporting bit is set."""
    n = 40
    policy, win, draw = synth.random_logits(n, seed=3)
    off, idx = synth.random_legal_moves(n, seed=3)
    rf = np.zeros(n, dtype=np.uint8)
    rf[[2, 11]] = nb.ROW_SKIP_SOFTMAX
    probs, logits, flag = orc.decode_ex(policy, win, draw, off, idx, nb.DECODE_BOTH, row_flags=rf, want_logits=True)
    raw, _ = orc.decode(policy, win, draw, off, idx, nb.DECODE_LOGITS)
    assert np.array_equal(logits.view(np.uint32), raw.view(np.uint32)) and not flag.any()
    ref = helpers.softmax_rows(np.nan_to_num(policy, nan=0.0), off, idx)
    for i in range(n):
        row, g = probs[off[i]:off[i + 1]], raw[off[i]:off[i + 1]]
        if rf[i]:
            assert np.array_equal(row.view(np.uint32), g.view(np.uint32))
        elif np.isnan(g).any():
            assert np.isnan(row).all()
        else:
            assert np.allclose(row, ref[off[i]:off[i + 1]], rtol=2e-6, atol=1e-9)
    assert probs[off[0]] == 1.0                                   # softmax of one finite logit
    _, _, flag = orc.decode_ex(policy, win, draw, off, idx, nb.DECODE_BOTH | nb.DECODE_NAN_FALLBACK, row_flags=rf)
    assert list(np.nonzero(flag)[0]) == [5, 6, 8, 9]


def test_value_fallback_and_dirichlet_mix(orc):
    """feedworker.cc:58-85 and frame.cc:121-133, against hand-computed values."""
    nan = float("nan")
    assert orc.value_fallback(0.3, 0.1, True, 5.0, 1.0, 10) == (np.float32(0.3), np.float32(0.1), False)
    w, d, f = orc.value_fallback(nan, 0.1, True, 6.0, 1.0, 8)
    assert f and w == np.float32(1.0 - 6.0 / 8.0) and d == np.float32(0.1)
    w, d, f = orc.value_fallback(0.3, nan, True, 6.0, 1.0, 8)
    assert f and w == np.float32(0.3) and d == np.float32(1.0 / 8.0)
    assert orc.value_fallback(nan, nan, False) == (0.5, 0.0, True)
    rng = np.random.default_rng(4)
    p = rng.random(50).astype(np.float32)
    noise = rng.gamma(0.15, 1.0, size=600)
    noise /= noise.sum()                                          # worker.cc:170-176
    mixed = orc.dirichlet_mix(p, noise)
    want = (0.75 * p.astype(np.float64) + 0.25 * noise[:50]).astype(np.float32)
    assert np.array_equal(mixed.view(np.uint32), want.view(np.uint32))


# ---- forward oracle vs PyTorch fp32 ----------------------------------------------------------------------
def test_forward_oracle_matches_torch_and_golden(orc, nb, synth, golden_dir):
    g = np.load(os.path.join(golden_dir, "forward_small.npz"))
    desc = nb.net_desc(128, 1)
    blob = nb.random_blob(desc, int(g["blob_seed"]))
    assert hashlib.sha256(blob.tobytes()).digest() == g["blob_sha256"].tobytes()
    pos = np.frombuffer(g["positions"].tobytes(), dtype=nb.POSITION)
    planes = orc.expand(orc.pack(pos), len(pos))
    p32, w32, d32 = orc.forward(desc, blob, planes, emulate_bf16=False)
    assert np.allclose(p32, g["policy_fp32"], atol=1e-5) and np.allclose(w32, g["win_fp32"], atol=1e-6)
    tp, tw, td = helpers.forward_torch(desc, blob, planes)
    assert np.max(np.abs(p32 - tp)) < 2e-4
    assert np.max(np.abs(w32 - tw)) < 1e-5 and np.max(np.abs(d32 - td)) < 1e-5
    p16, w16, d16 = orc.forward(desc, blob, planes, emulate_bf16=True)
    assert np.allclose(p16, g["policy_bf16"], atol=1e-5)
    # bf16 activations stay close to fp32 (tolerance of the GPU parity test, stated there too)
    assert np.max(np.abs(p16 - p32)) < 0.15 and np.max(np.abs(w16 - w32)) < 1e-2


def test_weight_blob_is_bf16_exact(orc, nb):
    desc = nb.net_desc(128, 1)
    blob = nb.random_blob(desc, 1)
    assert blob.size == ctypes.c_size_t(nb.lib().nsb_weight_blob_floats(ctypes.byref(desc))).value
    assert np.all((blob.view(np.uint32) & 0xFFFF) == 0)
    assert np.array_equal(blob, nb.random_blob(desc, 1)) and not np.array_equal(blob, nb.random_blob(desc, 2))


# ---- C-ABI surface ---------------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol(nb):
    hdr = open(os.path.join(ROOT, "include", "nsb.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(nsb_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 30
    out = subprocess.check_output(["nm", "-D", "--defined-only", nb.LIB_PATH], text=True)
    exported = set(re.findall(r" T (nsb_[a-z0-9_]+)", out))
    assert declared == exported, (declared - exported, exported - declared)
    assert declared == set(nb.SIGNATURES), (declared ^ set(nb.SIGNATURES))
    l = nb.lib()
    assert b"sm_100a" in l.nsb_version()
    # the diagnostic build (include/nsb_diag.h): every product symbol + the nsb_debug_* entry points, nothing else
    dhdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "nsb_diag.h")).read(), flags=re.S)
    diag_declared = set(re.findall(r"\b(nsb_[a-z0-9_]+)\s*\(", dhdr))
    assert diag_declared == set(nb.DIAG_SIGNATURES) and all(n.startswith("nsb_debug_") for n in diag_declared)
    out = subprocess.check_output(["nm", "-D", "--defined-only", nb.DIAG_LIB_PATH], text=True)
    assert set(re.findall(r" T (nsb_[a-z0-9_]+)", out)) == declared | diag_declared
    assert b"diagnostic build" in nb.diag_lib().nsb_version() and b"diagnostic" not in l.nsb_version()


def test_library_is_sm100a_tcgen05_and_has_no_oracle(nb):
    """The product binary carries sm_100a SASS with tcgen05 (UTCHMMA) + bulk copies (UBLKCP), and
    neither the library nor the package sources reference the oracle."""
    sass = subprocess.run(["cuobjdump", "-sass", nb.LIB_PATH], capture_output=True, text=True)
    if sass.returncode == 0 and sass.stdout:
        assert "sm_100a" in sass.stdout
        assert "UTCHMMA" in sass.stdout and "UBLKCP" in sass.stdout and "LDTM" in sass.stdout
        # probes, the experimental trunk_ts.cu and the superseded one-CTA 256-channel kernel are not in the product
        kernels = set(re.findall(r"Function : (\S+)", sass.stdout))
        assert kernels and not any(k for k in kernels if "umma_probe" in k or "bulk_" in k or "trunk_ts" in k or "trunk_fused_kernelILi256" in k), kernels
        # one 128-channel one-CTA kernel, with no cluster-size template argument
        assert len([k for k in kernels if "trunk_fused_kernelILi128E" in k]) == 1, kernels
        assert not any("trunk_fused_kernelILi128ELi" in k for k in kernels), kernels
        assert any("trunk_duo_kernel" in k for k in kernels) and any("trunk_pair_kernel" in k for k in kernels)
    needed = subprocess.check_output(["readelf", "-d", nb.LIB_PATH], text=True)
    assert "oracle" not in needed
    pkg_dir = os.path.dirname(nb.LIB_PATH)
    for d, _, files in os.walk(pkg_dir):
        if "build" in d or "__pycache__" in d:
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cc", ".h", ".cpp")):
                src = open(os.path.join(d, f), errors="ignore").read()
                assert "nsb_oracle" not in src and "libnsb_oracle" not in src, f


def test_fails_loudly_without_gpu(nb):
    """No CPU fallback: on a box without a GPU nsb_create must fail with NSB_ERR_NO_DEVICE."""
    if nb.device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(nb.NsbError) as e:
        nb.Context(nb.net_desc(128, 1), batch_max=4)
    assert "-3" in str(e.value) and "no CPU fallback" in str(e.value)


def test_create_rejects_bad_arguments(nb, monkeypatch):
    l = nb.lib()
    h = ctypes.c_void_p()
    bad = nb.net_desc(96, 1)
    assert l.nsb_create(ctypes.byref(h), 0, 8, 1, ctypes.byref(bad)) == -1
    good = nb.net_desc(128, 1)
    assert l.nsb_create(ctypes.byref(h), 0, 0, 1, ctypes.byref(good)) == -1
    assert l.nsb_create(ctypes.byref(h), 0, 8, 0, ctypes.byref(good)) == -1
    # an unknown kernel override fails before any device query instead of running some other kernel
    monkeypatch.delenv("NSB_TRUNK256", raising=False)
    for value in ("mc2", "mc4", "ts", "bogus", ""):
        monkeypatch.setenv("NSB_TRUNK128", value)
        assert l.nsb_create(ctypes.byref(h), 0, 8, 1, ctypes.byref(good)) == -1, value
        err = l.nsb_last_error()
        assert b"NSB_TRUNK128" in err and b"classic" in err and b"duo" in err and b"quad" in err, err
    monkeypatch.delenv("NSB_TRUNK128")
    monkeypatch.setenv("NSB_TRUNK256", "bogus")
    assert l.nsb_create(ctypes.byref(h), 0, 8, 1, ctypes.byref(nb.net_desc(256, 1))) == -1
    err = l.nsb_last_error()
    assert b"NSB_TRUNK256" in err and b"single" in err, err
    assert l.nsb_await(None, 0) == -1 and b"null ctx" in l.nsb_last_error()
