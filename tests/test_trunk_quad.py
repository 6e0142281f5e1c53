"""trunk_quad_kernel: the 128-channel trunk with four positions per CTA (two groups of two, each with the duo kernel's
layout) and one CTA per SM, launched by unforced 128-channel contexts with >= 4 slots.

Both kernels are instances of one body in csrc/trunk_tmem.cu (one and two position groups per CTA), and every
accumulator of the quad kernel receives exactly the MMA sequence of trunk_duo_kernel (layer, K block, tap, step,
same accumulate flags), so the two kernels must agree bit for bit on every output of every entry point; around that,
the depth tolerances of test_depth_parity.py against the oracle at config 2, batch invariance at B = 4,096, the paths
that touch the kernel's work list and I/O, and the kernel choice per slot count."""
import re
import subprocess

import numpy as np
import pytest

import helpers
import test_depth_parity as depth
import test_evalcache
import test_gpu_parity as parity

QUAD = "trunk_quad_kernel (128 ch, 4 positions per CTA, weights via TMEM, 1 CTA per SM)"


def _u32(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_quad_kernel_is_in_the_product_library(nb):
    sass = subprocess.run(["cuobjdump", "-sass", nb.LIB_PATH], capture_output=True, text=True)
    if sass.returncode != 0 or not sass.stdout:
        pytest.skip("cuobjdump cannot read the library here")
    kernels = re.split(r"\n\s*Function : ", sass.stdout)
    quad = [k for k in kernels if k.split("\n", 1)[0].find("trunk_quad_kernel") >= 0]
    assert len(quad) == 1
    assert all(op in quad[0] for op in ("UTCHMMA", "STTM", "LDTM"))


# ---- GPU: bit-identity with the duo kernel -----------------------------------------------------------------------
def _outputs(nb, orc, synth, monkeypatch, force, n, paths):
    """Every output of the entry points in `paths` for n positions on a 2-slot context forced to `force`."""
    monkeypatch.setenv("NSB_TRUNK128", force)
    monkeypatch.delenv("NSB_IO", raising=False)
    desc = nb.net_desc(128, 10)
    blob = nb.random_blob(desc, 1)
    pos = synth.random_positions(n, seed=500 + n)
    fb = orc.pack(pos)
    off, idx = synth.random_legal_moves(n, seed=600 + n, edge_rows=n >= 4)
    total = int(off[-1])
    out = {}
    with nb.Context(desc, batch_max=n, slots=2, blob=blob) as ctx:
        assert ctx.trunk_kernel_name().startswith("trunk_quad_kernel" if force == "quad" else "trunk_duo_kernel")
        policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
        win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
        ctx.eval_async(0, fb, n, policy, win, draw)
        ctx.await_(0)
        out["dense"] = (policy, win, draw)
        legal, flag = np.zeros(total, dtype=np.float32), np.full(n, 7, dtype=np.uint8)
        w2, d2 = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
        ctx.eval_decode_async(1, fb, n, off, idx, nb.DECODE_PROBS, legal, w2, d2, flag)
        ctx.await_(1)
        out["decode"] = (legal, w2, d2, flag)
        if "positions" in paths:   # packed positions in, DECODE_BOTH with raw logits beside the probabilities, rank order
            legal, logits, order = np.zeros(total, np.float32), np.zeros(total, np.float32), np.zeros(total, np.uint16)
            w3, d3, f3 = np.zeros(n, np.float32), np.zeros(n, np.float32), np.full(n, 7, np.uint8)
            ctx.eval_request_async(0, n, off, idx, nb.DECODE_BOTH, legal, w3, d3, positions=pos, order_out=order,
                                   nan_flag=f3, logits_out=logits)
            ctx.await_(0)
            out["positions_both_ranked"] = (legal, logits, order, w3, d3, f3)
        if "direct" in paths:      # the kernel reads and writes the caller's page-locked buffers itself
            P = nb.PinnedArray
            h = [P((n,), nb.POSITION), P((n + 1,), np.uint32), P((total,), np.uint16), P((total,), np.float32),
                 P((n,), np.float32), P((n,), np.float32), P((n,), np.uint8)]
            h[0].array[:], h[1].array[:], h[2].array[:] = pos, off, idx
            ctx.set_io_mode(True)
            ctx.eval_positions_decode_async(1, h[0].array, n, h[1].array, h[2].array, nb.DECODE_PROBS, h[3].array, h[4].array,
                                            h[5].array, h[6].array)
            ctx.await_(1)
            ctx.set_io_mode(False)
            out["direct"] = tuple(x.array.copy() for x in h[3:])
            for x in h:
                x.free()
        if "cached" in paths:      # behind a cache probe: the trunk runs on the miss list
            ctx.cache_create(4)
            hashes = np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(99)
            hits = out["cached_hits"] = []   # which rows hit depends on store timing (a contended bundle skips the store)
            for rep in range(2):
                legal, w4, d4 = np.zeros(total, np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
                f4, hit = np.full(n, 7, np.uint8), np.zeros(n, np.uint8)
                sel = slice(0, n // 2 + 1) if rep == 0 else slice(0, n)   # second call: half hits, half misses
                m = len(range(n)[sel])
                o = off[: m + 1]
                ctx.eval_cached_decode_async(0, np.ascontiguousarray(fb[: m * 86]), m, np.ascontiguousarray(hashes[:m]), o,
                                             idx[: int(o[-1])], nb.DECODE_PROBS, legal[: int(o[-1])], w4[:m], d4[:m], f4[:m],
                                             hit[:m])
                ctx.await_(0)
                out[f"cached{rep}"] = (legal, w4, d4, f4)
                hits.append(hit)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 5, 256, 1000, 4096])
def test_bit_identical_to_duo_kernel(nb, orc, synth, monkeypatch, n):
    """Dense logits, decoded legal rows, win, draw and NaN flags; n = 1, 3, 5 leave positions of the last CTA empty,
    1,000 and 4,096 take several passes per CTA.  At n = 5 and 1,000 also packed positions with DECODE_BOTH and the rank
    order, direct host I/O, and the cached path (misses only, then a mix of hits and misses)."""
    paths = ("positions", "direct", "cached") if n in (5, 1000) else ()
    want = _outputs(nb, orc, synth, monkeypatch, "duo", n, paths)
    got = _outputs(nb, orc, synth, monkeypatch, "quad", n, paths)
    assert want.keys() == got.keys()
    hits = got.pop("cached_hits", None)
    want.pop("cached_hits", None)
    for key in want:
        for i, (w, g) in enumerate(zip(want[key], got[key])):
            assert np.array_equal(_u32(w), _u32(g)), (n, key, i)
    assert np.all(np.isfinite(got["dense"][0])) and got["dense"][1].min() > 0 and not got["decode"][3].any()
    if hits:   # the second cached call found rows of the first in the cache and evaluated the rest
        assert hits[1].any() and not hits[1][n // 2 + 1:].any()


# ---- GPU: against the oracle, batch invariance ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [256, 5])
def test_config2_depth_parity_vs_oracle(nb, orc, synth, monkeypatch, n):
    """Config 2 (10 x 128, seed 1) on an unforced 4-slot context - the kernel the benchmark's pipeline launches -
    with test_depth_parity.py's metrics and tolerances against the fp32 and bf16-emulating oracles."""
    monkeypatch.delenv("NSB_TRUNK128", raising=False)
    desc = nb.net_desc(128, 10)
    blob = nb.random_blob(desc, 1)
    pos = synth.random_positions(n, seed=2024)
    fb = orc.pack(pos)
    off, idx = synth.random_legal_moves(n, seed=3, edge_rows=False)
    legal = np.zeros(int(off[-1]), dtype=np.float32)
    w2, d2 = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    with nb.Context(desc, batch_max=n, slots=4, blob=blob) as ctx:
        assert ctx.trunk_kernel_name() == QUAD
        policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
        win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
        ctx.eval_async(0, fb, n, policy, win, draw)
        ctx.await_(0)
        ctx.eval_positions_decode_async(3, pos, n, off, idx, nb.DECODE_PROBS, legal, w2, d2, None)
        ctx.await_(3)
    m = helpers.drift_metrics(nb, orc, desc, blob, fb, n, (policy, win, draw), off, idx)
    assert m["win_spread_fp32"] > 1e-2, ("dead value head: pick another seed", m)
    depth._check(m, f"10x128@{n}:quad")
    want, _ = orc.decode(policy, win, draw, off, idx, nb.DECODE_PROBS)
    assert np.allclose(legal, want, rtol=1e-6, atol=1e-9) and np.array_equal(w2, win) and np.array_equal(d2, draw)


@pytest.mark.gpu
def test_full_size_batch_invariance_quad(nb, orc, synth, monkeypatch):
    """B = 4,096 on the quad kernel: every row equals, bit for bit, the same position in a batch of 16, whichever CTA,
    pass and position group computed it."""
    parity.test_full_size_batch_invariance(nb, orc, synth, monkeypatch, 4096, "quad")


# ---- GPU: the paths that touch the kernel's work list and I/O, as test_gpu_parity.py / test_evalcache.py run them --
@pytest.mark.gpu
def test_packed_positions_equal_bitboards_quad(nb, orc, synth, monkeypatch):
    parity.test_stage1_fused_into_trunk_prologue(nb, orc, synth, monkeypatch, 128, 4)


@pytest.mark.gpu
def test_direct_io_equals_staged_quad(nb, orc, synth, monkeypatch):
    parity.test_direct_io_equals_staged(nb, orc, synth, monkeypatch, 128, 4)


@pytest.mark.gpu
def test_rank_order_of_decoded_rows_quad(nb, orc, synth, monkeypatch):
    parity.test_rank_order_of_decoded_rows(nb, orc, synth, monkeypatch, 128, 4)


@pytest.mark.gpu
def test_nan_semantics_quad(nb, orc, synth, monkeypatch):
    parity.test_nan_semantics_follow_feedworker(nb, orc, synth, monkeypatch, 128, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("direct", [False, True])
def test_cached_path_quad(nb, orc, synth, monkeypatch, direct):
    monkeypatch.setenv("NSB_TRUNK128", "quad")
    test_evalcache.test_eval_cached_serves_hits_and_evaluates_misses(nb, orc, synth, 128, direct)


# ---- GPU: which kernel a context launches -----------------------------------------------------------------------
@pytest.mark.gpu
def test_kernel_selection_by_slot_count(nb, monkeypatch):
    desc = nb.net_desc(128, 2)
    blob = nb.random_blob(desc, 3)

    def name(slots, force=None, batch_max=1024):
        if force:
            monkeypatch.setenv("NSB_TRUNK128", force)
        else:
            monkeypatch.delenv("NSB_TRUNK128", raising=False)
        with nb.Context(desc, batch_max=batch_max, slots=slots, blob=blob) as ctx:
            return ctx.trunk_kernel_name()

    assert name(4) == QUAD and name(8) == QUAD
    assert name(2).startswith("trunk_duo_kernel") and "2 CTAs per SM" in name(2) and name(3).startswith("trunk_duo_kernel")
    assert name(1).startswith("trunk_fused_kernel<128>") and "trunk_duo_kernel" in name(1)   # per-batch choice, unchanged
    assert name(1, "quad") == QUAD and name(2, "quad") == QUAD
    assert name(4, "duo").startswith("trunk_duo_kernel") and name(4, "classic") == "trunk_fused_kernel<128>"
