"""CPU tests (-m "not gpu"): the oracle against the committed golden vectors (made from the
reference's own kernels by tests/golden/make_golden.py), against the reference kernels' outputs
for seeded random inputs (digests by tests/golden/make_reference_golden.py), and the reference's own
round-trip properties (SURVEY.md section 4)."""
import os

import numpy as np
import pytest

import oracle_lib as O
import oracle_pipeline as P
import reference_golden as RG
import grok_b200 as G

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ht_gold():
    return np.load(os.path.join(GOLD, "ht_blocks.npz"))


@pytest.fixture(scope="module")
def dwt_gold():
    return np.load(os.path.join(GOLD, "dwt_cases.npz"))


def test_ht_encoder_matches_reference_golden(ht_gold):
    for i in range(int(ht_gold["count"])):
        sm, kmax = ht_gold["in%03d" % i], int(ht_gold["kmax%03d" % i])
        assert np.array_equal(O.ht_encode(sm, kmax), ht_gold["out%03d" % i]), i


def test_ht_decoder_matches_reference_golden(ht_gold):
    for i in range(int(ht_gold["count"])):
        sm, kmax = ht_gold["in%03d" % i], int(ht_gold["kmax%03d" % i])
        h, w = sm.shape
        rc, dec = O.ht_decode(ht_gold["out%03d" % i], kmax, w, h)
        assert rc == 0
        assert np.array_equal(dec, ht_gold["dec%03d" % i]), i
        # and the decoded word is sign | (2*mu+1) << (p-1)  (ojph_block_decoder32.cpp L1130-1136)
        mu = (sm & 0x7FFFFFFF) >> (30 - kmax)
        want = np.where(mu > 0, (sm & 0x80000000) | ((2 * mu.astype(np.uint64) + 1) << (29 - kmax)), 0).astype(np.uint32)
        assert np.array_equal(dec, want), i


def test_dwt_forward_matches_reference_golden(dwt_gold):
    L = O.lib()
    for i in range(int(dwt_gold["count"])):
        x0, y0, w, h, numres = (int(v) for v in dwt_gold["geom%d" % i])
        a = np.ascontiguousarray(dwt_gold["src%d" % i]).copy()
        L.orc_dwt53_fwd_2d(a, w, x0, y0, x0 + w, y0 + h, numres)
        assert np.array_equal(a, dwt_gold["dwt53_%d" % i]), i
        f = np.ascontiguousarray(dwt_gold["src%d" % i].astype(np.float32))
        L.orc_dwt97_fwd_2d(f, w, x0, y0, x0 + w, y0 + h, numres)
        assert np.array_equal(f.view(np.int32), dwt_gold["dwt97_%d" % i].view(np.int32)), i  # bit exact


def live_cases():
    """The seeded code blocks and tiles of test_oracle_vs_reference_live (also what the reference was given)."""
    rng = np.random.default_rng(11)
    blocks, tiles = [], []
    for _ in range(60):
        w = int(rng.choice([1, 2, 3, 5, 8, 31, 32, 33, 64, 100]))
        h = int(rng.choice([1, 2, 3, 4, 17, 32, 40]))
        kmax = int(rng.integers(1, 20))
        lim = (1 << kmax) - 1
        c = np.clip((rng.standard_normal((h, w)) * rng.choice([0, 2, 40, lim])).astype(np.int64), -lim, lim)
        blocks.append((O.to_sgnmag(c, kmax), kmax))
    for _ in range(30):
        x0, y0 = int(rng.integers(0, 9)), int(rng.integers(0, 9))
        w, h = int(rng.integers(1, 90)), int(rng.integers(1, 70))
        numres = int(rng.integers(1, 7))
        src = rng.integers(-4096, 4096, (h, w))
        fsrc = rng.integers(-4096, 4096, (h, w)).astype(np.float32)
        tiles.append(((x0, y0, w, h, numres), src, fsrc))
    return blocks, tiles


def dwt_fwd_aligned(fn, src, x0, y0, numres, *extra):
    """Forward DWT of `src` in place in a 64-byte aligned, padded tile buffer (the reference's SIMD kernels
    need one); returns the transformed (h, w) window."""
    h, w = src.shape
    stride = ((w + 15) // 16) * 16 + 16
    a = O.aligned_zeros((h + 2, stride), src.dtype)
    a[:h, :w] = src
    fn(a, stride, x0, y0, x0 + w, y0 + h, numres, *extra)
    return a[:h, :w]


def test_oracle_vs_reference_live():
    """HT encode / decode and both forward DWTs of seeded random blocks and tiles equal what the reference's own
    kernels (every SIMD variant they have) computed from the same inputs."""
    want = RG.digests()["oracle"]
    blocks, tiles = live_cases()
    L = O.lib()
    for i, (sm, kmax) in enumerate(blocks):
        h, w = sm.shape
        ours = O.ht_encode(sm, kmax)
        enc = [d for d in want["ht_encode"][i] if d is not None]
        assert enc and all(RG.sha(ours) == d for d in enc), i
        rc, d = O.ht_decode(ours, kmax, w, h)
        for rc2, d2 in want["ht_decode"][i]:
            if rc2 != -2:
                assert rc == 0 and rc2 == 0 and RG.sha(d) == d2, i
    for i, ((x0, y0, w, h, numres), src, fsrc) in enumerate(tiles):
        a = dwt_fwd_aligned(L.orc_dwt53_fwd_2d, src.astype(np.int32), x0, y0, numres)
        f = dwt_fwd_aligned(L.orc_dwt97_fwd_2d, fsrc, x0, y0, numres)
        assert [RG.sha(a), RG.sha(f.view(np.int32))] == want["dwt"][i], i


def test_reversible_exponents_known_answer():
    """SURVEY.md appendix A: `grk_dump` of config 1 (8-bit grey, 5 levels, HT) prints these."""
    cp = G.make_coding(512, 512, 1, 8, numres=6)
    expn, mant = P.quant_tables(cp)
    assert list(expn) == [10, 11, 11, 12, 11, 11, 12, 11, 11, 12, 11, 11, 11, 10, 10, 11]
    assert not mant.any()


def test_53_perfect_reconstruction_odd_geometry():
    """GrkShortTileRoundTripTest / GrkInt32Reversible53Test: any geometry round-trips exactly."""
    rng = np.random.default_rng(5)
    L = O.lib()
    for _ in range(80):
        x0, y0 = int(rng.integers(0, 12)), int(rng.integers(0, 12))
        w, h = int(rng.integers(1, 70)), int(rng.integers(1, 70))
        numres = int(rng.integers(1, 8))
        a = rng.integers(-(1 << 17), 1 << 17, (h, w)).astype(np.int32)
        b = a.copy()
        L.orc_dwt53_fwd_2d(b, w, x0, y0, x0 + w, y0 + h, numres)
        L.orc_dwt53_inv_2d(b, w, x0, y0, x0 + w, y0 + h, numres)
        assert np.array_equal(a, b)


def test_97_round_trip_within_two_codes():
    """GrkIrreversibleLiftingTest.cpp L26-28: 9/7 pattern round trip <= 2 codes.  The inverse
    consumes the decoder's convention (high bands carry half the encoder's gain per axis:
    TileProcessor.cpp L398-404), which dequantisation normally supplies."""
    rng = np.random.default_rng(6)
    L = O.lib()
    for _ in range(20):
        x0, y0 = int(rng.integers(0, 5)), int(rng.integers(0, 5))
        w, h = int(rng.integers(2, 80)), int(rng.integers(2, 80))
        numres = int(rng.integers(2, 6))
        a = rng.integers(0, 4096, (h, w)).astype(np.float32)
        b = a.copy()
        L.orc_dwt97_fwd_2d(b, w, x0, y0, x0 + w, y0 + h, numres)
        # undo the encoder-side band gains
        for blk in O.enumerate_blocks((x0, y0, x0 + w, y0 + h), numres, 10, 10):
            g = [1.0, 0.5, 0.5, 0.25][blk.orient]
            b[blk.buf_y:blk.buf_y + blk.y1 - blk.y0, blk.buf_x:blk.buf_x + blk.x1 - blk.x0] *= g
        L.orc_dwt97_inv_2d(b, w, x0, y0, x0 + w, y0 + h, numres)
        assert np.abs(a - b).max() <= 2.0


def test_rct_round_trip_and_ict_tolerance():
    rng = np.random.default_rng(8)
    L = O.lib()
    n = 4096
    r, g, b = (rng.integers(0, 4096, n).astype(np.int32) for _ in range(3))
    sh = np.array([-2048] * 3, np.int32)
    y, u, v = r.copy(), g.copy(), b.copy()
    L.orc_rct_fwd(y, u, v, n, sh)
    L.orc_rct_inv(y, u, v, n, -sh, np.zeros(3, np.int32), np.full(3, 4095, np.int32))
    assert np.array_equal(y, r) and np.array_equal(u, g) and np.array_equal(v, b)
    fy, fu, fv = (np.zeros(n, np.float32) for _ in range(3))
    L.orc_ict_fwd(r, g, b, fy, fu, fv, n, sh)
    r2, g2, b2 = (np.zeros(n, np.int32) for _ in range(3))
    L.orc_ict_inv(fy, fu, fv, r2, g2, b2, n, -sh, np.zeros(3, np.int32), np.full(3, 4095, np.int32))
    assert max(np.abs(r2 - r).max(), np.abs(g2 - g).max(), np.abs(b2 - b).max()) <= 1


def test_whole_tile_oracle_pipeline_round_trip():
    """config 1 shape: 512x512 8-bit grey, 5/3, 6 resolutions, HT, lossless (BASELINE.json configs[0])."""
    cp = G.make_coding(256, 192, 1, 8, numres=6)
    planes = P.synthetic_image(256, 192, 1, 8, 1234)
    coefs = P.forward(cp, planes)
    rects = P.tile_rects(cp)
    rebuilt = [np.zeros_like(c) for c in coefs]
    for t, c, b in P.enumerate_all(cp):
        if b.x1 == b.x0 or b.y1 == b.y0:
            continue
        data = P.encode_block(cp, coefs, rects[t], c, b)
        win = P.decode_block(cp, data, c, b)
        rebuilt[c][b.buf_y:b.buf_y + win.shape[0], b.buf_x:b.buf_x + win.shape[1]] = win
    assert np.array_equal(rebuilt[0], coefs[0])
    out = P.inverse(cp, rebuilt)
    assert np.array_equal(out[0], planes[0])


def test_ht_refinement_passes_match_reference_golden():
    """SigProp / MagRef (2- and 3-pass blocks, plain and stripe-causal): the oracle's restatement decodes
    the fixture streams to exactly what ojph_decode_codeblock32 returned for them, and the oracle's
    test-only refinement encoder still reproduces those streams from the decoded planes' source."""
    g = np.load(os.path.join(GOLD, "ht_refine.npz"))
    seen = set()
    for i in range(int(g["count"])):
        w, h, M, npass, len2, causal = (int(v) for v in g["meta%03d" % i])
        data = g["data%03d" % i]
        rc, dec = O.ht_decode_passes(data, len2, npass, M, w, h, causal=bool(causal))
        assert rc == 0
        assert np.array_equal(dec, g["dec%03d" % i]), i
        seen.add((npass, causal))
        # bin-centre convention after all three passes: every decoded sample carries the half bit at plane
        # p-2 and nothing below it (L1499, L1596-1599)
        p = 30 - M
        nz = dec != 0
        if npass == 3:
            assert np.all(((dec[nz] >> (p - 2)) & 1) == 1)
        assert np.all((dec[nz] & ((1 << (p - 2)) - 1)) == 0)
    assert seen == {(2, 0), (2, 1), (3, 0), (3, 1)}


def refine_cases():
    """The seeded blocks of test_ht_refinement_vs_reference_live: (w, h, missing MSBs, sign-magnitude samples)."""
    rng = np.random.default_rng(77)
    for _ in range(60):
        w, h = int(rng.integers(1, 65)), int(rng.integers(1, 65))
        M = int(rng.integers(8, 28))
        p = 30 - M
        nb = int(rng.integers(1, p + 3))
        mag = rng.integers(0, 1 << nb, (h, w)).astype(np.uint64) * (rng.random((h, w)) < rng.choice([0.05, 0.4, 1.0]))
        mag = np.minimum(mag, (1 << (31 - (p - 1))) - 1)
        v = (mag << np.uint64(p - 1)).astype(np.uint32)
        sm = np.where(v != 0, v | (rng.integers(0, 2, (h, w)).astype(np.uint32) << 31), 0).astype(np.uint32)
        yield w, h, M, sm


def refine_stream(sm, M, npass, causal):
    """cleanup + refinement segments of one block, and the refinement segment's length"""
    seg = O.ht_encode_refine(sm, M, npass, causal)
    return np.concatenate([O.ht_encode(sm, M), seg]), len(seg)


def test_ht_refinement_vs_reference_live():
    """2- and 3-pass streams of seeded blocks: the oracle decodes them to what the reference's decoder made of the
    same streams."""
    want = RG.digests()["refine"]
    for trial, (w, h, M, sm) in enumerate(refine_cases()):
        p = 30 - M
        for npass in (2, 3):
            for causal in (False, True):
                data, len2 = refine_stream(sm, M, npass, causal)
                rc1, a = O.ht_decode_passes(data, len2, npass, M, w, h, causal=causal)
                assert rc1 == 0 and [RG.sha(data), RG.sha(a)] == want[trial]["%d%d" % (npass, causal)], (trial, npass, causal)
                if npass == 3:   # cleanup-significant samples are exact down to plane p-1
                    m = sm & 0x7FFFFFFF
                    cs = (m >> p) != 0
                    want_a = ((m >> (p - 1)) << (p - 1)) | (1 << (p - 2)) | (sm & 0x80000000)
                    assert np.array_equal(a[cs], want_a[cs])
