"""GPU parity tests (-m gpu): the CUDA engine, called through the C ABI, against the oracle on the
same seeded inputs -- bit-exact for the reversible path (integer / byte work), and for the
irreversible path bit-exact against the oracle's fp32 restatement plus the reference's own
accelerator tolerances against the source (GrkPluginMemoryTest.cpp L39-52)."""
import ctypes as C

import numpy as np
import pytest

import grok_b200 as G
import oracle_lib as O
import oracle_pipeline as P

pytestmark = pytest.mark.gpu

GEOMS = [
    dict(width=512, height=512, numcomps=1, prec=8),                                   # BASELINE config 1
    dict(width=2048, height=1024, numcomps=3, prec=12, tile=(1024, 1024)),              # config 2 tiles
    dict(width=333, height=217, numcomps=3, prec=12, numres=4, origin=(3, 5)),          # odd origin (SURVEY 8d)
    dict(width=100, height=75, numcomps=4, prec=16, numres=3, tile=(61, 40), cblk=(32, 32)),  # config 4 shape, ragged tiles
    dict(width=61, height=9, numcomps=1, prec=8, numres=6),                             # levels run out of samples
    dict(width=64, height=64, numcomps=3, prec=10, numres=3, tile=(1, 64)),             # 1-pixel-wide tiles
    dict(width=40, height=33, numcomps=1, prec=12, numres=2, tile=(7, 1), cblk=(4, 4)), # 1-pixel-high tiles
    dict(width=300, height=200, numcomps=3, prec=8, numres=5, tile=(128, 128), origin=(129, 65), tile_origin=(1, 1),
         cblk=(16, 128)),
    dict(width=700, height=500, numcomps=3, prec=12, numres=5, tile=(512, 256), origin=(5, 11), precincts=[(128, 128)]),  # many precincts
    dict(width=260, height=140, numcomps=3, prec=16, sgnd=True, numres=4, numgbits=2),                                   # signed 16 bit, 2 guard bits
    dict(width=2100, height=40, numcomps=1, prec=10, numres=2, cblk=(1024, 4)),                                           # widest code blocks
    dict(width=40, height=2100, numcomps=1, prec=10, numres=2, cblk=(4, 1024)),                                           # tallest code blocks
    dict(width=500, height=300, numcomps=3, prec=12, numres=3, cblk=(128, 32)),
    dict(width=300, height=500, numcomps=1, prec=9, numres=3, cblk=(32, 128), tile=(150, 250)),
    dict(width=700, height=90, numcomps=1, prec=8, numres=3, cblk=(256, 16)),
    dict(width=333, height=217, numcomps=3, prec=12, numres=1, origin=(3, 5), tile=(100, 90)),     # no wavelet level, ragged tiles
    dict(width=200, height=120, numcomps=4, prec=16, numres=1),
]


def _compare_blocks(cp, res, coefs):
    blks = P.enumerate_all(cp)
    rects = P.tile_rects(cp)
    assert len(blks) == res.num_blocks
    for i, (t, c, b) in enumerate(blks):
        if b.x1 == b.x0 or b.y1 == b.y0:
            assert res.blocks[i]["length"] == 0
            continue
        want = P.encode_block(cp, coefs, rects[t], c, b)
        assert np.array_equal(want, res.block_bytes(i)), "code block %d (res %d orient %d)" % (i, b.resno, b.orient)


@pytest.mark.parametrize("args", GEOMS)
def test_reversible_stage_parity(engine, args):
    cp = G.make_coding(**args)
    planes = P.synthetic_image(args["width"], args["height"], args["numcomps"], args["prec"], seed=42,
                               origin=args.get("origin", (0, 0)))
    if args.get("sgnd"):
        planes = [p - (1 << (args["prec"] - 1)) for p in planes]
    ref = P.forward(cp, planes)
    job = engine.job(cp)
    job.upload(planes)
    job.forward()
    got = [np.zeros_like(p) for p in planes]
    job.download_coeffs(got)
    for g, r in zip(got, ref):
        assert np.array_equal(g, r)                      # DC shift + RCT + 5/3, every level
    job.t1_encode()
    res = job.fetch_result()
    _compare_blocks(cp, res, ref)                        # HT cleanup bytes, block by block
    for p in got:
        p[:] = -1
    job.upload_coeffs(got)                               # poison, then decode back
    job.t1_decode()
    job.download_coeffs(got)
    for g, r in zip(got, ref):
        assert np.array_equal(g, r)
    job.inverse()
    rec = [np.zeros_like(p) for p in planes]
    job.download(rec)
    for g, r in zip(rec, planes):
        assert np.array_equal(g, r)                      # lossless
    res.free()
    job.close()


@pytest.mark.parametrize("kind", ["zero", "max_checkerboard", "min_max_stripes", "noise_full_range"])
def test_adversarial_content(engine, kind):
    """SURVEY.md 8d adversarial row, from the reference's own tests: all-zero, max-amplitude
    checkerboard, stripes, full-range noise."""
    w, h, prec = 200, 136, 12
    cp = G.make_coding(w, h, 3, prec, numres=5, tile=(128, 128))
    y, x = np.mgrid[0:h, 0:w]
    rng = np.random.default_rng(3)
    if kind == "zero":
        planes = [np.zeros((h, w), np.int32) for _ in range(3)]
    elif kind == "max_checkerboard":
        planes = [(((x + y + c) & 1) * 4095).astype(np.int32) for c in range(3)]
    elif kind == "min_max_stripes":
        planes = [(((x >> c) & 1) * 4095).astype(np.int32) for c in range(3)]
    else:
        planes = [rng.integers(0, 4096, (h, w)).astype(np.int32) for _ in range(3)]
    res = engine.encode(cp, planes)
    _compare_blocks(cp, res, P.forward(cp, planes))
    out = [np.zeros_like(p) for p in planes]
    engine.decode(cp, res.blocks.copy(), res.bytes.copy(), out)
    for a, b in zip(out, planes):
        assert np.array_equal(a, b)
    res.free()


def test_host_api_strided_planes_and_sharding(engine):
    """Row stride larger than the width (64-byte aligned strides, gpu_plugin_shared.h L540-544) and
    tile sharding (tile_mod/tile_rem): two half jobs produce exactly the blocks of the full job."""
    cp = G.make_coding(700, 300, 3, 12, numres=4, tile=(256, 128))
    planes = P.synthetic_image(700, 300, 3, 12, seed=5)
    padded = [np.zeros((300, 704), np.int32) for _ in range(3)]
    for p, q in zip(padded, planes):
        p[:, :700] = q
    views = [p[:, :700] for p in padded]
    full = engine.encode(cp, views)
    fb, fbytes = full.blocks.copy(), full.bytes.copy()
    full.free()
    for rem in (0, 1):
        part = engine.encode(cp, views, tile_mod=2, tile_rem=rem)
        sel = np.nonzero(fb["tile"] % 2 == rem)[0]
        assert len(sel) == part.num_blocks
        for j, i in enumerate(sel):
            a = fbytes[int(fb[i]["offset"]):int(fb[i]["offset"]) + int(fb[i]["length"])]
            assert np.array_equal(a, part.block_bytes(j))
        part.free()


def test_irreversible_path(engine):
    """BASELINE config 3 shape (ICT + 9/7 + quantisation + HT, one tile, 5 levels, 64x64 blocks) at a
    size the oracle handles: forward coefficients and coded bytes bit-exact vs the oracle's fp32
    restatement; decode within the reference's accelerator tolerances vs the source:
    lossy 12-bit: <= 16 codes, PSNR > 50 dB (GrkPluginMemoryTest.cpp L39-52)."""
    w, h = 640, 384
    cp = G.make_coding(w, h, 3, 12, numres=6, irreversible=True)
    planes = P.synthetic_image(w, h, 3, 12, seed=20260925)
    ref = P.forward(cp, planes)
    job = engine.job(cp)
    job.upload(planes)
    job.forward()
    got = [np.zeros_like(p) for p in planes]
    job.download_coeffs(got)
    for c, (g, r) in enumerate(zip(got, ref)):
        assert np.array_equal(g, r), "9/7 + ICT coefficients of component %d are not bit-identical" % c
    job.t1_encode()
    res = job.fetch_result()
    _compare_blocks(cp, res, ref)
    job.t1_decode()
    job.download_coeffs(got)
    # dequantised coefficients: bit-exact vs the oracle's decode of the same bytes
    rects = P.tile_rects(cp)
    for i, (t, c, b) in enumerate(P.enumerate_all(cp)):
        if b.x1 == b.x0 or b.y1 == b.y0:
            continue
        win = P.decode_block(cp, res.block_bytes(i), c, b)
        sub = got[c][b.buf_y:b.buf_y + win.shape[0], b.buf_x:b.buf_x + win.shape[1]]
        assert np.array_equal(sub, win)
    job.inverse()
    rec = [np.zeros_like(p) for p in planes]
    job.download(rec)
    ref_rec = P.inverse(cp, got)
    for g, r, s in zip(rec, ref_rec, planes):
        assert np.abs(g - r).max() <= 1          # device vs host inverse wavelet: <= 2 codes (GrkPluginBatchMemoryTest.cpp L35-45)
        err = (g - s).astype(np.float64)
        assert np.abs(err).max() <= 16
        psnr = 10 * np.log10(4095.0 ** 2 / max(1e-12, (err ** 2).mean()))
        assert psnr > 50.0
    res.free()
    job.close()


def test_config2_full_size_properties(engine):
    """BASELINE config 2 at full size (8192x8192x3, 12 bit, 1024 tiles): size-independent
    properties -- lossless encode->decode round trip through the host API, block table sanity --
    plus byte parity with the oracle on two whole tiles."""
    W = H = 8192
    cp = G.make_coding(W, H, 3, 12, numres=6, tile=(1024, 1024))
    rng = np.random.default_rng(20260924)
    # cheap full-size synthetic: per-tile copies of one generated tile with a per-tile offset
    base = P.synthetic_image(1024, 1024, 3, 12, seed=20260924)
    planes = [np.empty((H, W), np.int32) for _ in range(3)]
    for ty in range(8):
        for tx in range(8):
            off = int(rng.integers(0, 512))
            for c in range(3):
                planes[c][ty * 1024:(ty + 1) * 1024, tx * 1024:(tx + 1) * 1024] = (base[c] + off) % 4096
    res = engine.encode(cp, planes)
    assert res.num_blocks == 49728
    lens = res.blocks["length"].astype(np.int64)
    assert lens.sum() == res.num_bytes and (lens > 0).all()
    assert np.array_equal(res.blocks["offset"], np.concatenate([[0], np.cumsum(lens)[:-1]]))
    # oracle parity on tiles 0 and 37
    for t in (0, 37):
        ty, tx = divmod(t, 8)
        sub = [np.ascontiguousarray(p[ty * 1024:(ty + 1) * 1024, tx * 1024:(tx + 1) * 1024]) for p in planes]
        cpt = G.make_coding(1024, 1024, 3, 12, numres=6, origin=(tx * 1024, ty * 1024))
        coefs = P.forward(cpt, sub)
        idx = np.nonzero(res.blocks["tile"] == t)[0]
        blks = P.enumerate_all(cpt)
        assert len(idx) == len(blks)
        for i, (_, c, b) in zip(idx, blks):
            want = P.encode_block(cpt, coefs, (tx * 1024, ty * 1024, 0, 0), c, b)
            assert np.array_equal(want, res.block_bytes(int(i)))
    out = [np.zeros_like(p) for p in planes]
    engine.decode(cp, res.blocks.copy(), res.bytes.copy(), out)
    for a, b in zip(out, planes):
        assert np.array_equal(a, b)
    res.free()


# ---- the stock plugin symbols ----------------------------------------------------------------
from gpup_ctypes import (GpupImageComp, GpupImage, GpupPass, GpupCodeBlock, GpupPrecinct, GpupBand, GpupResolution,  # noqa: E402
                         GpupTileComponent, GpupTile)


def test_stock_gpup_encode_mem(engine):
    """The unmodified host path: gpup_encode_mem(params, image, &tile) on config 1 (single tile),
    tree walked in Grok's order (plugin_bridge.cpp L62-111) and compared with the oracle."""
    assert C.sizeof(GpupCodeBlock) == 1672
    lib = G.lib()
    w = h = 512
    cp = G.make_coding(w, h, 1, 8, numres=6)
    planes = P.synthetic_image(w, h, 1, 8, seed=1234)
    params = (C.c_uint8 * 12696)()
    # fields at the offsets of gpup_compress_params (checked by tests/test_host.py against the header)
    def put(off, val, typ):
        typ.from_buffer(params, off).value = val
    import re, subprocess, os
    probe = r'''
#include <stdio.h>
#include <stddef.h>
#include "grok_b200.h"
#define O(f) printf(#f " %zu\n", offsetof(gpup_compress_params, f));
int main(void){ O(numlayers) O(csty) O(numgbits) O(numresolution) O(cblockw_init) O(cblockh_init) O(cblk_sty) O(irreversible) O(roi_compno) O(mct) return 0; }'''
    exe = "/tmp/b2k_off_%d" % os.getpid()
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(os.path.dirname(G._HERE), "include"), "-o", exe],
                   input=probe.encode(), check=True)
    off = dict((k, int(v)) for k, v in (l.split() for l in subprocess.check_output([exe]).decode().splitlines()))
    put(off["numlayers"], 1, C.c_uint16)
    put(off["numgbits"], 1, C.c_uint8)
    put(off["numresolution"], 6, C.c_uint8)
    put(off["cblockw_init"], 64, C.c_uint32)
    put(off["cblockh_init"], 64, C.c_uint32)
    put(off["cblk_sty"], 0x40, C.c_uint8)
    put(off["roi_compno"], -1, C.c_int32)
    comp = GpupImageComp(0, 0, w, w, h, 1, 1, 8, False, planes[0].ctypes.data_as(C.POINTER(C.c_int32)), False)
    img = GpupImage(0, 0, w, h, 1, 3, C.pointer(comp))
    tile = C.POINTER(GpupTile)()
    lib.gpup_encode_mem.argtypes = [C.c_void_p, C.POINTER(GpupImage), C.POINTER(C.POINTER(GpupTile))]
    rc = lib.gpup_encode_mem(params, C.byref(img), C.byref(tile))
    assert rc == 0, lib.b2k_last_error()
    coefs = P.forward(cp, planes)
    blks = [x for x in P.enumerate_all(cp)]
    T = tile.contents
    assert T.numComponents == 1
    tc = T.tileComponents[0].contents
    assert tc.numResolutions == 6
    k = 0
    for r in range(6):
        res = tc.resolutions[r].contents
        assert res.numBands == (1 if r == 0 else 3)
        for b in range(res.numBands):
            band = res.band[b].contents
            assert band.orientation == (0 if r == 0 else b + 1)
            for p in range(band.numPrecincts):
                prc = band.precincts[p].contents
                for j in range(prc.numBlocks):
                    cb = prc.blocks[j].contents
                    _, c, ob = blks[k]
                    k += 1
                    assert (cb.x0, cb.y0, cb.x1, cb.y1) == (ob.x0, ob.y0, ob.x1, ob.y1)
                    assert cb.numPasses == 1 and cb.numBitPlanes == 1
                    want = P.encode_block(cp, coefs, (0, 0, w, h), 0, ob)
                    have = np.ctypeslib.as_array(cb.compressedData, shape=(cb.compressedDataLength,))
                    assert np.array_equal(want, have)
                    assert cb.passes[0].rate == cb.compressedDataLength - 1
    assert k == len(blks)
    lib.gpup_tile_free(tile)


@pytest.mark.parametrize("sgnd", [False, True])
def test_16bit_containers(engine, sgnd):
    """b2k_encode16 / b2k_decode16 (cf. gpup_batch_memory_submit_planes: 16-bit sample containers):
    identical code blocks to the 32-bit entry point, lossless round trip into 16-bit planes."""
    w, h, prec = 600, 300, 12
    cp = G.make_coding(w, h, 3, prec, sgnd=sgnd, numres=5, tile=(256, 128), origin=(8, 0))
    planes = P.synthetic_image(w, h, 3, prec, seed=77)
    if sgnd:
        planes = [p - 2048 for p in planes]
    p16 = [p.astype(np.int16 if sgnd else np.uint16) for p in planes]
    a = engine.encode(cp, planes)
    b = engine.encode(cp, p16)
    assert a.num_blocks == b.num_blocks and np.array_equal(a.blocks["length"], b.blocks["length"])
    assert np.array_equal(a.bytes, b.bytes)
    out = [np.zeros_like(p) for p in p16]
    engine.decode(cp, b.blocks.copy(), b.bytes.copy(), out)
    for x, y in zip(out, p16):
        assert np.array_equal(x, y)
    a.free()
    b.free()


@pytest.mark.parametrize("case", [
    dict(w=600, h=300, n=3, tile=(256, 128), origin=(8, 0), sgnd=False, pad=0),    # tiled: partial-width runs, 2-D copies
    dict(w=501, h=77, n=3, tile=None, origin=(0, 0), sgnd=False, pad=5),           # rows not 16-byte aligned, padded stride
    dict(w=640, h=256, n=4, tile=None, origin=(0, 0), sgnd=True, pad=0),
    dict(w=333, h=64, n=1, tile=None, origin=(0, 0), sgnd=False, pad=0),
])
def test_interleaved_16bit_frames(engine, case):
    """b2k_encode16_interleaved (RGB48LE rows / gpup_batch_memory_submit's packed frames, grok.cpp L1806-1836): the frame
    crosses PCIe pixel-interleaved and is split into planes on the device; code blocks equal the planar entry point's."""
    w, h, n, prec = case["w"], case["h"], case["n"], 12
    cp = G.make_coding(w, h, n, prec, sgnd=case["sgnd"], numres=5, tile=case["tile"], origin=case["origin"])
    planes = P.synthetic_image(w, h, n, prec, seed=5)
    if case["sgnd"]:
        planes = [p - 2048 for p in planes]
    dt = np.int16 if case["sgnd"] else np.uint16
    buf = np.zeros((h, w * n + case["pad"]), dt)
    pixels = buf[:, :w * n].reshape(h, w, n) if case["pad"] == 0 else np.lib.stride_tricks.as_strided(
        buf, shape=(h, w, n), strides=(buf.strides[0], 2 * n, 2))
    for c in range(n):
        pixels[:, :, c] = planes[c].astype(dt)
    a = engine.encode(cp, planes)
    b = engine.encode_interleaved(cp, pixels)
    assert a.num_blocks == b.num_blocks and np.array_equal(a.blocks["length"], b.blocks["length"])
    assert np.array_equal(a.bytes, b.bytes)
    a.free()
    b.free()


@pytest.mark.parametrize("args", [
    dict(width=2048, height=1536, numcomps=3, prec=12, numres=6, tile=(512, 512)),
    dict(width=1000, height=700, numcomps=3, prec=12, numres=5, tile=(256, 256), origin=(17, 9), irreversible=True),
    dict(width=333, height=217, numcomps=1, prec=8, numres=4),                      # fewer blocks than one range
])
@pytest.mark.parametrize("shape", [(0, 0), (3, 2), (16, 8), (5, 1)])
def test_pipelined_round_trip_matches_the_sequential_one(engine, args, shape):
    """b2k_job_roundtrip_pipelined_n (block-coder stage cut into block ranges on side streams) against
    b2k_job_roundtrip_n: identical coded bytes and block lengths, identical pixels back."""
    cp = G.make_coding(**args)
    planes = P.synthetic_image(args["width"], args["height"], args["numcomps"], args["prec"], seed=31)
    job = engine.job(cp)
    job.upload(planes)
    job.roundtrip_n(1)
    a = job.fetch_result()
    ref_bytes, ref_len = a.bytes.copy(), a.blocks["length"].copy()
    a.free()
    ref_px = [np.zeros_like(p) for p in planes]
    job.download(ref_px)
    job.upload(planes)
    # a second lossy round trip would start from the first one's pixels: one step for 9/7
    _, stage, _, nbytes = job.roundtrip_pipelined_n(1 if args.get("irreversible") else 3, *shape)
    b = job.fetch_result()
    assert nbytes == ref_bytes.size and np.array_equal(b.blocks["length"], ref_len) and np.array_equal(b.bytes, ref_bytes)
    b.free()
    px = [np.zeros_like(p) for p in planes]
    job.download(px)
    for x, y in zip(px, ref_px):
        assert np.array_equal(x, y)
    if not args.get("irreversible"):
        for x, y in zip(px, planes):
            assert np.array_equal(x, y)
    job.close()


def _mock_host():
    import os
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    so = "/tmp/b2k_mock_host_%d.so" % os.getpid()
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", os.path.join(os.path.dirname(here), "grok_b200", "csrc"),
                    os.path.join(here, "mock_host.cpp"), "-o", so], check=True)
    return C.CDLL(so)


@pytest.mark.parametrize("irreversible", [False, True])
def test_stock_plugin_decompress_protocol(engine, irreversible):
    """plugin_decompress(): the HEADER -> T2 -> POST_T1 -> CLEAN callback protocol against a mock of
    Grok's host side (tests/mock_host.cpp) fed with this engine's own coded blocks.  Reversible: pixels
    equal the source; irreversible: equal to b2k_decode's.  A block claiming refinement passes must be
    handed back as "not handled" (1), never mis-decoded."""
    w, h = 320, 200
    cp = G.make_coding(w, h, 3, 12, numres=5, irreversible=irreversible)
    planes = P.synthetic_image(w, h, 3, 12, seed=99)
    res = engine.encode(cp, planes)
    blocks, data = res.blocks.copy(), res.bytes.copy()
    res.free()
    ref_out = [np.zeros_like(p) for p in planes]
    engine.decode(cp, blocks, data, ref_out)
    steps = []
    for c in range(3):
        for r in range(cp.numres):
            for b in range(1 if r == 0 else 3):
                steps.append(P.band_params(cp, r, 0 if r == 0 else b + 1)[2])
    steps = np.array(steps, np.float32)
    M = _mock_host()
    lib = G.lib()
    fn = C.cast(lib.plugin_decompress, C.c_void_p)
    out = [np.zeros((h, w), np.int32) for _ in range(3)]
    outp = (C.c_void_p * 3)(*[o.ctypes.data for o in out])
    strides = (C.c_uint32 * 3)(w, w, w)
    phases = C.c_int(0)
    M.mock_host_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int, C.POINTER(C.c_int)]
    rc = M.mock_host_run(fn, C.byref(cp), blocks.ctypes.data, len(blocks), data.ctypes.data, steps.ctypes.data, outp, strides, 0,
                         C.byref(phases))
    assert rc == 0 and phases.value == 15, (rc, phases.value, lib.b2k_last_error())
    for a, b, s in zip(out, ref_out, planes):
        assert np.array_equal(a, b)
        if not irreversible:
            assert np.array_equal(a, s)
    rc = M.mock_host_run(fn, C.byref(cp), blocks.ctypes.data, len(blocks), data.ctypes.data, steps.ctypes.data, outp, strides, 1,
                         C.byref(phases))
    assert rc == 1 and (phases.value & 4) == 0   # declined before POST_T1, CLEAN still delivered
    assert phases.value & 8


def _refined_blocks(cp, coefs, npass, dropped, seed):
    """Foreign-style HT streams for every block of `cp`: cleanup pass `dropped` bit-planes above the
    LSB + SigProp (+ MagRef) for the next plane, made by the oracle's encoders; returns the block
    table, the byte arena and the oracle's decode of it (dequantised coefficient planes)."""
    L = O.lib()
    blks = P.enumerate_all(cp)
    rects = P.tile_rects(cp)
    table = G.enumerate_blocks(cp)
    assert len(table) == len(blks)
    chunks, off = [], 0
    want = [np.zeros_like(c) for c in coefs]
    causal = bool(cp.cblk_sty & 0x08)
    rng = np.random.default_rng(seed)
    for i, (t, c, b) in enumerate(blks):
        w, h = b.x1 - b.x0, b.y1 - b.y0
        if w == 0 or h == 0:
            continue
        x0, y0 = rects[t][0] - cp.x0, rects[t][1] - cp.y0
        kmax, step_enc, step_dec = P.band_params(cp, b.resno, b.orient)
        win = np.ascontiguousarray(coefs[c][y0 + b.buf_y:y0 + b.buf_y + h, x0 + b.buf_x:x0 + b.buf_x + w])
        sm = np.zeros(w * h, np.uint32)
        if cp.irreversible:
            L.orc_ht_pre_irrev(win.view(np.float32), w, w, h, kmax, np.float32(1.0) / np.float32(step_enc), sm)
        else:
            L.orc_ht_pre_rev(win, w, w, h, kmax, sm)
        # decoder-aligned words: magnitude LSB at plane 31 - kmax
        W = (((sm & 0x7FFFFFFF) << 1) | (sm & 0x80000000)).astype(np.uint32).reshape(h, w)
        s = dropped if kmax - 1 - dropped >= 0 else 0
        mm = kmax - 1 - s
        np_blk = npass if (s > 0 and rng.random() < 0.85) else 1      # a few cleanup-only blocks in between
        cup = O.ht_encode(W, mm)
        seg = O.ht_encode_refine(W, mm, np_blk, causal) if np_blk > 1 else np.zeros(0, np.uint8)
        data = np.concatenate([cup, seg])
        rc, dec = O.ht_decode_passes(data, len(seg), np_blk, mm, w, h, causal=causal)
        assert rc == 0
        if cp.irreversible:
            out = np.zeros((h, w), np.float32)
            L.orc_ht_post_irrev(dec, w, w, h, kmax, step_dec, out, w)
            out = out.view(np.int32)
        else:
            out = np.zeros((h, w), np.int32)
            L.orc_ht_post_rev(dec, w, w, h, kmax, out, w)
        want[c][y0 + b.buf_y:y0 + b.buf_y + h, x0 + b.buf_x:x0 + b.buf_x + w] = out
        table[i]["length"], table[i]["length2"], table[i]["offset"] = len(cup), len(seg), off
        table[i]["numbps"], table[i]["numpasses"] = 1 + s, np_blk
        chunks.append(data)
        off += len(data)
    return table, np.concatenate(chunks), want


@pytest.mark.parametrize("case", [
    dict(args=dict(width=333, height=217, numcomps=3, prec=12, numres=4, origin=(3, 5)), npass=3, dropped=1),
    dict(args=dict(width=333, height=217, numcomps=3, prec=12, numres=4, origin=(3, 5)), npass=2, dropped=2),
    dict(args=dict(width=300, height=200, numcomps=3, prec=8, numres=5, tile=(128, 128), origin=(129, 65), tile_origin=(1, 1),
                   cblk=(16, 128)), npass=3, dropped=1),
    dict(args=dict(width=256, height=96, numcomps=1, prec=10, numres=3, cblk=(1024, 4)), npass=3, dropped=1),   # widest blocks
    dict(args=dict(width=200, height=160, numcomps=3, prec=12, numres=4), npass=3, dropped=1, causal=True),
    dict(args=dict(width=320, height=200, numcomps=3, prec=12, numres=5, irreversible=True), npass=3, dropped=2),
])
def test_refinement_passes_of_foreign_streams(engine, case):
    """SigProp / MagRef (T1OJPH::decompress with 2 or 3 passes, ojph_block_decoder32.cpp L1318-1616):
    block tables as a foreign HT encoder would produce them -- cleanup pass above the LSB plane,
    refinement for the next plane, cleanup-only blocks mixed in, stripe-causal variant -- decode on the
    device to exactly the coefficients the oracle decodes (which is pinned to the reference decoder),
    and b2k_decode returns the pixels of those coefficients."""
    args = case["args"]
    cp = G.make_coding(**args)
    if case.get("causal"):
        cp.cblk_sty = 0x08
    planes = P.synthetic_image(args["width"], args["height"], args["numcomps"], args["prec"], seed=7,
                               origin=args.get("origin", (0, 0)))
    coefs = P.forward(cp, planes)
    table, data, want = _refined_blocks(cp, coefs, case["npass"], case["dropped"], seed=3)
    assert (table["numpasses"] > 1).sum() > 0
    job = engine.job(cp)
    job.upload(planes)                                    # sizes the planes; content is overwritten below
    got = [np.full_like(p, -1) for p in planes]
    job.upload_coeffs(got)
    job.t1_decode_blocks(table, data)
    job.download_coeffs(got)
    for c, (g, r) in enumerate(zip(got, want)):
        assert np.array_equal(g, r), "component %d: %d coefficients differ" % (c, int((g != r).sum()))
    job.close()
    out = [np.zeros_like(p) for p in planes]
    engine.decode(cp, table, data, out)
    ref = P.inverse(cp, want)
    for g, r in zip(out, ref):
        if cp.irreversible:
            assert np.abs(g - r).max() <= 1               # device vs host inverse 9/7 (GrkPluginBatchMemoryTest.cpp L35-45)
        else:
            assert np.array_equal(g, r)
    if not cp.irreversible and case["npass"] == 3 and case["dropped"] == 1:
        # every plane was coded in the 3-pass blocks (only isolated +-1 coefficients, never SigProp members,
        # are missing) and the cleanup-only blocks lost one plane: nothing is off by more than one
        for g, s in zip(got, coefs):
            assert np.abs(g - s).max() <= 1


def test_corrupt_streams_are_rejected_or_decoded_never_fatal(engine):
    """Damaged block tables / byte arenas (flipped bytes, garbage Scup, wrong lengths, impossible bit-plane
    counts, bogus refinement segments): b2k_decode either decodes or reports rejected blocks (-2) or a bad
    table (-1); it never faults, and the engine decodes a clean stream right afterwards.  Blocks wider than
    64 samples go through the wide instantiation of the VLC parse (k_ht_decode_vlc<true>), so damaged bytes
    reach both.  (The 64x64 case was run under compute-sanitizer memcheck in profiles/r01g_memcheck.txt.)"""
    w, h = 256, 192
    planes = P.synthetic_image(w, h, 3, 12, seed=5)
    for cblk in ((64, 64), (1024, 4), (128, 32)):
        cp = G.make_coding(w, h, 3, 12, numres=4, cblk=cblk)
        res = engine.encode(cp, planes)
        blocks, data = res.blocks.copy(), res.bytes.copy()
        res.free()
        rng = np.random.default_rng(99)
        out = [np.zeros_like(p) for p in planes]
        outcomes = {"ok": 0, "rejected": 0, "bad_table": 0}
        coded = np.flatnonzero(blocks["length"] > 0)
        for trial in range(40):
            b, d = blocks.copy(), data.copy()
            kind = trial % 8
            if kind == 0:                                   # random byte flips all over the arena
                idx = rng.integers(0, len(d), 200)
                d[idx] ^= rng.integers(1, 256, 200).astype(np.uint8)
            elif kind == 1:                                 # garbage Scup (last two bytes of a block)
                for i in rng.choice(coded, 20):
                    e = int(b[i]["offset"]) + int(b[i]["length"])
                    d[e - 1], d[e - 2] = rng.integers(0, 256), rng.integers(0, 256)
            elif kind == 2:                                 # truncated cleanup segments
                for i in rng.choice(coded, 20):
                    b[i]["length"] = max(1, int(b[i]["length"]) // int(rng.integers(2, 6)))
            elif kind == 3:                                 # too many bit planes for the exponents in the stream
                for i in rng.choice(coded, 20):
                    b[i]["numbps"] = min(int(b[i]["kmax"]), int(b[i]["numbps"]) + int(rng.integers(1, 6)))
            elif kind == 4:                                 # refinement passes pointing into the neighbour's bytes
                for i in rng.choice(coded, 20):
                    b[i]["numpasses"], b[i]["length2"], b[i]["numbps"] = 3, min(64, len(d) - int(b[i]["offset"]) - int(b[i]["length"])), 3
            elif kind == 5:                                 # offsets past the arena
                b[rng.choice(coded)]["offset"] = len(d) + 1000
            elif kind == 6:                                 # all zero bytes
                d[:] = 0
            else:                                           # all ones
                d[:] = 0xFF
            try:
                engine.decode(cp, b, d, out)
                outcomes["ok"] += 1
            except G.EngineError as e:
                msg = str(e)
                assert "rejected" in msg or "exceed" in msg or "-1" in msg or "-2" in msg, (cblk, msg)
                outcomes["rejected" if "rejected" in msg else "bad_table"] += 1
        assert outcomes["rejected"] > 0 and outcomes["bad_table"] > 0, (cblk, outcomes)
        engine.decode(cp, blocks, data, out)               # still healthy
        for a, s in zip(out, planes):
            assert np.array_equal(a, s), cblk


@pytest.mark.parametrize("sgnd", [False, True])
def test_host_packing_matches_direct_copies(engine, sgnd):
    """int32 entry points with host packing forced on (16-bit PCIe containers through the pinned ring, host
    thread pool) against the same calls with packing off: same coded bytes, same pixels, lossless -- on a
    geometry with ragged tiles, an odd canvas origin and (second case) signed samples, large enough
    (>= 4 Msamples, several pipeline chunks) for the packed path to be taken, with unpinned caller planes."""
    w, h, prec = 2501, 1803, (16 if sgnd else 12)
    cp = G.make_coding(w, h, 3, prec, sgnd=sgnd, numres=5, tile=(700, 500), origin=(3, 5), numgbits=2 if sgnd else 1)
    planes = P.synthetic_image(w, h, 3, prec, seed=11, origin=(3, 5))
    if sgnd:
        planes = [p - (1 << (prec - 1)) for p in planes]
    strided = [np.zeros((h, w + 13), np.int32) for _ in planes]     # row stride != width
    for s, p in zip(strided, planes):
        s[:, :w] = p
    views = [s[:, :w] for s in strided]
    results = {}
    try:
        for mode, threads in (("direct", 0), ("packed", 3)):
            G.set_host_threads(threads)
            res = engine.encode(cp, views)
            assert G.host_pack_last()[0] == (1 if threads else 0)
            blocks, data = res.blocks.copy(), res.bytes.copy()
            res.free()
            out = [np.full((h, w + 5), -7, np.int32) for _ in planes]
            engine.decode(cp, blocks, data, [o[:, :w] for o in out])
            assert G.host_pack_last()[1] == (1 if threads else 0)
            for o, p in zip(out, planes):
                assert np.array_equal(o[:, :w], p)               # lossless
                assert np.all(o[:, w:] == -7)                    # nothing written past the rows
            results[mode] = (blocks, data)
    finally:
        G.set_host_threads(-1)
    assert np.array_equal(results["direct"][1], results["packed"][1])
    assert np.array_equal(results["direct"][0]["length"], results["packed"][0]["length"])


@pytest.mark.parametrize("irreversible", [False, True])
def test_codestream_files_round_trip_and_openjpeg_reads_them(engine, irreversible):
    """b2k_encode + b2k_codestream_write gives a file an independent decoder (OpenJPEG, through OpenCV) reads:
    exactly the source for the reversible path, within the reference's lossy tolerance for 9/7; and
    b2k_codestream_parse + b2k_decode read it back on the device, block bytes taken in place from the file."""
    cv2 = pytest.importorskip("cv2")
    w, h = 1100, 700
    cp = G.make_coding(w, h, 3, 12, numres=6, tile=(512, 512), irreversible=irreversible)
    planes = P.synthetic_image(w, h, 3, 12, seed=31)
    cs = engine.encode_codestream(cp, planes)
    ext = cv2.imdecode(np.frombuffer(cs.tobytes(), np.uint8), cv2.IMREAD_UNCHANGED)
    assert ext is not None and ext.shape == (h, w, 3)
    ext = ext[:, :, ::-1].astype(np.int64)
    src = np.stack(planes, axis=-1).astype(np.int64)
    cp2, ours = engine.decode_codestream(cs)
    ours = np.stack(ours, axis=-1).astype(np.int64)
    if irreversible:
        assert np.abs(ext - ours).max() <= 1
        for rec in (ext, ours):
            err = (rec - src).astype(np.float64)
            assert np.abs(err).max() <= 16 and 10 * np.log10(4095.0 ** 2 / (err ** 2).mean()) > 50.0
    else:
        assert np.array_equal(ext, src)
        assert np.array_equal(ours, src)
    assert cp2.numres == cp.numres and cp2.tw == 512 and cp2.irreversible == cp.irreversible


def test_explicit_qcd_on_the_device(engine):
    """b2k_coding.qcd_explicit (band exponents other than the HT quantiser's, as a foreign stream's QCD gives them):
    the device encodes and decodes with them -- OpenJPEG reads the file exactly, and so does the engine."""
    cv2 = pytest.importorskip("cv2")
    w, h = 640, 400
    cp = G.make_coding(w, h, 3, 8, numres=5, tile=(256, 256))
    e, _ = P.quant_tables(cp)
    cp.qcd_explicit = 1
    for i in range(len(e)):
        cp.qcd_expn[i] = int(e[i]) + 1 + (i % 2)
    planes = P.synthetic_image(w, h, 3, 8, seed=71)
    cs = engine.encode_codestream(cp, planes)
    ext = cv2.imdecode(np.frombuffer(cs.tobytes(), np.uint8), cv2.IMREAD_UNCHANGED)[:, :, ::-1].astype(np.int64)
    assert np.array_equal(ext, np.stack(planes, axis=-1))
    cp2, ours = engine.decode_codestream(cs)
    assert cp2.qcd_explicit == 1
    for a, b in zip(ours, planes):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("args", [
    dict(width=61, height=9, numcomps=1, prec=8, numres=6),                                          # levels run out of samples
    dict(width=64, height=64, numcomps=3, prec=10, numres=3, tile=(1, 64)),                          # 1-pixel-wide tiles
    dict(width=40, height=33, numcomps=1, prec=12, numres=2, tile=(7, 1), cblk=(4, 4)),              # 1-pixel-high tiles
    dict(width=333, height=217, numcomps=3, prec=12, numres=4, origin=(3, 5), tile=(100, 90)),       # odd origin, ragged tiles
    dict(width=333, height=217, numcomps=3, prec=12, numres=1, origin=(3, 5), tile=(100, 90)),       # no wavelet level
])
def test_irreversible_degenerate_geometry(engine, args):
    """GrkDegenerate97Test / GrkShortTileRoundTripTest shapes on the 9/7 + ICT path: width / height 1 special cases
    (WaveletFwd.cpp L444-455, L639-654), odd parities, ragged tiles -- coefficients and coded bytes bit-exact against
    the oracle's fp32 restatement, decode within the reference's lossy tolerance of the source."""
    cp = G.make_coding(irreversible=True, **args)
    planes = P.synthetic_image(args["width"], args["height"], args["numcomps"], args["prec"], seed=81,
                               origin=args.get("origin", (0, 0)))
    ref = P.forward(cp, planes)
    job = engine.job(cp)
    job.upload(planes)
    job.forward()
    got = [np.zeros_like(p) for p in planes]
    job.download_coeffs(got)
    for c, (g, r) in enumerate(zip(got, ref)):
        assert np.array_equal(g, r), "component %d: %d coefficients differ" % (c, int((g != r).sum()))
    job.t1_encode()
    res = job.fetch_result()
    _compare_blocks(cp, res, ref)
    job.t1_decode()
    job.inverse()
    rec = [np.zeros_like(p) for p in planes]
    job.download(rec)
    peak = (1 << args["prec"]) - 1
    for g, s in zip(rec, planes):
        assert np.abs(g - s).max() <= max(2, peak // 256)
    res.free()
    job.close()


def test_repeated_and_concurrent_calls_are_deterministic(engine):
    """GrkPluginBatchMemoryTest's determinism check (L970) and GrkConcurrencyTest's shape: the same image encoded
    repeatedly, packed and direct, and from four threads at once (the engine serialises them) gives the same bytes
    every time, and every decode gives the source back."""
    import threading
    w, h = 2048, 1536
    cp = G.make_coding(w, h, 3, 12, numres=6, tile=(512, 512))
    planes = P.synthetic_image(w, h, 3, 12, seed=91)
    res = engine.encode(cp, planes)
    want_blocks, want = res.blocks.copy(), res.bytes.copy()
    res.free()
    try:
        for threads in (0, 2, 0, 2):
            G.set_host_threads(threads)
            r = engine.encode(cp, planes)
            assert np.array_equal(r.bytes, want) and np.array_equal(r.blocks["length"], want_blocks["length"])
            r.free()
    finally:
        G.set_host_threads(-1)
    errors = []

    def worker(i):
        try:
            for _ in range(3):
                r = engine.encode(cp, planes)
                ok = np.array_equal(r.bytes, want)
                out = [np.zeros_like(p) for p in planes]
                engine.decode(cp, r.blocks, r.bytes, out)
                r.free()
                if not ok or not all(np.array_equal(a, b) for a, b in zip(out, planes)):
                    errors.append("thread %d: mismatch" % i)
        except Exception as e:      # noqa: BLE001
            errors.append("thread %d: %r" % (i, e))

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors


def test_two_engines_in_one_process(engine):
    """ADVICE r1 / VERDICT weak #7: kernel attributes (dynamic shared memory opt-in) are per device, and INTEGRATION.md
    offers "one engine per GPU" in one process.  A second engine -- on a second GPU when the box has one, else on the same
    device -- is created AFTER the first has already launched every kernel, and both then work concurrently from two
    threads: same bytes, lossless decode."""
    import threading
    import torch
    second_dev = 1 if torch.cuda.device_count() > 1 else 0
    w, h = 1024, 768
    cp = G.make_coding(w, h, 3, 12, numres=6, tile=(512, 512))
    cpi = G.make_coding(w, h, 3, 12, numres=6, irreversible=True)
    planes = P.synthetic_image(w, h, 3, 12, seed=17)
    r = engine.encode(cp, planes)
    want = r.bytes.copy()
    r.free()
    ri = engine.encode(cpi, planes)
    want_i = ri.bytes.copy()
    ri.free()
    e2 = G.Engine(second_dev)
    errors = []

    def worker(eng, tag):
        try:
            for _ in range(3):
                a = eng.encode(cp, planes)
                out = [np.zeros_like(p) for p in planes]
                eng.decode(cp, a.blocks, a.bytes, out)
                ok = np.array_equal(a.bytes, want) and all(np.array_equal(x, y) for x, y in zip(out, planes))
                a.free()
                b = eng.encode(cpi, planes)
                ok = ok and np.array_equal(b.bytes, want_i)
                b.free()
                if not ok:
                    errors.append(tag + ": mismatch")
        except Exception as e:      # noqa: BLE001
            errors.append("%s: %r" % (tag, e))

    ts = [threading.Thread(target=worker, args=(engine, "engine0")), threading.Thread(target=worker, args=(e2, "engine1"))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    e2.close()
    assert not errors, errors


def test_decode_with_byte_arena_not_in_tile_order(engine):
    """ADVICE r1 (medium): a caller arena / foreign code stream whose tiles are not laid out in tile-index order (legal:
    tile parts may come in any order).  The chunk-pipelined upload must not leave holes: tiles' byte ranges are permuted
    (last tile first, gaps between them), offsets patched, and the decode must still return the source."""
    w, h = 1536, 1024
    cp = G.make_coding(w, h, 3, 12, numres=5, tile=(256, 256))      # 24 tiles -> several pipeline chunks
    planes = P.synthetic_image(w, h, 3, 12, seed=23)
    res = engine.encode(cp, planes)
    blocks, data = res.blocks.copy(), res.bytes.copy()
    res.free()
    ntiles = int(blocks["tile"].max()) + 1
    order = np.random.default_rng(5).permutation(ntiles)
    new = np.zeros(data.size + 64 * ntiles + 1000, np.uint8)
    new[:] = 0xA5
    pos = 777
    nb = blocks.copy()
    for t in order:
        sel = np.nonzero((blocks["tile"] == t) & (blocks["length"] > 0))[0]
        for i in sel:
            o, n = int(blocks[i]["offset"]), int(blocks[i]["length"])
            new[pos:pos + n] = data[o:o + n]
            nb[i]["offset"] = pos
            pos += n
        pos += 61
    out = [np.zeros_like(p) for p in planes]
    engine.decode(cp, nb, new[:pos], out)
    for a, b in zip(out, planes):
        assert np.array_equal(a, b)


def test_streaming_encode_decode_matches_the_synchronous_calls(engine):
    """SURVEY 8f N2: frames in flight on several engines of one GPU.  Six different frames go through an encode stream
    (depth 3) whose callback feeds a decode stream (depth 3): every frame's coded bytes equal the synchronous
    b2k_encode's, every decoded frame equals its source -- GrkPluginBatchMemoryTest's property (all frames come back,
    each lossless) plus byte identity with the per-call path."""
    import threading
    w, h = 1536, 1024
    cp = G.make_coding(w, h, 3, 12, numres=6, tile=(512, 512))
    frames = [P.synthetic_image(w, h, 3, 12, seed=100 + i) for i in range(6)]
    want = []
    for f in frames:
        r = engine.encode(cp, f)
        want.append(r.bytes.copy())
        r.free()
    outs = [[np.zeros((h, w), np.int32) for _ in range(3)] for _ in frames]
    results, errors, done = {}, [], threading.Semaphore(0)

    def on_decoded(tag, status):
        if status != 0:
            errors.append("decode %r: status %d" % (tag, status))
        done.release()

    dec = G.DecodeStream(depth=3, on_decoded=on_decoded)

    def on_encoded(tag, res, status):
        if status != 0 or res is None:
            errors.append("encode %r: status %d" % (tag, status))
            done.release()
            return
        results[tag] = res
        dec.submit(cp, res.blocks, res.bytes, outs[tag], tag)

    enc = G.EncodeStream(cp, depth=3, on_encoded=on_encoded)
    for i, f in enumerate(frames):
        enc.submit(f, i)
    for _ in frames:
        assert done.acquire(timeout=120)
    assert enc.end() == 0 and dec.end() == 0
    assert not errors, errors
    for i, f in enumerate(frames):
        assert np.array_equal(results[i].bytes, want[i]), "frame %d: streamed bytes differ from b2k_encode's" % i
        for a, b in zip(outs[i], f):
            assert np.array_equal(a, b)
        results[i].free()


def test_stock_batch_memory_symbols(engine):
    """gpup_batch_memory_begin / _submit / _end (grok.cpp L1655-1857) driven the way the host drives them: frames as
    pixel-interleaved 16-bit samples, results through the compress callback as stock gpup_tile trees, concurrently."""
    import os
    import threading
    from gpup_ctypes import GpupTile
    lib = G.lib()
    w, h, nc, prec = 640, 384, 3, 12
    cp = G.make_coding(w, h, nc, prec, numres=6)
    frames = [P.synthetic_image(w, h, nc, prec, seed=300 + i) for i in range(5)]
    want = []
    for f in frames:
        r = engine.encode(cp, f)
        want.append([r.block_bytes(i).copy() for i in range(r.num_blocks)])
        r.free()

    class StreamParams(C.Structure):
        _fields_ = [("file", C.c_char_p), ("buf", C.c_void_p), ("buf_len", C.c_size_t), ("buf_compressed_len", C.c_size_t)]

    class CbInfo(C.Structure):
        _fields_ = [("input_file_name", C.c_char_p), ("outputFileNameIsRelative", C.c_bool), ("output_file_name", C.c_char_p),
                    ("compressor_parameters", C.c_void_p), ("image", C.c_void_p), ("tile", C.POINTER(GpupTile)),
                    ("stream_params", StreamParams), ("error_code", C.c_uint), ("host_data", C.c_void_p)]
    assert C.sizeof(CbInfo) == 96

    class BatchInfo(C.Structure):
        _fields_ = [("compress_parameters", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32), ("numcomps", C.c_uint32),
                    ("source_prec", C.c_uint32), ("prec", C.c_uint32), ("callback", C.c_void_p), ("xyz_on_device", C.c_bool),
                    ("source_format", C.c_int), ("yuv_matrix", C.c_int), ("yuv_full_range", C.c_bool)]
    assert C.sizeof(BatchInfo) == 56
    got, lock = {}, threading.Lock()
    CB = C.CFUNCTYPE(C.c_uint64, C.POINTER(CbInfo))

    def cb(pinfo):
        info = pinfo.contents
        blocks = []
        if info.error_code == 0 and info.tile:
            T = info.tile.contents
            for c in range(T.numComponents):
                tc = T.tileComponents[c].contents
                for r in range(tc.numResolutions):
                    res = tc.resolutions[r].contents
                    for b in range(res.numBands):
                        band = res.band[b].contents
                        for p in range(band.numPrecincts):
                            prc = band.precincts[p].contents
                            for j in range(prc.numBlocks):
                                cb_ = prc.blocks[j].contents
                                blocks.append(bytes(np.ctypeslib.as_array(cb_.compressedData, shape=(cb_.compressedDataLength,)))
                                              if cb_.compressedDataLength else b"")
        with lock:
            got[int(info.host_data)] = blocks
        return 1

    cb_keep = CB(cb)
    params = (C.c_uint8 * 12696)()
    probe = r'''
#include <stdio.h>
#include <stddef.h>
#include "grok_b200.h"
#define O(f) printf(#f " %zu\n", offsetof(gpup_compress_params, f));
int main(void){ O(numlayers) O(csty) O(numgbits) O(numresolution) O(cblockw_init) O(cblockh_init) O(cblk_sty) O(irreversible) O(roi_compno) O(mct) return 0; }'''
    import subprocess
    exe = "/tmp/b2k_off2_%d" % os.getpid()
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(os.path.dirname(G._HERE), "include"), "-o", exe], input=probe.encode(), check=True)
    off = dict((k, int(v)) for k, v in (l.split() for l in subprocess.check_output([exe]).decode().splitlines()))

    def put(o, val, typ):
        typ.from_buffer(params, o).value = val
    put(off["numlayers"], 1, C.c_uint16); put(off["numgbits"], 1, C.c_uint8); put(off["numresolution"], 6, C.c_uint8)
    put(off["cblockw_init"], 64, C.c_uint32); put(off["cblockh_init"], 64, C.c_uint32); put(off["cblk_sty"], 0x40, C.c_uint8)
    put(off["roi_compno"], -1, C.c_int32); put(off["mct"], 1, C.c_uint8)
    info = BatchInfo(C.addressof(params), w, h, nc, prec, prec, C.cast(cb_keep, C.c_void_p), False, 0, 0, False)
    lib.gpup_batch_memory_begin.argtypes = [C.POINTER(BatchInfo)]
    lib.gpup_batch_memory_submit.argtypes = [C.c_void_p, C.c_void_p]
    lib.gpup_batch_memory_submit.restype = C.c_bool
    lib.gpup_batch_memory_end.restype = C.c_bool
    assert lib.gpup_batch_memory_begin(C.byref(info)) == 0, lib.b2k_last_error()
    for i, f in enumerate(frames):
        packed = np.ascontiguousarray(np.stack(f, axis=-1).astype(np.uint16))       # pixel interleaved, little endian
        assert lib.gpup_batch_memory_submit(packed.ctypes.data, C.c_void_p(i + 1))   # copied before the call returns
        packed[:] = 0xFFFF
    assert lib.gpup_batch_memory_end()
    assert sorted(got) == [i + 1 for i in range(len(frames))]
    for i in range(len(frames)):
        assert got[i + 1] == [bytes(b) for b in want[i]]


def test_host_packing_with_pinned_caller_planes(engine):
    """Pinned caller planes + host packing (the bench's e2e configuration): same coded bytes as the all-direct call, lossless
    decode -- on an image with enough tiles for several pipeline chunks, odd tile sizes included.
    (Round 2 tried sending every n-th chunk as plain int32 DMA beside the packed ones: 21.1 -> 25.8 / 28.2 ms on config 2,
    dropped; DESIGN.md section 7.)"""
    w, h = 2500, 1900
    cp = G.make_coding(w, h, 3, 12, numres=5, tile=(300, 200))          # 9 x 10 tiles
    src = P.synthetic_image(w, h, 3, 12, seed=41)
    planes = [G.pinned_empty((h, w), np.int32) for _ in range(3)]
    out = [G.pinned_empty((h, w), np.int32) for _ in range(3)]
    for a, b in zip(planes, src):
        a[:] = b
    try:
        G.set_host_threads(0)
        r = engine.encode(cp, planes)
        want_blocks, want = r.blocks.copy(), r.bytes.copy()
        r.free()
        G.set_host_threads(4)
        for _ in range(2):
            r = engine.encode(cp, planes)
            assert G.host_pack_last()[0] == 1
            assert np.array_equal(r.bytes, want) and np.array_equal(r.blocks["length"], want_blocks["length"])
            for o in out:
                o[:] = -1
            engine.decode(cp, r.blocks, r.bytes, out)
            assert G.host_pack_last()[1] == 1
            r.free()
            for a, b in zip(out, src):
                assert np.array_equal(a, b)
    finally:
        G.set_host_threads(-1)
