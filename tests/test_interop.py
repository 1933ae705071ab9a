"""Interop parity gate against the REAL reference library (BASELINE.md 3.6).

The reference outputs are those of the unmodified GrokImageCompression/Grok (libgrokj2k built by
oracle/build_grok.sh, driven through its public API by tests/grok_ref.py: grk_compress / grk_decompress on memory
streams), kept in tests/golden/ by tests/golden/make_reference_golden.py: digests of its code streams and of its
decoded images, its COM marker segments, and its decode itself where only a tolerance applies.
What is pinned here, on the reference's own outputs:

* reversible path: our codestream (b2k_codestream_write over oracle- or GPU-coded blocks) is BYTE-IDENTICAL to
  grk_compress's once Grok's COM marker segment is removed; every code block's bytes are equal; Grok decodes ours to
  the source exactly; our parser + decoder read Grok's stream exactly;
* irreversible path (9/7 + ICT): every code block's bytes equal Grok's (which pins ICT's FMA contraction
  `fma(a_b,b, fma(a_g,g, a_r*r))`, the 9/7 lifting, the step sizes and the T1 pre-quantiser), and for
  precision >= 9 bits our decode of Grok's stream equals Grok's own decode sample for sample (Grok decodes
  <= 8-bit irreversible images through its 16-bit fixed-point engine: a different algorithm; there the bar is
  the reference's own <= 2 codes, GrkPluginBatchMemoryTest.cpp L35-45).

The CPU tests use the oracle as the block coder (no GPU), the `-m gpu` tests the CUDA engine."""
import numpy as np
import pytest

import grok_b200 as G
import oracle_pipeline as P
import reference_golden as RG
from test_codestream import oracle_decode, oracle_encode


def strip_com(cs):
    """Remove COM (0xFF64) marker segments from the main header: Grok writes 'Created by Grok ...' there."""
    cs = bytes(cs)
    out, i = bytearray(cs[:2]), 2
    while True:
        m = (cs[i] << 8) | cs[i + 1]
        if m == 0xFF90:
            break
        ln = (cs[i + 2] << 8) | cs[i + 3]
        if m != 0xFF64:
            out += cs[i:i + 2 + ln]
        i += 2 + ln
    return bytes(out) + cs[i:]


def grok_compress(args, planes, R):
    """grk_compress with TLM + PLT (`R`: tests/grok_ref.py; the golden data's generator calls this)"""
    cs, _ = R.compress(planes, args["prec"], tile=args.get("tile"), numres=args.get("numres", 6),
                       irreversible=args.get("irreversible", False), tlm=True, plt=True, cblk=args.get("cblk", (64, 64)),
                       precinct=args.get("grok_precinct"))
    return np.frombuffer(bytes(cs), np.uint8)


def oracle_codestream(args, planes):
    table, data, _ = oracle_encode(mk(args), planes)
    return G.codestream_write(mk(args), table, data, G.CS_TLM | G.CS_PLT)


def block_bytes(table, data, i):
    o, n = int(table[i]["offset"]), int(table[i]["length"])
    return data[o:o + n]


REVERSIBLE = [
    dict(width=512, height=512, numcomps=1, prec=8),                                  # BASELINE config 1
    dict(width=640, height=384, numcomps=3, prec=12, tile=(256, 256)),                # config 2 in small
    dict(width=333, height=217, numcomps=3, prec=12),                                 # odd size, one tile
    dict(width=200, height=150, numcomps=4, prec=16, tile=(128, 64), numres=4),       # config 4 in small
    dict(width=300, height=260, numcomps=3, prec=8, numres=3, cblk=(32, 32)),
    dict(width=1100, height=700, numcomps=3, prec=10, numres=10),                      # 9 decomposition levels (VERDICT r1: > 8 resolutions)
    dict(width=900, height=600, numcomps=1, prec=12, numres=10, tile=(512, 512)),      # as many levels as a 512 tile takes (the host clamps more)
    dict(width=333, height=217, numcomps=3, prec=12, numres=1, tile=(128, 128)),       # no wavelet level: DC shift + RCT only
    dict(width=130, height=90, numcomps=4, prec=16, numres=1),                         # ... with an untransformed 4th component
]
IRREVERSIBLE = [
    dict(width=640, height=384, numcomps=3, prec=12, irreversible=True),              # config 3 in small
    dict(width=333, height=217, numcomps=3, prec=12, irreversible=True, tile=(128, 128), numres=4),
    dict(width=300, height=200, numcomps=1, prec=12, irreversible=True),
    dict(width=320, height=192, numcomps=3, prec=16, irreversible=True, numres=5),
    dict(width=1100, height=700, numcomps=3, prec=10, irreversible=True, numres=10),
    dict(width=200, height=150, numcomps=3, prec=12, irreversible=True, numres=1),     # no wavelet level: ICT + quantiser only
    dict(width=130, height=90, numcomps=1, prec=10, irreversible=True, numres=1, tile=(64, 64)),
]


def synth(args, seed=5):
    return P.synthetic_image(args["width"], args["height"], args["numcomps"], args["prec"], seed=seed)


def mk(args):
    a = {k: v for k, v in args.items() if k != "grok_precinct"}
    return G.make_coding(**a)


@pytest.mark.parametrize("args", REVERSIBLE)
def test_reversible_codestream_is_byte_identical_to_grok(args):
    cp = mk(args)
    planes = synth(args)
    table, data, _ = oracle_encode(cp, planes)
    ours = G.codestream_write(cp, table, data, G.CS_TLM | G.CS_PLT)
    theirs = RG.grok_codestream(ours, args, 5)
    # Grok decodes its stream, which is ours, exactly
    assert RG.planes_sha(planes) == RG.grok_decoded(args, 5)
    # we decode Grok's exactly, block bytes equal
    cp2, blocks = G.codestream_parse(theirs)
    assert len(blocks) == len(table)
    for i in range(len(table)):
        assert np.array_equal(block_bytes(table, data, i), block_bytes(blocks, theirs, i)), "block %d" % i
    rec = oracle_decode(cp2, blocks, theirs)
    for a, b in zip(rec, planes):
        assert np.array_equal(a, b)


def test_precinct_spec_shorter_than_resolutions_matches_grok():
    """`-c [128,128]` style: one precinct size given (res_spec = 1), the coarser resolutions take it halved per level
    (CodeStreamCompress.cpp L793-825).  The packet order then depends on the derived precinct grid."""
    args = dict(width=600, height=500, numcomps=3, prec=12, numres=5)
    planes = synth(args)
    cp = G.make_coding(precincts=[(max(128 >> k, 2),) * 2 for k in range(5)][::-1], **args)
    table, data, _ = oracle_encode(cp, planes)
    ours = G.codestream_write(cp, table, data, G.CS_TLM | G.CS_PLT)
    RG.grok_codestream(ours, dict(args, grok_precinct=(128, 128)), 5)   # grk_compress -c [128,128]


@pytest.mark.parametrize("args", IRREVERSIBLE)
def test_irreversible_blocks_are_byte_identical_to_grok(args):
    cp = mk(args)
    planes = synth(args)
    table, data, _ = oracle_encode(cp, planes)
    ours = G.codestream_write(cp, table, data, G.CS_TLM | G.CS_PLT)
    theirs = RG.grok_codestream(ours, args, 5)
    cp2, blocks = G.codestream_parse(theirs)
    same = sum(int(np.array_equal(block_bytes(table, data, i), block_bytes(blocks, theirs, i))) for i in range(len(table)))
    assert same == len(table), "%d of %d irreversible code blocks equal Grok's" % (same, len(table))
    # decode: ours of theirs == Grok's of theirs, sample for sample (precision >= 9)
    od = oracle_decode(cp2, blocks, theirs)
    assert RG.planes_sha(od) == RG.grok_decoded(args, 5)


def test_irreversible_8bit_decode_within_reference_tolerance():
    """<= 8-bit irreversible images: Grok decodes with its int16 fixed-point 9/7 engine; the float path here agrees
    with it to within the reference's own device-vs-host bar (<= 2 codes), coded blocks are still identical."""
    args = dict(width=320, height=256, numcomps=3, prec=8, irreversible=True)
    cp = mk(args)
    planes = synth(args)
    table, data, _ = oracle_encode(cp, planes)
    theirs = RG.grok_codestream(G.codestream_write(cp, table, data, G.CS_TLM | G.CS_PLT), args, 5)
    cp2, blocks = G.codestream_parse(theirs)
    for i in range(len(table)):
        assert np.array_equal(block_bytes(table, data, i), block_bytes(blocks, theirs, i))
    gd = RG.outputs()["decoded_8bit_irreversible_minus_source"] + np.stack(planes)      # Grok's decode
    assert RG.planes_sha(gd) == RG.grok_decoded(args, 5)
    od = oracle_decode(cp2, blocks, theirs)
    for a, b in zip(gd, od):
        assert np.abs(a.astype(np.int64) - b).max() <= 2


# ------------------------------------------------------------------------------------------------------
# the same gate with GPU-coded blocks / GPU decode
# ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("args", REVERSIBLE + IRREVERSIBLE)
def test_gpu_codestream_is_byte_identical_to_grok_and_decodes_it(engine, args):
    cp = mk(args)
    planes = synth(args, seed=9)
    ours = engine.encode_codestream(cp, planes, flags=G.CS_TLM | G.CS_PLT)
    theirs = RG.grok_codestream(ours, args, 9)
    # the GPU decodes Grok's stream (which Grok decodes as its own: it is the GPU's) to what Grok gave back
    _, ours_of_theirs = engine.decode_codestream(theirs)
    if args.get("irreversible"):
        # Grok's decode of >= 9-bit 9/7 streams is the oracle's, sample for sample (test_irreversible_blocks_are_...)
        cp2, blocks = G.codestream_parse(theirs)
        g_of_theirs = oracle_decode(cp2, blocks, theirs)
        assert RG.planes_sha(g_of_theirs) == RG.grok_decoded(args, 9)
        for b, c in zip(g_of_theirs, ours_of_theirs):
            assert np.abs(c.astype(np.int64) - b).max() <= 1      # device inverse 9/7 vs Grok's host inverse
    else:
        assert RG.planes_sha(planes) == RG.grok_decoded(args, 9)
        for c, src in zip(ours_of_theirs, planes):
            assert np.array_equal(c, src)


@pytest.mark.gpu
def test_gpu_config2_tiles_match_grok_at_full_tile_size(engine):
    """Four full-size 1024x1024 tiles of config 2 (2048x2048x3, 12 bit, 6 resolutions): whole codestream equal."""
    args = dict(width=2048, height=2048, numcomps=3, prec=12, tile=(1024, 1024))
    cp = mk(args)
    planes = P.synthetic_image(2048, 2048, 3, 12, seed=20260924)
    ours = engine.encode_codestream(cp, planes, flags=G.CS_TLM | G.CS_PLT)
    theirs = RG.grok_codestream(ours, args, 20260924)
    _, rec = engine.decode_codestream(theirs)
    for a, b in zip(rec, planes):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------------------------
# BASELINE.json's configurations at the sizes they name (VERDICT r1 item 9), against the real library
# ------------------------------------------------------------------------------------------------------
CONFIG3 = dict(width=8192, height=8192, numcomps=3, prec=12, numres=6, irreversible=True)
CONFIG4 = dict(width=16384, height=16384, numcomps=4, prec=16, numres=6, tile=(1024, 1024), mct=1)


@pytest.mark.gpu
def test_config3_full_size_single_tile_irreversible_matches_grok(engine):
    """configs[2]: 8192x8192x3 12-bit, ONE tile, 9/7 + ICT, 5 levels (6 resolutions), 64x64 blocks.  The GPU's code
    stream must equal grk_compress's byte for byte (COM aside) -- every one of the 49,152 + ... code blocks -- and the
    GPU's decode of it must agree with Grok's own to within one code (device inverse 9/7 vs host; the reference's bar is
    <= 2, GrkPluginBatchMemoryTest.cpp L35-45) and sit > 50 dB from the source (GrkPluginMemoryTest.cpp L39-52)."""
    w = h = 8192
    cp = mk(CONFIG3)
    planes = P.synthetic_image(w, h, 3, 12, seed=20260925)
    ours = engine.encode_codestream(cp, planes, flags=G.CS_TLM | G.CS_PLT)
    theirs = RG.grok_codestream(ours, CONFIG3, 20260925)
    _, rec = engine.decode_codestream(theirs)
    # Grok's decode of a 12-bit 9/7 stream is the oracle's, sample for sample
    cp2, blocks = G.codestream_parse(theirs)
    gd = oracle_decode(cp2, blocks, theirs)
    assert RG.planes_sha(gd) == RG.grok_decoded(CONFIG3, 20260925)
    for a, b, s in zip(rec, gd, planes):
        assert np.abs(a.astype(np.int64) - b).max() <= 1
        err = (a.astype(np.float64) - s)
        assert 10 * np.log10(4095.0 ** 2 / (err ** 2).mean()) > 50.0


@pytest.mark.gpu
def test_config4_full_size_sharded_tiles_match_grok(engine):
    """configs[3]: 16384x16384x4 16-bit lossless, 256 tiles of 1024x1024 (RCT on components 0-2).  The tiles are coded
    as two shards (tile t -> shard t % 2, what two ranks would do), merged with b2k_result_merge and written as ONE
    code stream: byte-identical to grk_compress's, and the decode of Grok's stream gives the source back."""
    w = h = 16384
    cp = mk(CONFIG4)
    base = P.synthetic_image(1024, 1024, 4, 16, seed=20260926)
    planes = [np.empty((h, w), np.int32) for _ in range(4)]
    for t in range(256):
        ty, tx = divmod(t, 16)
        for c in range(4):
            planes[c][ty * 1024:(ty + 1) * 1024, tx * 1024:(tx + 1) * 1024] = (base[c] + 257 * t) & 0xFFFF
    shards = []
    for rem in (0, 1):
        r = engine.encode(cp, planes, tile_mod=2, tile_rem=rem)
        shards.append((r.blocks.copy(), r.bytes.copy()))
        r.free()
    merged = G.merge_shards(cp, shards)
    ours = G.codestream_write(cp, merged.blocks, merged.bytes, G.CS_TLM | G.CS_PLT, num_tiles=256)
    merged.free()
    theirs = RG.grok_codestream(ours, CONFIG4, 20260926)
    del ours, shards
    _, rec = engine.decode_codestream(theirs)
    for a, b in zip(rec, planes):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------------------------
# windowed / reduced-resolution decode (SURVEY 8f N3): the virtual coding b2k_codestream_parse_window derives
# ------------------------------------------------------------------------------------------------------
def _parse_window(cs, window, reduce):
    import ctypes as C
    L = G.lib()
    L.b2k_codestream_parse_window.restype = C.c_int64
    L.b2k_codestream_parse_window.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(G.Coding), C.c_void_p, C.c_uint64]
    win = (C.c_uint32 * 4)(*window) if window is not None else None
    cp = G.Coding()
    n = L.b2k_codestream_parse_window(cs.ctypes.data, len(cs), win, reduce, C.byref(cp), None, 0)
    assert n > 1, (n, L.b2k_last_error())
    blocks = np.zeros(n, G.BLOCK_DTYPE)
    assert L.b2k_codestream_parse_window(cs.ctypes.data, len(cs), win, reduce, C.byref(cp), blocks.ctypes.data, n) == n, L.b2k_last_error()
    return cp, blocks


WINDOW_CASES = [
    (dict(width=700, height=500, numcomps=3, prec=12, tile=(256, 128), numres=5), (300, 150, 520, 300), 0),
    (dict(width=700, height=500, numcomps=3, prec=12, tile=(256, 128), numres=5), None, 1),
    (dict(width=700, height=500, numcomps=3, prec=12, tile=(256, 128), numres=5), (10, 300, 400, 500), 2),
    (dict(width=640, height=384, numcomps=1, prec=8, tile=(128, 128), numres=4), (129, 1, 255, 127), 1),
    (dict(width=333, height=217, numcomps=3, prec=12, numres=5), None, 2),                      # single tile, reduce only
    (dict(width=900, height=700, numcomps=1, prec=12, numres=6), (411, 303, 475, 351), 0),      # a window far smaller than its tile
    (dict(width=900, height=700, numcomps=3, prec=12, numres=6, irreversible=True), (411, 303, 475, 351), 0),   # ... with the 9/7 support
    (dict(width=1000, height=600, numcomps=3, prec=12, tile=(512, 512), numres=5, irreversible=True), (500, 100, 530, 140), 1),
]


def window_args(args, window, reduce):
    return dict(args, window=window, reduce=reduce)


@pytest.mark.parametrize("args,window,reduce", WINDOW_CASES)
def test_window_and_reduce_parse_matches_grok(args, window, reduce):
    """The virtual coding decodes (on the oracle) to exactly what Grok delivers for the same window / reduce factor:
    grk_decompress at `reduce` gives the reference for the resolution, the window is a crop of it."""
    planes = synth(args, seed=12)
    theirs = RG.grok_codestream(oracle_codestream(args, planes), args, 12)
    w, h = args["width"], args["height"]
    # Grok's own reduced decode of the whole image, cropped to the window
    ref = RG.grok_decoded(window_args(args, window, reduce), 12, "window")
    sh = (1 << reduce) - 1
    full_win = (0, 0, w, h) if window is None else window
    x0, y0, x1, y1 = [(v + sh) >> reduce for v in full_win]
    if reduce == 0 and not args.get("irreversible"):
        assert RG.planes_sha([p[y0:y1, x0:x1] for p in planes]) == ref
    vcp, blocks = _parse_window(theirs, window, reduce)
    rec = oracle_decode(vcp, blocks, theirs)
    assert vcp.x0 <= x0 and vcp.y0 <= y0 and vcp.x1 >= x1 and vcp.y1 >= y1
    if window is not None:       # tile-granular: at most the touched tiles are decoded
        tw, th = args.get("tile", (w, h))
        assert (vcp.x1 - vcp.x0) <= ((-(-window[2] // tw) - window[0] // tw) * tw + sh) >> reduce
    assert RG.planes_sha([a[y0 - vcp.y0:y1 - vcp.y0, x0 - vcp.x0:x1 - vcp.x0] for a in rec]) == ref


@pytest.mark.parametrize("irreversible", [False, True])
def test_window_parse_keeps_exactly_the_blocks_a_window_can_depend_on(irreversible):
    """Block-granular selection inside the touched tiles (SURVEY 8f N3): code blocks whose coefficients cannot reach the
    window come back with length 0.  Random small windows of one image: every window's pixels equal the crop of the full
    decode, and most of the touched tiles' coded bytes are not needed."""
    args = dict(width=768, height=640, numcomps=1, prec=12, tile=(512, 512), numres=6, irreversible=irreversible)
    planes = synth(args, seed=21)
    theirs = RG.grok_codestream(oracle_codestream(args, planes), args, 21)
    fcp, fblocks = G.codestream_parse(theirs)
    full = oracle_decode(fcp, fblocks, theirs)
    rng = np.random.default_rng(7)
    saved = []
    for _ in range(8):
        x0, y0 = int(rng.integers(0, 700)), int(rng.integers(0, 580))
        win = (x0, y0, min(768, x0 + int(rng.integers(1, 90))), min(640, y0 + int(rng.integers(1, 70))))
        vcp, blocks = _parse_window(theirs, win, 0)
        rec = oracle_decode(vcp, blocks, theirs)
        a = rec[0][win[1] - vcp.y0:win[3] - vcp.y0, win[0] - vcp.x0:win[2] - vcp.x0]
        assert np.array_equal(a, full[0][win[1]:win[3], win[0]:win[2]]), win
        # against the same tiles parsed whole
        tiles_cp, tiles_blocks = _parse_window(theirs, (vcp.x0, vcp.y0, vcp.x1, vcp.y1), 0)
        saved.append(1.0 - blocks["length"].sum() / max(1, tiles_blocks["length"].sum()))
    assert min(saved) > 0.3 and np.mean(saved) > 0.6, saved


@pytest.mark.gpu
@pytest.mark.parametrize("args,window,reduce", WINDOW_CASES)
def test_gpu_window_and_reduce_decode_matches_grok(engine, args, window, reduce):
    planes = synth(args, seed=12)
    theirs = RG.grok_codestream(engine.encode_codestream(mk(args), planes, flags=G.CS_TLM | G.CS_PLT), args, 12)
    _, got = engine.decode_window(theirs, window, reduce)
    assert RG.planes_sha(got) == RG.grok_decoded(window_args(args, window, reduce), 12, "window")


@pytest.mark.gpu
def test_config5_random_rois_of_a_large_tiled_stream(engine):
    """configs[4] in shape: a TLM / PLT indexed code stream of 1024x1024 tiles, 8 seeded 2048x2048 windows at random
    positions; every window equals the crop of the source (lossless) -- here on an 8192x8192 canvas (64 tiles) so that the
    test stays in seconds; tools/config5_roi_bench.py runs the 32768x32768 version."""
    w = h = 8192
    cp = G.make_coding(w, h, 3, 12, numres=6, tile=(1024, 1024))
    base = P.synthetic_image(1024, 1024, 3, 12, seed=20260927)
    planes = [np.empty((h, w), np.int32) for _ in range(3)]
    for t in range(64):
        ty, tx = divmod(t, 8)
        for c in range(3):
            planes[c][ty * 1024:(ty + 1) * 1024, tx * 1024:(tx + 1) * 1024] = (base[c] + 37 * t) & 0xFFF
    cs = engine.encode_codestream(cp, planes, flags=G.CS_TLM | G.CS_PLT)
    rng = np.random.default_rng(20260927)
    for _ in range(8):
        x0, y0 = int(rng.integers(0, w - 2048)), int(rng.integers(0, h - 2048))
        _, got = engine.decode_window(cs, (x0, y0, x0 + 2048, y0 + 2048))
        for a, b in zip(got, planes):
            assert np.array_equal(a, b[y0:y0 + 2048, x0:x0 + 2048])
