"""CPU tests (-m "not gpu") of the host side: the C-ABI library loads and exports everything
include/grok_b200.h declares, the product's geometry/quantiser agree with the oracle, the
engine fails loudly without a GPU, and the tile-sharding logic works at world_size 2 (gloo)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import grok_b200 as G
import oracle_pipeline as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "grok_b200.h")).read()
    # the two entry points that take Grok's C++ callback type live beside its restated layout
    hdr += open(os.path.join(ROOT, "grok_b200", "csrc", "plugin_decode_abi.h")).read()
    hdr = hdr.replace("#define B2K_API __attribute__((visibility(\"default\")))", "")
    declared = set(re.findall(r"B2K_API[^;(]*?\b(\w+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = G.lib()
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, missing
    assert declared == set(G.EXPORTS)


_ABI_PROBE = r'''
#include <stdio.h>
#include <stddef.h>
%s
int main(void){
  printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu\n", sizeof(gpup_code_block), sizeof(gpup_compress_params),
   offsetof(gpup_compress_params, cblk_sty), sizeof(gpup_image_comp), sizeof(gpup_image), sizeof(gpup_tile), sizeof(gpup_band),
   sizeof(gpup_header_info), sizeof(gpup_decompress_params), sizeof(gpup_decompress_callback_info),
   offsetof(gpup_compress_params, apply_xyz_transform), sizeof(gpup_batch_memory_info), offsetof(gpup_batch_memory_info, source_format),
   sizeof(gpup_compress_callback_info), offsetof(gpup_compress_callback_info, host_data),
   sizeof(gpup_batch_decompress_memory_info), offsetof(gpup_batch_decompress_memory_info, pull),
   offsetof(gpup_batch_decompress_memory_info, rgb8_on_device));
  return 0; }'''
# measured from the reference's own gpu_plugin_shared.h (g++ 13, x86-64); re-checked live below when the tree is here
_ABI_REFERENCE = [1672, 12696, 4152, 40, 32, 24, 32, 312, 8272, 424, 12694, 56, 44, 96, 88, 368, 328, 360]


def _probe(include_line, flags, compiler):
    exe = "/tmp/b2k_abi_probe_%d" % os.getpid()
    subprocess.run([compiler, "-x", "c++" if compiler == "g++" else "c", "-", "-o", exe] + flags,
                   input=(_ABI_PROBE % include_line).encode(), check=True)
    return [int(v) for v in subprocess.check_output([exe]).split()]


def test_abi_struct_layout_matches_reference_contract():
    mine = _probe('#include "grok_b200.h"', ["-I", os.path.join(ROOT, "include")], "gcc")
    assert mine == _ABI_REFERENCE
    ref_dir = "/root/reference/src/lib/core/plugin/gpup"
    if os.path.isdir(ref_dir):
        theirs = _probe('#define GPUP_TYPES_ONLY\n#include "gpu_plugin_shared.h"', ["-I", ref_dir], "g++")
        assert theirs == mine


def test_engine_struct_sizes_match_ctypes():
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "grok_b200.h"
int main(void){ printf("%zu %zu %zu %zu\n", sizeof(b2k_coding), sizeof(b2k_block), offsetof(b2k_block, offset), sizeof(b2k_result)); return 0; }'''
    exe = "/tmp/b2k_abi_check_%d" % os.getpid()
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    vals = [int(v) for v in subprocess.check_output([exe]).split()]
    assert vals[0] == C.sizeof(G.Coding)
    assert vals[1] == C.sizeof(G.Block) == G.BLOCK_DTYPE.itemsize
    assert vals[2] == G.Block.offset.offset == G.BLOCK_DTYPE.fields["offset"][1]
    assert vals[3] == C.sizeof(G.Result)


@pytest.mark.parametrize("args", [
    dict(width=512, height=512, numcomps=1, prec=8),
    dict(width=2048, height=2048, numcomps=3, prec=12, tile=(1024, 1024)),
    dict(width=333, height=217, numcomps=3, prec=12, numres=4, origin=(3, 5)),
    dict(width=100, height=75, numcomps=4, prec=16, numres=3, tile=(61, 40), cblk=(32, 32)),
    dict(width=7, height=5, numcomps=1, prec=8, numres=6),
    dict(width=1000, height=600, numcomps=3, prec=10, numres=5, tile=(256, 256), origin=(17, 9), tile_origin=(5, 3),
         cblk=(16, 128)),
    dict(width=700, height=500, numcomps=3, prec=12, numres=5, tile=(512, 256), origin=(5, 11), precincts=[(128, 128)]),
    dict(width=513, height=300, numcomps=1, prec=10, numres=4, precincts=[(32, 64), (64, 32), (128, 128), (256, 256)],
         cblk=(64, 64)),
])
def test_geometry_matches_oracle(args):
    cp = G.make_coding(**args)
    mine = G.enumerate_blocks(cp)
    ref = P.enumerate_all(cp)
    assert len(mine) == len(ref)
    for gb, (t, c, ob) in zip(mine, ref):
        assert (gb["tile"], gb["comp"], gb["resno"], gb["orient"], gb["band_index"], gb["precno"], gb["cblkno"]) == \
               (t, c, ob.resno, ob.orient, ob.band_index, ob.precno, ob.cblkno)
        assert (gb["x0"], gb["y0"], gb["x1"], gb["y1"], gb["buf_x"], gb["buf_y"]) == \
               (ob.x0, ob.y0, ob.x1, ob.y1, ob.buf_x, ob.buf_y)
        kmax, step_enc, _ = P.band_params(cp, ob.resno, ob.orient)
        assert gb["kmax"] == kmax and gb["stepsize"] == np.float32(step_enc)


def test_irreversible_quantiser_matches_oracle():
    cp = G.make_coding(256, 256, 3, 12, numres=6, irreversible=True)
    for gb in G.enumerate_blocks(cp):
        kmax, step_enc, _ = P.band_params(cp, int(gb["resno"]), int(gb["orient"]))
        assert gb["kmax"] == kmax and gb["stepsize"] == np.float32(step_enc)


def test_config2_block_count():
    """SURVEY.md section 8a: 8192x8192x3, 1024 tiles, 6 resolutions, 64x64 blocks -> 49,728 blocks."""
    cp = G.make_coding(8192, 8192, 3, 12, numres=6, tile=(1024, 1024))
    assert len(G.enumerate_blocks(cp)) == 49728


def test_engine_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(G.EngineError) as e:
        G.Engine(0)
    assert "no CUDA device" in str(e.value)


def test_unsupported_coding_is_not_handled_not_an_error():
    cp = G.make_coding(64, 64, 1, 8, numres=17)  # more resolutions than the engine plans for: left to the host
    assert G.lib().b2k_enumerate(C.byref(cp), 1, 0, None, 0) < 0
    cp = G.make_coding(64, 64, 1, 8, numres=1)   # no wavelet level is fine (DC shift + colour transform only)
    assert G.lib().b2k_enumerate(C.byref(cp), 1, 0, None, 0) == 1


_WORKER = r'''
import os, sys
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, "tests"))
import numpy as np, torch, torch.distributed as dist
import grok_b200 as G
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% sys.argv[1], rank=int(sys.argv[2]), world_size=2)
rank = dist.get_rank()
cp = G.make_coding(4096, 3072, 3, 12, numres=6, tile=(1024, 1024))
mine = G.enumerate_blocks(cp, 2, rank)
full = G.enumerate_blocks(cp)
# every rank's share is exactly the blocks of its tiles, in order
assert np.array_equal(mine, full[full["tile"] %% 2 == rank])
counts = [torch.zeros(1, dtype=torch.int64) for _ in range(2)]
dist.all_gather(counts, torch.tensor([len(mine)], dtype=torch.int64))
assert int(sum(c.item() for c in counts)) == len(full)
# gather of variable-length "coded segments" to rank 0 in tile order (the codestream writer)
seg = torch.from_numpy(np.full(len(mine), rank, np.uint8))
sizes = [int(c.item()) for c in counts]
if rank == 0:
    bufs = [torch.zeros(s, dtype=torch.uint8) for s in sizes]
    dist.gather(seg, bufs, dst=0)
    assert all(int(b.float().mean().round().item()) == r for r, b in enumerate(bufs) if len(b))
else:
    dist.gather(seg, None, dst=0)
dist.barrier()
print("rank", rank, "ok")
'''


def test_tile_sharding_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % (ROOT, ROOT))
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), port, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_plugin_decode_callback_struct_matches_reference():
    """PluginDecodeCallbackInfo (std::string members: C++ ABI, plugin_interface.h L78-115) restated in
    grok_b200/csrc/plugin_decode_abi.h: same size and member offsets as the reference's own header."""
    probe = r'''
#include <cstdio>
#include <cstddef>
%s
int main(){ printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu\n", sizeof(PluginDecodeCallbackInfo), offsetof(PluginDecodeCallbackInfo, inputFile),
  offsetof(PluginDecodeCallbackInfo, header_info), offsetof(PluginDecodeCallbackInfo, image), offsetof(PluginDecodeCallbackInfo, tile),
  offsetof(PluginDecodeCallbackInfo, decompress_flags), offsetof(PluginDecodeCallbackInfo, codestream)); return 0; }'''

    def run(include, flags):
        exe = "/tmp/b2k_abi_dec_%d" % os.getpid()
        subprocess.run(["g++", "-std=c++20", "-w", "-x", "c++", "-", "-o", exe] + flags, input=(probe % include).encode(), check=True)
        return [int(v) for v in subprocess.check_output([exe]).split()]

    mine = run('#include "plugin_decode_abi.h"', ["-I", os.path.join(ROOT, "grok_b200", "csrc")])
    assert mine == [488, 16, 104, 416, 432, 444, 464]   # measured from the reference header (g++ 13, x86-64)
    ref = "/root/reference/src/lib/core"
    if os.path.isdir(ref):
        theirs = run('#include "plugin_interface.h"\nusing namespace grk;',
                     ["-I", ref + "/plugin", "-I", ref + "/plugin/gpup", "-I", ref, "-I", ref + "/util",
                      "-I", os.path.join(ROOT, "oracle", "ref_shim")])
        assert theirs == mine


def test_stock_symbols_exported():
    lib = G.lib()
    for s in ("minpf_post_load_plugin", "plugin_init", "plugin_get_debug_state", "gpup_encode_mem", "gpup_tile_free",
              "plugin_decompress"):
        assert hasattr(lib, s), s


def test_host_pack_container_conversion(tmp_path):
    """host_pack.cpp (int32 planes <-> pinned 16-bit PCIe containers on a host thread pool): exact
    truncation / zero- and sign-extension over ragged widths, strides and 1/3/8 threads, nothing
    written outside the rows.  Built straight from the product source, no GPU involved."""
    exe = str(tmp_path / "host_pack_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "host_pack_check.cpp"),
                    os.path.join(ROOT, "grok_b200", "csrc", "host_pack.cpp"), "-o", exe, "-lpthread"], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


_WRITER_WORKER = r'''
import io, os, sys
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, "tests"))
import numpy as np, torch, torch.distributed as dist
import grok_b200 as G
import oracle_pipeline as P
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% sys.argv[1], rank=int(sys.argv[2]), world_size=2)
rank, world = dist.get_rank(), 2
w, h = 200, 136
cp = G.make_coding(w, h, 3, 8, numres=4, tile=(64, 64))
planes = P.synthetic_image(w, h, 3, 8, seed=77)
# this rank's tiles only: transform + block-code them with the oracle (the GPU engine's stand-in on a CPU box)
rects = P.tile_rects(cp)
my_tiles = [t for t in range(len(rects)) if t %% world == rank]
coefs = P.forward(cp, planes, tiles=my_tiles)
table = G.enumerate_blocks(cp, world, rank)
blks = P.enumerate_all(cp, tiles=my_tiles)
assert len(blks) == len(table)
chunks, off = [], 0
for i, (t, c, b) in enumerate(blks):
    data = P.encode_block(cp, coefs, rects[t], c, b)
    table[i]["length"], table[i]["offset"], table[i]["numbps"], table[i]["numpasses"] = len(data), off, 1, 1
    chunks.append(data)
    off += len(data)
arena = np.concatenate(chunks)
# gather block tables + byte arenas on the writer rank (sizes first: the segments are variable length)
sizes = [torch.zeros(2, dtype=torch.int64) for _ in range(world)]
dist.all_gather(sizes, torch.tensor([len(arena), len(table)], dtype=torch.int64))
sizes = [(int(s[0]), int(s[1])) for s in sizes]
def padded(a, n):                                    # gloo's gather wants equal sizes (NCCL's does not)
    t = torch.zeros(n, dtype=torch.uint8)
    t[:len(a)] = torch.from_numpy(a.copy())
    return t
nseg, ntab = max(n for n, _ in sizes), max(k for _, k in sizes) * G.BLOCK_DTYPE.itemsize
seg = padded(arena, nseg)
tab = padded(table.view(np.uint8).reshape(-1), ntab)
if rank == 0:
    segs = [torch.zeros(nseg, dtype=torch.uint8) for _ in sizes]
    tabs = [torch.zeros(ntab, dtype=torch.uint8) for _ in sizes]
    dist.gather(seg, segs, dst=0)
    dist.gather(tab, tabs, dst=0)
    segs = [s[:n] for s, (n, _) in zip(segs, sizes)]
    tabs = [t[:k * G.BLOCK_DTYPE.itemsize] for t, (_, k) in zip(tabs, sizes)]
    shards = [(np.frombuffer(tabs[r].numpy().tobytes(), dtype=G.BLOCK_DTYPE), segs[r].numpy()) for r in range(world)]
    merged = G.merge_shards(cp, shards)              # b2k_result_merge: full enumeration order, offsets rebased
    assert merged.num_tiles == len(rects) and merged.num_blocks == len(G.enumerate_blocks(cp))
    cs = G.codestream_write(cp, merged.blocks, merged.bytes, num_tiles=merged.num_tiles)   # ONE tiled codestream
    merged.free()
    from PIL import Image
    im = Image.open(io.BytesIO(cs.tobytes())); im.load()
    assert np.array_equal(np.asarray(im).astype(np.int64), np.stack(planes, axis=-1)), "OpenJPEG does not give the source back"
else:
    dist.gather(seg, None, dst=0)
    dist.gather(tab, None, dst=0)
dist.barrier()
# ---- per-rank writers: every rank packetises ITS tiles, the writer rank gets finished tile parts + their lengths ----
parts, lens = G.codestream_write_tiles(cp, table, arena, G.CS_TLM | G.CS_PLT, world, rank)
assert len(lens) == len(my_tiles) and int(lens.sum()) == len(parts)
ntiles = len(rects)
all_lens = [torch.zeros(ntiles, dtype=torch.int64) for _ in range(world)]
mine = torch.zeros(ntiles, dtype=torch.int64)
mine[torch.tensor(my_tiles)] = torch.from_numpy(lens.astype(np.int64))
dist.all_gather(all_lens, mine)
tile_len = sum(all_lens).numpy().astype(np.uint64)          # every tile's tile-part length, on every rank
if rank == 0:
    head = G.codestream_write_header(cp, G.CS_TLM | G.CS_PLT, tile_len)
    out = np.zeros(len(head) + int(tile_len.sum()) + 2, np.uint8)
    out[:len(head)] = head
    at = len(head) + np.concatenate([[0], np.cumsum(tile_len)]).astype(np.int64)
    pos = 0
    for t, n in zip(my_tiles, lens):                         # own tile parts: straight into place
        out[at[t]:at[t] + int(n)] = parts[pos:pos + int(n)]
        pos += int(n)
    buf = torch.zeros(int(sum(int(tile_len[t]) for t in range(ntiles) if t %% world == 1)), dtype=torch.uint8)
    dist.recv(buf, src=1)                                    # the other rank's tile parts, in its tile order
    pos = 0
    for t in range(1, ntiles, world):
        n = int(tile_len[t])
        out[at[t]:at[t] + n] = buf[pos:pos + n].numpy()
        pos += n
    out[-2:] = [0xFF, 0xD9]
    assert np.array_equal(out, cs), "header + per-rank tile parts differ from the merged writer's code stream"
else:
    dist.send(torch.from_numpy(parts.copy()), dst=0)
dist.barrier()
print("rank", rank, "ok")
'''


def test_sharded_ranks_gather_into_one_codestream_gloo(tmp_path):
    """world size 2, gloo: each rank codes the tiles t %% 2 == rank (oracle on the CPU), the variable-length segments
    and block tables are gathered on rank 0, which writes one tiled codestream that OpenJPEG decodes to the source."""
    pytest.importorskip("PIL.Image")
    script = tmp_path / "writer_worker.py"
    script.write_text(_WRITER_WORKER % (ROOT, ROOT))
    port = str(31500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), port, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=300)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_ht_bit_plane_limits_are_declined_with_a_reason():
    """GrkHTBandBitPlanesTest: the 32-bit HT block coder carries at most 30 magnitude bits.  Codings whose bands would
    need more (deep samples + guard bits + sub-band gain) are 'not handled' with a reason -- the host keeps them --
    rather than coded wrongly; the deepest supported one still enumerates."""
    lib = G.lib()
    ok = G.make_coding(256, 256, 3, 16, numres=6, numgbits=2)
    assert lib.b2k_enumerate(C.byref(ok), 1, 0, None, 0) > 0
    kmax = G.enumerate_blocks(ok)["kmax"]
    assert kmax.max() <= 29 and kmax.min() >= 1
    deep = G.make_coding(256, 256, 3, 16, numres=6, numgbits=7)       # 16 bits + RCT + gains + 7 guard bits: Kmax 27, fine
    assert lib.b2k_enumerate(C.byref(deep), 1, 0, None, 0) > 0 and G.enumerate_blocks(deep)["kmax"].max() == 27
    deep.qcd_explicit = 1                                                # a foreign QCD asking for 31 + 6 bit planes
    for i in range(16):
        deep.qcd_expn[i] = 31
    assert lib.b2k_enumerate(C.byref(deep), 1, 0, None, 0) < 0
    assert b"bit planes" in lib.b2k_last_error()
    for bad in (dict(prec=17), dict(numcomps=5), dict(cblk=(1024, 8)), dict(numres=17), dict(numres=0)):
        args = dict(width=64, height=64, numcomps=1, prec=8, numres=3)
        args.update(bad)
        assert lib.b2k_enumerate(C.byref(G.make_coding(**args)), 1, 0, None, 0) < 0, bad


def test_gpup_tile_tree_from_a_result_multi_tile_with_precincts():
    """b2k_result_to_gpup_tile (the per-tile seam of INTEGRATION.md section 2) without a GPU: a result built from
    oracle-coded blocks of a multi-tile image with user precincts is turned into the gpup_tile tree of each tile;
    walking it in Grok's order (plugin_bridge.cpp L62-111: comp -> res -> band -> precinct -> block) meets exactly the
    enumeration's blocks, with their rectangles, bytes, pass bookkeeping (rate = length - 1) and band step sizes."""
    from gpup_ctypes import GpupTile
    lib = G.lib()
    cp = G.make_coding(200, 150, 3, 8, numres=4, tile=(128, 96), precincts=[(32, 32), (64, 64)], cblk=(16, 16))
    planes = P.synthetic_image(200, 150, 3, 8, seed=5)
    coefs = P.forward(cp, planes)
    table = G.enumerate_blocks(cp)
    blks = P.enumerate_all(cp)
    rects = P.tile_rects(cp)
    chunks, off = [], 0
    for i, (t, c, b) in enumerate(blks):
        data = P.encode_block(cp, coefs, rects[t], c, b)
        table[i]["length"], table[i]["offset"], table[i]["numbps"], table[i]["numpasses"] = len(data), off, 1, 1
        chunks.append(data)
        off += len(data)
    arena = np.concatenate(chunks)
    r = G.Result()
    r.num_blocks, r.blocks = len(table), C.cast(table.ctypes.data, C.POINTER(G.Block))
    r.bytes, r.num_bytes, r.num_tiles = C.cast(arena.ctypes.data, C.POINTER(C.c_uint8)), len(arena), len(rects)
    lib.b2k_result_to_gpup_tile.restype = C.POINTER(GpupTile)
    lib.b2k_result_to_gpup_tile.argtypes = [C.POINTER(G.Coding), C.POINTER(G.Result), C.c_uint32]
    lib.gpup_tile_free.argtypes = [C.POINTER(GpupTile)]
    k = 0
    for t in range(len(rects)):
        tile = lib.b2k_result_to_gpup_tile(C.byref(cp), C.byref(r), t)
        assert tile, lib.b2k_last_error()
        T = tile.contents
        assert T.numComponents == 3
        for c in range(3):
            tc = T.tileComponents[c].contents
            assert tc.numResolutions == cp.numres
            for rr in range(cp.numres):
                res = tc.resolutions[rr].contents
                assert res.numBands == (1 if rr == 0 else 3)
                for b in range(res.numBands):
                    band = res.band[b].contents
                    assert band.orientation == (0 if rr == 0 else b + 1)
                    for p in range(band.numPrecincts):
                        prc = band.precincts[p].contents
                        for j in range(prc.numBlocks):
                            cb = prc.blocks[j].contents
                            row = table[k]
                            assert (row["tile"], row["comp"], row["resno"], row["band_index"], row["precno"], row["cblkno"]) == (t, c, rr, b, p, j)
                            assert (cb.x0, cb.y0, cb.x1, cb.y1) == (row["x0"], row["y0"], row["x1"], row["y1"])
                            assert cb.numPasses == 1 and cb.numBitPlanes == 1 and cb.compressedDataLength == row["length"]
                            assert cb.passes[0].rate == row["length"] - 1
                            have = np.ctypeslib.as_array(cb.compressedData, shape=(cb.compressedDataLength,))
                            assert np.array_equal(have, arena[int(row["offset"]):int(row["offset"]) + int(row["length"])])
                            assert band.stepsize == row["stepsize"]
                            k += 1
        lib.gpup_tile_free(tile)
    assert k == len(table)


def test_bench_reference_arm_runs_to_completion_and_prints_its_json_line():
    """`bench.py --impl reference` (the driver's anchor for vs_reference) must not rot: run it for one step on the CPU and
    parse the line.  Round 1's arm died with a NameError after doing all the work."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    line = json.loads(lines[0])
    assert line["impl"] == "reference"
    if "unavailable" in line:
        assert not os.path.exists(os.path.join(root, "oracle", "_ref", "grok", "bin", "libgrk_ref_bench.so"))
        return
    assert line["unit"] == "Mpixels/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "reference" and "grk_compress" in line["cpu_baseline"]["sample"]
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["steps"] == 1 and line["n_gpus"] == 1


def test_stock_parameters_give_the_hosts_precinct_sizes(tmp_path):
    """ADVICE r1 (high): with `-c [128,128]` style parameters (csty & 1, res_spec = 1 < numresolution) the host derives the
    coarser resolutions' precinct sizes by halving the last given one (CodeStreamCompress.cpp L793-825).  The coding the
    stock entry points derive (b2k_coding_from_gpup) must give the same exponents -- checked against what the real
    library wrote into its COD marker when it is built, else against the rule."""
    src = r'''
#include <stdio.h>
#include <string.h>
#include "grok_b200.h"
int main(void) {
  static gpup_compress_params p; static gpup_image im; static gpup_image_comp comps[3]; static int32_t px[4];
  memset(&p, 0, sizeof p);
  p.numlayers = 1; p.numgbits = 1; p.numresolution = 5; p.cblockw_init = 64; p.cblockh_init = 64; p.cblk_sty = 0x40;
  p.roi_compno = -1; p.mct = 1; p.csty = 1; p.res_spec = 1; p.prcw_init[0] = 128; p.prch_init[0] = 128;
  im.x1 = 600; im.y1 = 500; im.numcomps = 3; im.comps = comps;
  for (int c = 0; c < 3; ++c) { comps[c].w = 600; comps[c].h = 500; comps[c].stride = 600; comps[c].dx = comps[c].dy = 1; comps[c].prec = 12; comps[c].data = px; }
  b2k_coding cp;
  int rc = b2k_coding_from_gpup(&p, &im, 0, &cp);
  printf("%d", rc);
  for (int r = 0; r < 5; ++r) printf(" %d %d", cp.prcw_exp[r], cp.prch_exp[r]);
  p.res_spec = 2; p.prcw_init[1] = 1; p.prch_init[1] = 64;      /* runs down to 1-sample precincts: declined */
  printf(" %d", b2k_coding_from_gpup(&p, &im, 0, &cp));
  p.res_spec = 1; p.tile_size_on = 1; p.t_width = 256; p.t_height = 256;   /* tiles: only with allow_tiles */
  printf(" %d %d\n", b2k_coding_from_gpup(&p, &im, 0, &cp), b2k_coding_from_gpup(&p, &im, 1, &cp));
  return 0;
}'''
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    c = tmp_path / "probe.c"
    c.write_text(src)
    exe = str(tmp_path / "probe")
    subprocess.run(["gcc", str(c), "-I", os.path.join(root, "include"), "-L", os.path.join(root, "grok_b200"),
                    "-l:libgrokj2k_plugin.so", "-Wl,-rpath," + os.path.join(root, "grok_b200"), "-o", exe], check=True)
    out = [int(v) for v in subprocess.check_output([exe]).decode().split()]
    assert out[0] == 0
    exps = out[1:11]
    want = [3, 3, 4, 4, 5, 5, 6, 6, 7, 7]        # resolution 0..4: 128 >> (4 - r)
    assert exps == want
    assert out[11] == 1 and out[12] == 1 and out[13] == 0
    import grok_ref as R
    if R.available():
        R.init(2)
        planes = P.synthetic_image(600, 500, 3, 12, seed=3)
        cs, _ = R.compress(planes, 12, numres=5, precinct=(128, 128))
        cp2, _ = G.codestream_parse(np.frombuffer(bytes(cs), np.uint8))
        assert [v for r in range(5) for v in (cp2.prcw_exp[r], cp2.prch_exp[r])] == exps
