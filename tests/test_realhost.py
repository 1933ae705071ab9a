"""The plugin under the REAL host (VERDICT r1 item 3): libgrokj2k -- built from the reference's sources with its plugin
loader enabled -- dlopens grok_b200/libgrokj2k_plugin.so through its own minpf loader, resolves minpf_post_load_plugin /
plugin_init / gpup_encode_mem / plugin_decompress by name and routes grk_compress() / grk_decompress() through them.

* stock host (oracle/_ref/grok, unmodified sources): single-tile images (the stock contract);
* patched host (oracle/_ref/grok_patched = sources + baseline/patches/0001-multi-tile-plugin-encode-decode.patch):
  multi-tile images through gpup_encode_mem_tiles / plugin_decompress_codestream.
The assertion is the strongest one available: the code stream the host writes with the plugin's code blocks is
byte-identical to the one it writes on its own CPU path, and the pixels it hands back are identical.
Each case runs in a subprocess (tests/realhost_driver.py).  Without a GPU the same driver checks the fallback:
the plugin loads, plugin_init reports no device, the host compresses on the CPU."""
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


HOST_DIR = {"_ref": "grok", "_ref_patched": "grok_patched"}     # flavour -> oracle/_ref/<dir> (oracle/build_grok*.sh)


def built(flavour):
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", HOST_DIR[flavour], "bin", "libgrk_ref_bench.so"))


def run(case, flavour):
    env = dict(os.environ)
    if flavour == "_ref_patched":
        env["GROK_REF_FLAVOUR"] = "patched"
    else:
        env.pop("GROK_REF_FLAVOUR", None)
    p = subprocess.run([sys.executable, os.path.join(HERE, "realhost_driver.py"), json.dumps(case)], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    lines = [l for l in p.stdout.splitlines() if l.startswith("REALHOST ")]
    assert p.returncode == 0 and lines, "driver failed (rc %d)\n%s\n%s" % (p.returncode, p.stdout[-3000:], p.stderr[-3000:])
    return json.loads(lines[-1][len("REALHOST "):])


@pytest.mark.parametrize("flavour", ["_ref", "_ref_patched"])
def test_host_loads_the_plugin_and_falls_back_without_a_device(flavour):
    """CPU box: the loader finds the library, every symbol resolves, plugin_init says "no device", the host carries on
    on its own path (grok.cpp L1344-1370) -- and nothing crashes on the way."""
    if not built(flavour):
        pytest.skip("oracle/_ref/%s not built" % HOST_DIR[flavour])
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    r = run(dict(width=256, height=192, numcomps=3, prec=12, tile=[128, 128] if flavour == "_ref_patched" else None), flavour)
    assert r["cpu"]["lossless"]
    assert r["plugin_loaded"] is False
    assert r["plugin"]["enc_accelerated"] == 0 and r["plugin"]["codestream_identical"] and r["plugin"]["decode_identical"]


STOCK_CASES = [
    dict(width=512, height=512, numcomps=1, prec=8),                                   # BASELINE config 1
    dict(width=640, height=384, numcomps=3, prec=12),
    dict(width=600, height=500, numcomps=3, prec=12, numres=5, precinct=[128, 128]),    # res_spec < numresolution (ADVICE r1)
    dict(width=640, height=384, numcomps=3, prec=12, irreversible=True),
    dict(width=333, height=217, numcomps=4, prec=16, numres=4),
    dict(width=300, height=200, numcomps=3, prec=12, numres=1),                          # no wavelet level
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", STOCK_CASES)
def test_stock_host_compresses_and_decompresses_through_the_plugin(case):
    if not built("_ref"):
        pytest.skip("oracle/_ref/grok not built")
    r = run(case, "_ref")
    assert r["plugin_loaded"], "the host did not load / initialise the plugin"
    assert r["plugin"]["enc_accelerated"] == 1, "grk_compress did not take the plugin route"
    assert r["plugin"]["codestream_identical"], "code stream through the plugin differs from the host's own"
    assert r["plugin"]["dec_accelerated"] == 1, "grk_decompress did not take the plugin route"
    if case.get("irreversible"):
        assert r["plugin"]["decode_maxdiff"] <= 1
    else:
        assert r["plugin"]["decode_identical"] and r["cpu"]["lossless"]


PATCHED_CASES = [
    dict(width=640, height=384, numcomps=3, prec=12, tile=[256, 256]),
    dict(width=2048, height=2048, numcomps=3, prec=12, tile=[1024, 1024], seed=20260924),     # config 2's tiles
    dict(width=700, height=500, numcomps=4, prec=16, tile=[256, 128], numres=4),              # config 4 in small
    dict(width=640, height=384, numcomps=3, prec=12, tile=[256, 256], irreversible=True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATCHED_CASES)
def test_patched_host_multi_tile_through_the_plugin(case):
    if not built("_ref_patched"):
        pytest.skip("oracle/_ref/grok_patched not built")
    r = run(case, "_ref_patched")
    assert r["plugin_loaded"]
    assert r["plugin"]["enc_accelerated"] == 1, "multi-tile grk_compress did not take gpup_encode_mem_tiles"
    assert r["plugin"]["codestream_identical"]
    assert r["plugin"]["dec_accelerated"] == 1, "multi-tile grk_decompress did not take plugin_decompress_codestream"
    if case.get("irreversible"):
        assert r["plugin"]["decode_maxdiff"] <= 1
    else:
        assert r["plugin"]["decode_identical"] and r["cpu"]["lossless"]


@pytest.mark.gpu
def test_patched_host_still_serves_single_tile_through_the_stock_symbols():
    if not built("_ref_patched"):
        pytest.skip("oracle/_ref/grok_patched not built")
    r = run(dict(width=512, height=512, numcomps=1, prec=8), "_ref_patched")
    assert r["plugin_loaded"] and r["plugin"]["enc_accelerated"] == 1 and r["plugin"]["codestream_identical"]
    assert r["plugin"]["dec_accelerated"] == 1 and r["plugin"]["decode_identical"]


BATCH_CASES = [
    dict(batch=True, width=640, height=384, numcomps=3, prec=12, frames=5, odd_one=True),
    dict(batch=True, width=500, height=333, numcomps=3, prec=16, frames=4, numres=5),      # W * 3 * 2 bytes not 16-aligned
    dict(batch=True, width=512, height=256, numcomps=3, prec=12, frames=4, irreversible=True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", BATCH_CASES)
def test_stock_host_batch_interfaces_through_the_plugin(case):
    """grk_plugin_batch_memory_begin/_submit/_end and grk_plugin_batch_decompress_memory_begin/_end (grok.h; host side
    grok.cpp L1655-1857, L2094-2188) with the plugin loaded by the unmodified host: planar int32 frames (the host packs
    them pixel-interleaved, L1806-1836) and GRK_SOURCE_RGB48LE frames go in, the host runs T2 in the plugin's callback,
    and every code stream equals the one grk_compress() writes on its own; code streams go in through the pull callback,
    the frames that come back equal grk_decompress()'s."""
    if not built("_ref"):
        pytest.skip("oracle/_ref/grok not built")
    r = run(case, "_ref")
    assert r["declined_without_plugin"] == 1
    assert r["plugin_loaded"]
    for name in ("compress_planar", "compress_rgb48le"):
        assert r[name]["rc"] == 0, r
        assert r[name]["identical"], "%s: a batch code stream differs from the host's own" % name
    assert r["decompress"]["good"] == case["frames"], r
    assert r["decompress"]["maxdiff"] <= (1 if case.get("irreversible") else 0), r
    if case.get("odd_one"):
        assert r["decompress_odd"] == {"good": 2, "first_ok": True, "last_ok": True}, r


def test_batch_interfaces_decline_without_a_device():
    """no GPU: plugin_init fails, so both batch begins answer 1 and the caller stays on the CPU (grok.h)"""
    if not built("_ref"):
        pytest.skip("oracle/_ref/grok not built")
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    r = run(dict(batch=True, width=128, height=96, numcomps=3, prec=12, frames=2), "_ref")
    assert r["declined_without_plugin"] == 1 and r["plugin_loaded"] is False
    assert r["compress_planar"]["rc"] == 1 and r["compress_rgb48le"]["rc"] == 1
    assert r["decompress"]["good"] == -101
