"""Runs in a SUBPROCESS of tests/test_realhost.py (a crash of the host library must not take pytest down):
the real reference host -- stock (oracle/_ref/grok) or patched (oracle/_ref/grok_patched, GROK_REF_FLAVOUR=patched) --
first on its own CPU path, then with grok_b200/libgrokj2k_plugin.so loaded through its own plugin loader
(grk_initialize(plugin_path) + grk_plugin_init), and prints one JSON line comparing the two.

usage: python realhost_driver.py '<json case>'"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(HERE), HERE]
import grok_ref as R            # noqa: E402
import oracle_pipeline as P     # noqa: E402


def batch(case):
    """the host's in-memory batch interfaces with the plugin loaded: grk_plugin_batch_memory_* (frames in, code streams out)
    and grk_plugin_batch_decompress_memory_* (code streams in, frames out), against the host's own CPU results"""
    w, h, n, prec, nframes = case["width"], case["height"], case["numcomps"], case["prec"], case["frames"]
    frames = [P.synthetic_image(w, h, n, prec, seed=case.get("seed", 7) + f) for f in range(nframes)]
    kw = dict(numres=case.get("numres", 6), irreversible=case.get("irreversible", False))
    out = {"flavour": R.FLAVOUR}
    R.init(case.get("threads", 4))
    cpu = [R.compress(f, prec, **kw)[0].copy() for f in frames]
    out["declined_without_plugin"] = R.batch_compress(frames, prec, **kw)[0]
    out["plugin_loaded"] = bool(R.init(case.get("threads", 4), plugin_path=R.PLUGIN_DIR, device_id=0))
    for name, rgb48 in (("planar", False), ("rgb48le", True)):
        rc, streams, sec = R.batch_compress(frames, prec, rgb48=rgb48, **kw)
        out["compress_" + name] = {"rc": rc, "seconds": sec, "identical": bool(
            rc == 0 and all(a.size == b.size and np.array_equal(a, b) for a, b in zip(streams, cpu)))}
    good, decoded, sec = R.batch_decompress(cpu, w, h, n)
    ref = [R.decompress(c, w, h, n)[0] for c in cpu]     # batch over: this decompresses per call again
    out["decompress"] = {"good": good, "seconds": sec, "maxdiff": int(max(
        np.abs(a.astype(np.int64) - b).max() for fa, fb in zip(decoded, ref) for a, b in zip(fa, fb)))}
    # a frame of another shape inside the batch fails alone (NULL image), the others still arrive
    if case.get("odd_one"):
        other = R.compress(P.synthetic_image(w // 2, h, n, prec, seed=3), prec, **kw)[0].copy()
        good, decoded, _ = R.batch_decompress([cpu[0], other, cpu[-1]], w, h, n)
        out["decompress_odd"] = {"good": good, "first_ok": bool(all(np.array_equal(a, b) for a, b in zip(decoded[0], ref[0]))),
                                 "last_ok": bool(all(np.array_equal(a, b) for a, b in zip(decoded[2], ref[-1])))}
    print("REALHOST " + json.dumps(out))


def main():
    case = json.loads(sys.argv[1])
    if case.get("batch"):
        return batch(case)
    w, h, n, prec = case["width"], case["height"], case["numcomps"], case["prec"]
    kw = dict(tile=tuple(case["tile"]) if case.get("tile") else None, numres=case.get("numres", 6),
              irreversible=case.get("irreversible", False), tlm=True, plt=True,
              precinct=tuple(case["precinct"]) if case.get("precinct") else None)
    planes = P.synthetic_image(w, h, n, prec, seed=case.get("seed", 7))
    threads = case.get("threads", 4)
    out = {"flavour": R.FLAVOUR}
    # 1. the host alone
    R.init(threads)
    cs_cpu, t_enc_cpu = R.compress(planes, prec, **kw)
    cs_cpu = cs_cpu.copy()
    dec_cpu, t_dec_cpu, _ = R.decompress(cs_cpu, w, h, n)
    out["cpu"] = {"enc_s": t_enc_cpu, "dec_s": t_dec_cpu, "bytes": int(cs_cpu.size),
                  "lossless": bool(all(np.array_equal(a, b) for a, b in zip(dec_cpu, planes)))}
    # 2. the same host with the plugin loaded by its own loader
    loaded = R.init(threads, plugin_path=R.PLUGIN_DIR, device_id=0)
    out["plugin_loaded"] = bool(loaded)
    f0 = R.accelerated_frames()
    cs_gpu, t_enc = R.compress(planes, prec, device_id=0, **kw)
    cs_gpu = cs_gpu.copy()
    f1 = R.accelerated_frames()
    dec_gpu, t_dec, _ = R.decompress(cs_cpu, w, h, n, device_id=0)
    f2 = R.accelerated_frames()
    for _ in range(case.get("repeat", 0)):      # steady-state timing through the host
        _, t_enc = R.compress(planes, prec, device_id=0, **kw)
        _, t_dec, _ = R.decompress(cs_cpu, w, h, n, device_id=0, out=dec_gpu)
    out["plugin"] = {"enc_s": t_enc, "dec_s": t_dec, "enc_accelerated": f1 - f0, "dec_accelerated": f2 - f1,
                     "codestream_identical": bool(cs_gpu.size == cs_cpu.size and np.array_equal(cs_gpu, cs_cpu)),
                     "bytes": int(cs_gpu.size),
                     "decode_identical": bool(all(np.array_equal(a, b) for a, b in zip(dec_gpu, dec_cpu))),
                     "decode_maxdiff": int(max(np.abs(a.astype(np.int64) - b).max() for a, b in zip(dec_gpu, dec_cpu)))}
    print("REALHOST " + json.dumps(out))


if __name__ == "__main__":
    main()
