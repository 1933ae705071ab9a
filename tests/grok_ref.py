"""ctypes binding of oracle/_ref/grok/bin/libgrk_ref_bench.so: the UNMODIFIED reference library
(libgrokj2k, built by oracle/build_grok.sh from the Grok source tree) driven through its public API --
grk_compress() into a memory stream, grk_decompress() from one (baseline/grk_ref_bench.cpp).

Test / measurement infrastructure only: tests/, bench.py's reference arm and cpu_baseline leg.
`available()` is False when the reference was not built (no Grok source tree at build time)."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# GROK_REF_FLAVOUR=patched selects the host built with baseline/patches/ applied (oracle/build_grok_patched.sh)
FLAVOUR = "grok_patched" if os.environ.get("GROK_REF_FLAVOUR") == "patched" else "grok"
BIN = os.path.join(ROOT, "oracle", "_ref", FLAVOUR, "bin")
LIB = os.path.join(BIN, "libgrk_ref_bench.so")
PLUGIN_DIR = os.path.join(ROOT, "grok_b200")     # holds libgrokj2k_plugin.so, the name the host's loader looks for


class Params(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("w", "h", "ncomp", "prec", "sgnd", "tile_w", "tile_h", "numres", "cblk_w", "cblk_h",
                                          "irreversible", "mct", "ht", "tlm", "plt")] + \
               [("device_id", C.c_int32), ("numgbits", C.c_uint32), ("prc_w", C.c_uint32), ("prc_h", C.c_uint32)]


_lib = None


def available():
    return os.path.exists(LIB) and os.path.exists(os.path.join(BIN, "libgrokj2k.so.1"))


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError("oracle/_ref/%s is not built (build() does it where the Grok source tree is)" % FLAVOUR)
        L = C.CDLL(LIB)
        L.grb_init.restype = C.c_int
        L.grb_init.argtypes = [C.c_uint32, C.c_char_p, C.c_int32]
        L.grb_compress.restype = C.c_double
        L.grb_compress.argtypes = [C.POINTER(Params), C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.grb_decompress.restype = C.c_double
        L.grb_decompress.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                     C.c_int32, C.c_uint32, C.POINTER(C.c_double)]
        L.grb_batch_compress.restype = C.c_int
        L.grb_batch_compress.argtypes = [C.POINTER(Params), C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                         C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_double)]
        L.grb_batch_decompress.restype = C.c_int
        L.grb_batch_decompress.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32,
                                           C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_double)]
        L.grb_accelerated_frames.restype = C.c_uint64
        L.grb_plugin_set_enabled.argtypes = [C.c_int]
        _lib = L
    return _lib


def accelerated_frames():
    return int(lib().grb_accelerated_frames())


def plugin_set_enabled(on):
    lib().grb_plugin_set_enabled(int(bool(on)))


def init(threads=0, plugin_path=None, device_id=0):
    """grk_initialize(plugin_path, threads); returns True when a plugin was loaded and initialised."""
    return bool(lib().grb_init(threads, plugin_path.encode() if plugin_path else None, device_id))


def compress(planes, prec, sgnd=False, tile=None, numres=6, irreversible=False, mct=None, ht=True, tlm=False, plt=False,
             cblk=(64, 64), device_id=-1, precinct=None, out=None):
    """-> (codestream bytes as np.uint8 array, seconds inside grk_compress())"""
    planes = [np.ascontiguousarray(p, dtype=np.int32) for p in planes]
    h, w = planes[0].shape
    n = len(planes)
    p = Params(w=w, h=h, ncomp=n, prec=prec, sgnd=int(sgnd), tile_w=tile[0] if tile else 0, tile_h=tile[1] if tile else 0,
               numres=numres, cblk_w=cblk[0], cblk_h=cblk[1], irreversible=int(irreversible),
               mct=int(n >= 3 if mct is None else mct), ht=int(ht), tlm=int(tlm), plt=int(plt), device_id=device_id,
               numgbits=0, prc_w=precinct[0] if precinct else 0, prc_h=precinct[1] if precinct else 0)
    cap = w * h * n * 4 + (1 << 20)
    if out is None or out.size < cap:
        out = np.empty(cap, np.uint8)
    ptrs = (C.c_void_p * n)(*[q.ctypes.data for q in planes])
    ln = C.c_uint64(0)
    sec = lib().grb_compress(C.byref(p), ptrs, w, out.ctypes.data, out.size, C.byref(ln))
    if sec < 0:
        raise RuntimeError("grk_compress failed (%g)" % sec)
    return out[:ln.value], sec


def decompress(cs, w, h, ncomp, device_id=-1, reduce=0, out=None):
    """-> (planes, seconds from grk_decompress() to the composite image, header seconds)"""
    cs = np.ascontiguousarray(cs, dtype=np.uint8)
    if out is None:
        out = [np.zeros((h, w), np.int32) for _ in range(ncomp)]
    ptrs = (C.c_void_p * ncomp)(*[q.ctypes.data for q in out])
    hs = C.c_double(0)
    sec = lib().grb_decompress(cs.ctypes.data, cs.size, ptrs, out[0].strides[0] // 4, ncomp, w, h, device_id, reduce, C.byref(hs))
    if sec < 0:
        raise RuntimeError("grk_decompress failed (%g)" % sec)
    return out, sec, hs.value


def batch_compress(frames, prec, rgb48=False, numres=6, irreversible=False, mct=None, cblk=(64, 64)):
    """grk_plugin_batch_memory_begin / _submit / _end (grok.h) over `frames` (each a list of int32 planes of one shape).
    -> (return code: 0 ran, 1 the plugin declined, <0 failure; list of code streams; seconds)"""
    frames = [[np.ascontiguousarray(p, dtype=np.int32) for p in f] for f in frames]
    h, w = frames[0][0].shape
    n = len(frames[0])
    p = Params(w=w, h=h, ncomp=n, prec=prec, sgnd=0, tile_w=0, tile_h=0, numres=numres, cblk_w=cblk[0], cblk_h=cblk[1],
               irreversible=int(irreversible), mct=int(n >= 3 if mct is None else mct), ht=1, tlm=0, plt=0, device_id=0,
               numgbits=0, prc_w=0, prc_h=0)
    cap = w * h * n * 4 + (1 << 20)
    out = np.zeros((len(frames), cap), np.uint8)
    lens = (C.c_uint64 * len(frames))()
    ptrs = (C.c_void_p * (n * len(frames)))(*[q.ctypes.data for f in frames for q in f])
    sec = C.c_double(0)
    rc = lib().grb_batch_compress(C.byref(p), ptrs, w, len(frames), int(rgb48), out.ctypes.data, cap, lens, C.byref(sec))
    return rc, [out[i, :lens[i]].copy() for i in range(len(frames))], sec.value


def batch_decompress(streams, w, h, ncomp):
    """grk_plugin_batch_decompress_memory_begin / _end over code streams of one shape.
    -> (frames that came back good, or a negative code: -101 = the plugin declined; decoded frames; seconds)"""
    streams = [np.ascontiguousarray(s, dtype=np.uint8) for s in streams]
    blob = np.concatenate(streams)
    offs = (C.c_uint64 * (len(streams) + 1))(*np.concatenate([[0], np.cumsum([s.size for s in streams])]).tolist())
    out = [[np.zeros((h, w), np.int32) for _ in range(ncomp)] for _ in streams]
    ptrs = (C.c_void_p * (ncomp * len(streams)))(*[q.ctypes.data for f in out for q in f])
    sec = C.c_double(0)
    rc = lib().grb_batch_decompress(blob.ctypes.data, offs, len(streams), ptrs, w, ncomp, w, h, C.byref(sec))
    return rc, out, sec.value


def cli_env(extra=None):
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = BIN + os.pathsep + env.get("LD_LIBRARY_PATH", "")
    if extra:
        env.update(extra)
    return env


def run_cli(tool, args, env=None, timeout=600):
    """Run oracle/_ref/grok/bin/<tool> (grk_compress / grk_decompress / grk_dump); returns CompletedProcess."""
    return subprocess.run([os.path.join(BIN, tool)] + list(args), env=cli_env(env), stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=timeout)
