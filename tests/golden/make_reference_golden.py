#!/usr/bin/env python3
"""Writes tests/golden/reference_digests.json and tests/golden/reference_outputs.npz (read through
tests/reference_golden.py) from the reference itself, on the inputs the tests use:

  oracle, refine   the reference's HT coder and forward DWTs (oracle/_ref/libgrok_ref.so, `make -C oracle ref`)
                   on the seeded blocks and tiles of tests/test_oracle.py's *_vs_reference_live tests
  codestream       grk_compress's code streams (libgrokj2k, oracle/build_grok.sh) for the images of
                   tests/test_interop.py: SHA-256 of the whole stream, and its COM marker segment with its offset
  decoded, window  digests of grk_decompress's images (windows: the crop of the reduced-resolution decode)
  npz              Grok's decode where a tolerance applies and the oracle's is not the same, as the difference
                   from the source image

Both reference builds need the Grok source tree, so this runs where it is; the tests need neither."""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import grok_b200 as G            # noqa: E402
import grok_ref as R             # noqa: E402
import oracle_lib as O           # noqa: E402
import oracle_pipeline as P      # noqa: E402
import reference_golden as RG    # noqa: E402
import test_interop as TI        # noqa: E402
import test_oracle as TO         # noqa: E402
from test_codestream import oracle_decode   # noqa: E402


def oracle_kernels():
    assert O.ref() is not None, "build oracle/_ref first (make -C oracle ref)"
    Rk = O.ref()
    blocks, tiles = TO.live_cases()
    enc, dec, dwt = [], [], []
    for sm, kmax in blocks:
        h, w = sm.shape
        ours = O.ht_encode(sm, kmax)
        theirs = [O.ref_ht_encode(sm, kmax, v) for v in (0, 1, 2)]
        assert all(t is None or np.array_equal(t, ours) for t in theirs)
        enc.append([None if t is None else RG.sha(t) for t in theirs])
        row = []
        for v in (0, 1, 2):
            rc2, d2 = O.ref_ht_decode(ours, kmax, w, h, v)
            row.append([int(rc2), RG.sha(d2)])
        dec.append(row)
    for (x0, y0, w, h, numres), src, fsrc in tiles:
        a = TO.dwt_fwd_aligned(Rk.ref_dwt53_fwd_2d, src.astype(np.int32), x0, y0, numres, 0)
        f = TO.dwt_fwd_aligned(Rk.ref_dwt97_fwd_2d, fsrc, x0, y0, numres, 0.0, 0)
        dwt.append([RG.sha(a), RG.sha(f.view(np.int32))])
    refine = []
    for w, h, M, sm in TO.refine_cases():
        row = {}
        for npass in (2, 3):
            for causal in (False, True):
                data, len2 = TO.refine_stream(sm, M, npass, causal)
                rc2, b = O.ref_ht_decode(data, M, w, h, variant=-1, num_passes=npass, len2=len2, causal=causal)
                assert rc2 == 0
                row["%d%d" % (npass, causal)] = [RG.sha(data), RG.sha(b)]
        refine.append(row)
    return {"ht_encode": enc, "ht_decode": dec, "dwt": dwt}, refine


def com_segment(cs):
    """offset and bytes of the one COM marker segment of Grok's main header"""
    cs = bytes(cs)
    i, found = 2, []
    while True:
        m, ln = (cs[i] << 8) | cs[i + 1], (cs[i + 2] << 8) | cs[i + 3]
        if m == 0xFF90:
            break
        if m == 0xFF64:
            found.append((i, cs[i:i + 2 + ln]))
        i += 2 + ln
    assert len(found) == 1
    return found[0]


class Interop:
    def __init__(self):
        assert R.available(), "build oracle/_ref/grok first (oracle/build_grok.sh)"
        R.init(os.cpu_count() or 1)
        self.d = {"codestream": {}, "decoded": {}, "window": {}}
        self.npz = {}

    def stream(self, args, seed, theirs):
        at, com = com_segment(theirs)
        theirs = bytes(theirs)
        assert TI.strip_com(theirs) == theirs[:at] + theirs[at + len(com):]
        self.d["codestream"][RG.key("codestream", args, seed)] = {"sha256": RG.sha(theirs), "com_at": at, "com": com.hex()}
        return np.frombuffer(theirs, np.uint8)

    def compress(self, args, seed, planes=None):
        planes = TI.synth(args, seed) if planes is None else planes
        return planes, self.stream(args, seed, TI.grok_compress(args, planes, R))

    def decoded(self, args, seed, theirs, reduce=0):
        w, h, n = args["width"], args["height"], args["numcomps"]
        out, _, _ = R.decompress(theirs, -(-w >> reduce), -(-h >> reduce), n, reduce=reduce)
        return out

    def run(self):
        for args in TI.REVERSIBLE + TI.IRREVERSIBLE:
            for seed in (5, 9):
                _, theirs = self.compress(args, seed)
                gd = self.decoded(args, seed, theirs)
                self.d["decoded"][RG.key("decoded", args, seed)] = RG.planes_sha(gd)
                if seed == 9 and args.get("irreversible"):    # the GPU test takes the oracle's decode for Grok's
                    cp2, blocks = G.codestream_parse(theirs)
                    assert RG.planes_sha(oracle_decode(cp2, blocks, theirs)) == RG.planes_sha(gd)
        self.compress(dict(width=600, height=500, numcomps=3, prec=12, numres=5, grok_precinct=(128, 128)), 5)
        args = dict(width=320, height=256, numcomps=3, prec=8, irreversible=True)
        planes, theirs = self.compress(args, 5)
        gd = self.decoded(args, 5, theirs)
        self.d["decoded"][RG.key("decoded", args, 5)] = RG.planes_sha(gd)
        self.npz["decoded_8bit_irreversible_minus_source"] = np.stack(gd).astype(np.int64) - np.stack(planes)
        self.compress(dict(width=2048, height=2048, numcomps=3, prec=12, tile=(1024, 1024)), 20260924,
                      P.synthetic_image(2048, 2048, 3, 12, seed=20260924))
        for args, window, reduce in TI.WINDOW_CASES:
            _, theirs = self.compress(args, 12)
            ref = self.decoded(args, 12, theirs, reduce)
            sh = (1 << reduce) - 1
            x0, y0, x1, y1 = [(v + sh) >> reduce for v in ((0, 0, args["width"], args["height"]) if window is None else window)]
            self.d["window"][RG.key("window", TI.window_args(args, window, reduce), 12)] = RG.planes_sha([b[y0:y1, x0:x1] for b in ref])
        for irreversible in (False, True):
            self.compress(dict(width=768, height=640, numcomps=1, prec=12, tile=(512, 512), numres=6, irreversible=irreversible), 21)
        self.config3()
        self.config4()

    def config3(self):
        a = TI.CONFIG3
        planes = P.synthetic_image(a["width"], a["height"], 3, 12, seed=20260925)
        cs, _ = R.compress(planes, 12, numres=6, irreversible=True, tlm=True, plt=True)
        theirs = self.stream(a, 20260925, cs)
        gd = self.decoded(a, 20260925, theirs)
        self.d["decoded"][RG.key("decoded", a, 20260925)] = RG.planes_sha(gd)
        cp2, blocks = G.codestream_parse(theirs)
        assert RG.planes_sha(oracle_decode(cp2, blocks, theirs)) == RG.planes_sha(gd)

    def config4(self):
        a = TI.CONFIG4
        w, h = a["width"], a["height"]
        base = P.synthetic_image(1024, 1024, 4, 16, seed=20260926)
        planes = [np.empty((h, w), np.int32) for _ in range(4)]
        for t in range(256):
            ty, tx = divmod(t, 16)
            for c in range(4):
                planes[c][ty * 1024:(ty + 1) * 1024, tx * 1024:(tx + 1) * 1024] = (base[c] + 257 * t) & 0xFFFF
        cs, _ = R.compress(planes, 16, tile=(1024, 1024), numres=6, tlm=True, plt=True, mct=1)
        self.stream(a, 20260926, cs)


def main():
    oracle, refine = oracle_kernels()
    it = Interop()
    it.run()
    for k, v in it.npz.items():
        assert np.abs(v).max() < 128, k
        it.npz[k] = v.astype(np.int8)
    with open(RG.DIGESTS, "w") as f:
        json.dump(dict(oracle=oracle, refine=refine, **it.d), f, indent=0, sort_keys=True)
        f.write("\n")
    np.savez_compressed(RG.OUTPUTS, **it.npz)


if __name__ == "__main__":
    main()
