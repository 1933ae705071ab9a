"""What the reference computed, kept as SHA-256 digests (tests/golden/reference_digests.json) and a few
small arrays (tests/golden/reference_outputs.npz), so that the tests that compare with Grok run without it.
tests/golden/make_reference_golden.py writes both from the reference's own kernels (oracle/_ref) and
library (oracle/_ref/grok).  A digest stands for an exact comparison: the array or byte string computed here
must hash to what the reference produced."""
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DIGESTS = os.path.join(GOLD, "reference_digests.json")
OUTPUTS = os.path.join(GOLD, "reference_outputs.npz")

_digests = None


def sha(a):
    """Digest of a byte string, or of an array's values as int32 (codestreams: as uint8)."""
    if isinstance(a, (bytes, bytearray)):
        return hashlib.sha256(bytes(a)).hexdigest()
    a = np.asarray(a)
    a = np.ascontiguousarray(a, dtype=np.uint8 if a.dtype == np.uint8 else np.int32)
    return hashlib.sha256(a.tobytes()).hexdigest()


def planes_sha(planes):
    return [sha(p) for p in planes]


def key(what, args, seed):
    return "%s %s seed=%d" % (what, json.dumps(args, sort_keys=True), seed)


def digests():
    global _digests
    if _digests is None:
        with open(DIGESTS) as f:
            _digests = json.load(f)
    return _digests


def outputs():
    return np.load(OUTPUTS)


def grok_codestream(ours, args, seed):
    """grk_compress's code stream for `args` and the image of `seed`, rebuilt from ours and Grok's COM marker
    segment ('Created by Grok ...', the one segment ours lacks).  Fails unless ours is byte-identical to Grok's
    stream with that segment removed."""
    g = digests()["codestream"][key("codestream", args, seed)]
    ours = bytes(ours)
    theirs = ours[:g["com_at"]] + bytes.fromhex(g["com"]) + ours[g["com_at"]:]
    assert sha(theirs) == g["sha256"], "code stream differs from grk_compress's"
    return np.frombuffer(theirs, np.uint8)


def grok_decoded(args, seed, what="decoded"):
    """Digests (one per component) of what grk_decompress gave back for Grok's stream of `args` / `seed`."""
    return digests()[what][key(what, args, seed)]
