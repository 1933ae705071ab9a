#!/usr/bin/env python3
"""bench.py -- Mpixels/s of the HTJ2K tile-engine hot path on BASELINE.json's config 2.

Workload (config.workload): 8192x8192, 3 components, 12 bit unsigned, 1024x1024 tiles, 5/3 + RCT,
6 resolutions, 64x64 code blocks, HT cleanup coding, lossless.  One STEP = encode the image
(DC shift + RCT + 5-level DWT + HT block coding of 49,728 blocks) and decode it back (HT decode +
inverse DWT + inverse RCT).  Mpixels/s = image pixels / step time, so every pixel is encoded AND
decoded once per step.

  value   device-resident: planes already in HBM, coded blocks stay in HBM (b2k_job_* stages)
  e2e     through the reference-facing C ABI with HOST (pinned) buffers: b2k_encode() then
          b2k_decode(), host<->device copies inside the timed region
  roofline  the dominant memory-bound kernel: the fused DC-shift + RCT + level-1 5/3 DWT
          (k_dwt53_fwd<3>): algorithmic bytes = samples x 8 B (one 4-byte read + one 4-byte
          write per sample per level, SURVEY.md 8d) / CUDA-event duration of that launch
  cpu_baseline  the UNMODIFIED reference library (oracle/_ref/grok/bin/libgrokj2k.so.1, built from
          Grok's sources by oracle/build_grok.sh): grk_compress() into a memory stream +
          grk_decompress() from it (grok.cpp L1025 ff.; harness baseline/grk_ref_bench.cpp), same
          image, all host threads and one thread; the round-1 kernel composite (oracle/_ref) is
          kept as a second, labelled figure

`--impl reference` times that CPU path (grk_compress + grk_decompress) as the step.  N>1 (torchrun): one process per GPU, each
rank runs the whole workload on its own image ("weak": tiles shard with no data-path
collective; NCCL only carries the barrier / max-reduction and the coded-size gather).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

W = H = 8192
NCOMP, PREC, NUMRES, TILE = 3, 12, 6, 1024
SEED = 20260924
METRIC = "Mpixels/s encode+decode 8K RGB 12-bit HTJ2K; DWT HBM GB/s vs roofline"
WORKLOAD = ("8192x8192x3 12-bit HTJ2K lossless (5/3 + RCT), 1024x1024 tiles, 6 resolutions, 64x64 blocks; "
            "step = encode + decode of the whole image")


def make_image():
    """SURVEY.md 8d config-2 generator (global coordinates), int32 planar."""
    import oracle_pipeline as P
    return P.synthetic_image(W, H, NCOMP, PREC, SEED)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, indices, enabled=True):
        """one nvidia-smi process for all the job's GPUs, on rank 0 only (eight pollers contend in the driver)"""
        self.index, self.proc, self.lines = ",".join(str(i) for i in indices), None, []
        self.mark0 = self.mark1 = None
        self.enabled = enabled

    def start(self):
        if not self.enabled:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.index, "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_ready(self, timeout=20.0):
        """nvidia-smi takes a second or two to start (and perturbs the GPUs while it does): start it
        before the warm-up and do not enter the timed region until it is streaming."""
        t0 = time.time()
        while self.proc and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.05)

    def begin(self):
        self.mark0 = len(self.lines)

    def end(self):
        time.sleep(0.06)
        self.mark1 = len(self.lines)

    def stop(self):
        if not self.enabled:
            return None
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines[self.mark0:self.mark1] if self.mark0 is not None else self.lines
        for l in lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
def cpu_reference_setup(planes):
    """Block list of one tile + output slots for the oracle/_ref threaded driver."""
    import oracle_lib as O
    import oracle_pipeline as P
    import grok_b200 as G
    R = O.ref()
    if R is None:
        return None
    cp1 = G.make_coding(TILE, TILE, NCOMP, PREC, numres=NUMRES)

    class Desc(C.Structure):
        _fields_ = [("comp", C.c_uint32), ("buf_x", C.c_uint32), ("buf_y", C.c_uint32), ("w", C.c_uint32),
                    ("h", C.c_uint32), ("kmax", C.c_uint32)]
    blks = [(c, b) for (_, c, b) in P.enumerate_all(cp1) if b.x1 > b.x0 and b.y1 > b.y0]
    descs = (Desc * len(blks))()
    for i, (c, b) in enumerate(blks):
        kmax, _, _ = P.band_params(cp1, b.resno, b.orient)
        descs[i] = Desc(c, b.buf_x, b.buf_y, b.x1 - b.x0, b.y1 - b.y0, kmax)
    ntiles = (W // TILE) * (H // TILE)
    slot = 16384
    st = dict(R=R, descs=descs, nblocks=len(blks), ntiles=ntiles, slot=slot,
              coded=np.zeros((ntiles * len(blks), slot), np.uint8), lengths=np.zeros(ntiles * len(blks), np.uint32),
              ptrs=(C.c_void_p * NCOMP)(*[p.ctypes.data for p in planes]), stride=planes[0].strides[0] // 4,
              threads=os.cpu_count() or 1)
    R.ref_bench_encode.restype = C.c_double
    R.ref_bench_decode.restype = C.c_double
    R.ref_bench_encode.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_int,
                                   C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.c_void_p, C.c_int]
    R.ref_bench_decode.argtypes = [C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                   C.c_void_p, C.c_uint32, C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    return st


def cpu_reference_step(st):
    """One encode+decode of the whole image with the reference's kernels; returns (seconds, info)."""
    R = st["R"]
    te = R.ref_bench_encode(st["ptrs"], st["stride"], NCOMP, st["ntiles"], W // TILE, TILE, TILE, PREC, NUMRES,
                            C.cast(st["descs"], C.c_void_p), st["nblocks"], st["coded"].ctypes.data, st["slot"],
                            st["lengths"].ctypes.data, st["threads"])
    dwt = C.c_double()
    td = R.ref_bench_decode(NCOMP, st["ntiles"], TILE, TILE, PREC, NUMRES, C.cast(st["descs"], C.c_void_p), st["nblocks"],
                            st["coded"].ctypes.data, st["slot"], st["lengths"].ctypes.data, st["threads"], C.byref(dwt))
    return te + td, dict(enc_s=te, dec_s=td, coded_bytes=int(st["lengths"].sum()), inv_dwt_ms_per_tilecomp=dwt.value * 1e3)


def bind_to_gpu_numa_node(local, nlocal=1):
    """Best effort: run this rank (and first-touch its pinned buffers) on the NUMA node its GPU hangs off,
    so host<->device copies do not cross the socket interconnect.  Ranks whose GPUs share a node split that
    node's physical cores between them (each keeps both SMT siblings of its cores), so their host threads do
    not land on one another.  Returns (node, cpus given to this rank) or (None, 0)."""
    try:
        import torch

        def node_of(dev):
            prop = torch.cuda.get_device_properties(dev)
            bus = "%04x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
            return int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())

        node = node_of(local)
        if node < 0:
            return None, 0
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        ndev = min(nlocal, torch.cuda.device_count())
        peers = [d for d in range(ndev) if node_of(d) == node]
        if len(peers) > 1 and local in peers:
            cores = {}
            for c in cpus:
                try:
                    key = int(open("/sys/devices/system/cpu/cpu%d/topology/core_id" % c).read())
                except Exception:
                    key = c
                cores.setdefault(key, []).append(c)
            keys = sorted(cores)
            i, n = peers.index(local), len(peers)
            mine = keys[i * len(keys) // n:(i + 1) * len(keys) // n]
            cpus = [c for k in mine for c in cores[k]] or cpus
        os.sched_setaffinity(0, set(cpus))
        return node, len(cpus)
    except Exception:
        return None, 0


def cpu_quota():
    """CPUs' worth of time the container may use (cgroup cpu.max), or None."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            return q / per if q > 0 else None
        except Exception:
            return None



# ------------------------------------------------------------------------------------------------
# The reference itself: libgrokj2k's public API on memory streams (tests/grok_ref.py -> oracle/_ref/grok)
# ------------------------------------------------------------------------------------------------
def grok_setup(img, w=W, h=H):
    import grok_ref as R
    if not R.available():
        return None
    planes = [np.ascontiguousarray(p[:h, :w]) for p in img]
    return dict(R=R, planes=planes, w=w, h=h, buf=np.empty(w * h * NCOMP * 4 + (1 << 20), np.uint8),
                out=[np.zeros((h, w), np.int32) for _ in range(NCOMP)], threads=os.cpu_count() or 1, checked=False)


def grok_step(st):
    """One grk_compress() + grk_decompress() of the image (config-2 coding); returns (seconds, info).  Only the two
    library calls are timed (SURVEY.md 8d: no image construction, no file I/O)."""
    R = st["R"]
    R.init(st["threads"])
    cs, te = R.compress(st["planes"], PREC, tile=(TILE, TILE), numres=NUMRES, tlm=True, plt=True, out=st["buf"])
    out, td, _ = R.decompress(cs, st["w"], st["h"], NCOMP, out=st["out"])
    if not st["checked"]:
        assert all(np.array_equal(a, b) for a, b in zip(out, st["planes"])), "reference round trip is not lossless"
        st["checked"] = True
    return te + td, dict(enc_s=te, dec_s=td, codestream_bytes=int(len(cs)))


def grok_tune_threads(st):
    """All logical CPUs, or the cgroup quota's worth when the container has one (oversubscribing a quota only burns it)."""
    cands = [os.cpu_count() or 1]
    q = cpu_quota()
    if q and int(q) < cands[0]:
        # a container with a CPU-time quota: the quota's worth of threads, and twice that (never every logical CPU of a
        # 128-way host against a 16-CPU quota: that only burns the quota and the box's memory)
        cands = [max(1, int(q)), min(cands[0], 2 * max(1, int(q)))]
    if os.environ.get("B2K_REF_THREADS"):
        cands = [int(os.environ["B2K_REF_THREADS"])]
    best = None
    for t in cands:
        st["threads"] = t
        sec = min(grok_step(st)[0] for _ in range(2))
        if best is None or sec < best[0]:
            best = (sec, t)
    st["threads"] = best[1]
    return best[1]


def tune_reference_threads(st):
    """The reference arm gets whichever thread count serves it best here: every logical CPU, or -- when the
    container has a CPU-time quota that oversubscription would only burn -- the quota's worth."""
    cands = [os.cpu_count() or 1]
    q = cpu_quota()
    if q and int(q) < cands[0]:
        cands.append(max(1, int(q)))
    if os.environ.get("B2K_REF_THREADS"):
        cands = [int(os.environ["B2K_REF_THREADS"])]
    best = None
    for t in cands:
        st["threads"] = t
        sec = min(cpu_reference_step(st)[0] for _ in range(2))
        if best is None or sec < best[0]:
            best = (sec, t)
    st["threads"] = best[1]
    return best[1]


def cpu_model():
    try:
        for l in open("/proc/cpuinfo"):
            if l.startswith("model name"):
                return l.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation is the step (rank 0 only): grk_compress() into a
    memory stream + grk_decompress() from it, whole config-2 image, all the host threads it can use."""
    if rank != 0:
        return
    img = make_image()
    st = grok_setup(img)
    if st is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/grok (libgrokj2k built from Grok's sources) is not in the tree"}))
        return
    grok_tune_threads(st)
    for _ in range(args.warmup):
        grok_step(st)
    secs, encs, decs, info = [], [], [], None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sec, info = grok_step(st)
        secs.append(sec)
        encs.append(info["enc_s"])
        decs.append(info["dec_s"])
    wall = (time.perf_counter() - t0) / max(1, args.steps)
    dt = float(np.mean(secs))
    val = W * H / dt / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mpixels/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "timing": "steady_clock around grk_compress() and grk_decompress()+grk_decompress_get_image() only (mean of K steps); "
                                 "host wall clock per step incl. image construction and copies: %.1f ms" % (wall * 1e3),
                       "host": cpu_model(), "codestream_bytes": info["codestream_bytes"]},
            "encode_only": {"value": W * H / float(np.mean(encs)) / 1e6, "unit": "Mpixels/s", "ms": float(np.mean(encs)) * 1e3},
            "decode_only": {"value": W * H / float(np.mean(decs)) / 1e6, "unit": "Mpixels/s", "ms": float(np.mean(decs)) * 1e3},
            "cpu_baseline": {"value": val, "unit": "Mpixels/s", "cores": st["threads"], "cpu_quota": cpu_quota(), "kind": "reference",
                             "sample": "whole image (64 of 64 tiles) per step: grk_compress() + grk_decompress() of the unmodified "
                                       "libgrokj2k (oracle/_ref/grok) on memory streams, TLM + PLT, %d threads" % st["threads"]},
            "e2e": {"value": val, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def run_config4(args, rank, world, local):
    """--workload config4 (BASELINE.json configs[3]): ONE 16384x16384x4 16-bit lossless image, 256 tiles of 1024x1024
    sharded over the N ranks (tile t -> rank t % N, no data-path collective), STRONG scaling.  The timed step holds
    everything north_star names: every rank encodes its tiles from pinned host planes (b2k_encode with tile_mod / tile_rem),
    an NCCL all_gather of the segment sizes, the NCCL gather of the variable-length coded segments + block tables to the
    writer rank, b2k_result_merge and b2k_codestream_write (TLM + PLT) there.  value = image pixels / step time."""
    import torch
    import grok_b200 as G
    import oracle_pipeline as P
    torch.cuda.set_device(local)
    bind_to_gpu_numa_node(local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W4 = H4 = int(os.environ.get("B2K_CONFIG4_SIZE", "16384"))
    NC4, PREC4 = 4, 16
    cp = G.make_coding(W4, H4, NC4, PREC4, numres=NUMRES, tile=(TILE, TILE), mct=1)
    base = P.synthetic_image(TILE, TILE, NC4, PREC4, seed=20260926)
    reps = W4 // TILE
    # every rank holds the planes of the tiles it codes (the others' stay untouched zeros): 16-bit containers, pinned
    planes = [G.pinned_empty((H4, W4), np.uint16) for _ in range(NC4)]
    for t in range(reps * reps):
        if t % world == rank:
            ty, tx = divmod(t, reps)
            for c in range(NC4):
                planes[c][ty * TILE:(ty + 1) * TILE, tx * TILE:(tx + 1) * TILE] = (base[c] + 257 * t) & 0xFFFF
    eng = G.Engine(local)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    info = {}

    pinned_cache = {}

    def pinned_like(key, n):
        """pinned host landing buffers of the writer rank, kept between steps (re-pinning costs more than the copy)"""
        t = pinned_cache.get(key)
        if t is None or t.numel() < n:
            t = torch.empty(int(n * 1.1) + 4096, dtype=torch.uint8, pin_memory=True)
            pinned_cache[key] = t
        return t[:n]

    ntiles = reps * reps
    my_tiles = list(range(rank, ntiles, world))
    FL = G.CS_TLM | G.CS_PLT
    parts_buf = [None]

    def step():
        """sharded encode -> every rank packetises ITS tiles into finished tile parts (b2k_codestream_write_tiles) -> NCCL
        all_gather of the per-tile lengths -> grouped NCCL send / recv of the tile parts to the writer rank -> the writer
        lays header + tile parts (tile-index order) + EOC into one pinned buffer."""
        tp = [time.perf_counter()]
        res = eng.encode(cp, planes, tile_mod=world, tile_rem=rank)
        tp.append(time.perf_counter())
        if rank == 0:       # the writer needs every tile's length before it can place its own: lengths now, bytes below
            parts, lens = G.codestream_write_tiles(cp, res.blocks, res.bytes, FL, world, rank, sizes_only=True)
        else:
            if parts_buf[0] is None or parts_buf[0].size < res.num_bytes + (1 << 22):
                parts_buf[0] = G.pinned_empty((int(res.num_bytes * 1.1) + (1 << 22),), np.uint8)
            parts, lens = G.codestream_write_tiles(cp, res.blocks, res.bytes, FL, world, rank, out=parts_buf[0])
            res.free()
        tp.append(time.perf_counter())
        info["coded_bytes_rank0"] = int(res.num_bytes) if rank == 0 else 0
        mine = torch.zeros(ntiles, dtype=torch.int64, device="cuda")
        mine[torch.tensor(my_tiles, device="cuda")] = torch.from_numpy(lens.astype(np.int64)).cuda()
        if world > 1:
            dist.all_reduce(mine)                       # every tile's tile-part length on every rank (disjoint supports)
        tile_len = mine.cpu().numpy().astype(np.uint64)
        cs_len = 0
        if rank == 0:
            head = G.codestream_write_header(cp, FL, tile_len)
            total = len(head) + int(tile_len.sum()) + 2
            out_t = pinned_like(("cs", 0), total)
            out = out_t.numpy()
            out[:len(head)] = head
            at = len(head) + np.concatenate([[0], np.cumsum(tile_len)]).astype(np.int64)
            bufs = [None] * world
            if world > 1:
                bufs = [None] + [torch.empty(int(tile_len[r::world].sum()), dtype=torch.uint8, device="cuda") for r in range(1, world)]
                for w_ in dist.batch_isend_irecv([dist.P2POp(dist.irecv, bufs[r], r) for r in range(1, world)]):
                    w_.wait()
            tp.append(time.perf_counter())
            # own tiles: packetised straight into their places (host pool)
            G.codestream_write_tiles(cp, res.blocks, res.bytes, FL, world, rank, out=out, tile_at=at[my_tiles].astype(np.uint64))
            res.free()
            for r in range(1, world):                   # the others': device -> their place in the pinned code stream
                pos = 0
                for t in range(r, ntiles, world):
                    n = int(tile_len[t])
                    out_t[at[t]:at[t] + n].copy_(bufs[r][pos:pos + n], non_blocking=True)
                    pos += n
            torch.cuda.synchronize()
            out[total - 2:total] = [0xFF, 0xD9]
            tp.append(time.perf_counter())
            cs_len = total
            info["codestream"] = out[:total]
            info["phase_ms_rank0"] = dict(zip(["encode_own_tiles", "plan_own_tiles", "nccl_lengths_and_recv", "write_own_and_place_others"],
                                              [round((b_ - a_) * 1e3, 2) for a_, b_ in zip(tp, tp[1:])]))
        else:
            seg = torch.from_numpy(parts).cuda(non_blocking=True)
            for w_ in dist.batch_isend_irecv([dist.P2POp(dist.isend, seg, 0)]):
                w_.wait()
        return cs_len

    sampler = ClockSampler(range(int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))) if world > 1 else [local], enabled=(rank == 0))
    sampler.start()
    for _ in range(max(3, args.warmup)):
        step()
    sampler.wait_ready()
    barrier()
    sampler.begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cs_len = step()
    barrier()
    dt = (time.perf_counter() - t0) / args.steps
    sampler.end()
    clocks = sampler.stop()
    tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt[0])
    if rank == 0:
        # outside the timed region: the assembled code stream decodes to what the ranks were given (rank 0 checks its own tiles)
        cs_final = info.pop("codestream")
        _, rec = eng.decode_codestream(cs_final, dtype=np.uint16)
        for t in my_tiles[:8]:
            ty, tx = divmod(t, reps)
            for c in range(NC4):
                assert np.array_equal(rec[c][ty * TILE:(ty + 1) * TILE, tx * TILE:(tx + 1) * TILE],
                                      planes[c][ty * TILE:(ty + 1) * TILE, tx * TILE:(tx + 1) * TILE]), "config 4 code stream does not decode to the source"
        del rec
        pix = W4 * H4
        line = {"metric": "Mpixels/s encode %dx%dx4 16-bit HTJ2K lossless, 1024x1024 tiles sharded over the GPUs (BASELINE config 4)" % (W4, H4),
                "value": pix / dt / 1e6, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
                "config": {"workload": "config4: one %dx%dx4 16-bit lossless image (5/3 + RCT on components 0-2), %d tiles, tile t -> rank t %% N; "
                                       "step = sharded b2k_encode16 from pinned host planes + per-rank packetisation of the rank's tiles "
                                       "(b2k_codestream_write_tiles) + NCCL all_reduce of tile-part lengths + grouped NCCL send/recv of the "
                                       "finished tile parts to rank 0, which lays header (TLM) + tile parts + EOC into one pinned buffer" % (W4, H4, reps * reps),
                           "timing": "host wall clock around the K steps incl. barriers, max over ranks (the step ends on the host: the code stream is in host memory)",
                           "codestream_bytes": int(cs_len), **info},
                "e2e": {"value": pix / dt / 1e6, "unit": "Mpixels/s", "h2d_bytes_per_step": int(W4 * H4 * NC4 * 2), "d2h_bytes_per_step": int(cs_len)},
                "clocks": clocks}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="config2", choices=["config2", "config4"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the device-resident round trip returned in its last step "
                         "as DIR/<name>.npy (fixed seeded samples of the large arrays)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "config2"):
        ap.error("--dump-outputs covers the config2 GPU workload only")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "config4":
        run_config4(args, rank, world, local)
        return

    import torch
    import grok_b200 as G
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    numa, ncpus = bind_to_gpu_numa_node(local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    cp = G.make_coding(W, H, NCOMP, PREC, numres=NUMRES, tile=(TILE, TILE))
    img = make_image()
    # pinned host buffers: the image planes Grok would hand over (int32, 64-byte aligned rows) and the output
    planes = [G.pinned_empty((H, W), np.int32) for _ in range(NCOMP)]
    out = [G.pinned_empty((H, W), np.int32) for _ in range(NCOMP)]
    for p, q in zip(planes, img):
        p[:] = q
    eng = G.Engine(local)
    lib = G.lib()

    # ---------------- device-resident: `value` ----------------
    job = eng.job(cp)
    job.upload(planes)

    def device_step():
        _, st4, nbytes = job.roundtrip()   # fwd -> HT encode -> HT decode -> inverse, one synchronisation
        return tuple(st4), nbytes

    sampler = ClockSampler(range(int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))) if world > 1 else [local], enabled=(rank == 0))
    sampler.start()
    for _ in range(args.warmup):
        device_step()
    sampler.wait_ready()
    barrier()
    sampler.begin()
    l0 = lib.b2k_launch_count()
    t0 = time.perf_counter()
    # the K steps are queued back to back on the stream and synchronised once (b2k_job_roundtrip_n): per-step events
    # give the stage and level-1 kernel times, the host is not in the loop
    ms_dev, stage_sum, l1_sum, nbytes = job.roundtrip_n(args.steps)
    barrier()
    wall_dev = time.perf_counter() - t0     # host clock around the same region (reported next to the device time)
    dt_dev = ms_dev * 1e-3                  # CUDA events on the launching stream: first step's start to last step's end
    stage = np.array(stage_sum)
    lvl1 = [(l1_sum / args.steps, job.kernel_stats(0)[1])]
    launches = lib.b2k_launch_count() - l0
    job.download(out)
    assert all(np.array_equal(a, b) for a, b in zip(out, planes)), "device-resident round trip is not lossless"
    dumped = None
    if args.dump_outputs and rank == 0:
        res = job.fetch_result()
        dumped = sample_outputs(out, res)
        res.free()
    pipe = None
    if world == 1 or bool(os.environ.get("B2K_BENCH_ALL_LEGS")):
        # extra: the same K round trips with the block-coder stage pipelined over 2 block ranges on 2 streams
        # (b2k_job_roundtrip_pipelined_n); `value` stays the back-to-back schedule, whose stage times add up
        job.roundtrip_pipelined_n(2, 2, 2)
        ms_p, st_p, _, nb_p = job.roundtrip_pipelined_n(args.steps, 2, 2)
        job.download(out)
        assert nb_p == nbytes and all(np.array_equal(a, b) for a, b in zip(out, planes)), "pipelined round trip differs"
        pipe = {"ms_per_step": ms_p / args.steps, "value": W * H / (ms_p / args.steps * 1e-3) / 1e6, "unit": "Mpixels/s",
                "stage_ms": {"fwd_mct_dwt": st_p[0] / args.steps, "ht_encode_and_decode": st_p[1] / args.steps,
                             "inv_dwt_mct": st_p[2] / args.steps},
                "api": "b2k_job_roundtrip_pipelined_n: block-coder stage cut into 2 block ranges on 2 streams, transforms alone"}
    job.close()

    # ---------------- end to end through the C ABI with host buffers: `e2e` ----------------
    split = [0.0, 0.0]   # seconds inside b2k_encode / b2k_decode (both return with host buffers complete)

    def e2e_step():
        ta = time.perf_counter()
        res = eng.encode(cp, planes)
        tb = time.perf_counter()
        blocks, data = res.blocks, res.bytes
        eng.decode(cp, blocks, data, out)
        tc = time.perf_counter()
        split[0] += tb - ta
        split[1] += tc - tb
        nb, nbk = res.num_bytes, res.num_blocks
        res.free()
        return nb, nbk

    host_threads = G.set_host_threads(-1)   # default policy: the engine times packed vs direct on its first calls
    for _ in range(max(8, args.warmup)):
        e2e_step()
    pack_mode = G.host_pack_last()
    barrier()
    split[0] = split[1] = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        nb, nbk = e2e_step()
    barrier()
    dt_e2e = time.perf_counter() - t0
    dt_enc, dt_dec = split[0], split[1]
    sampler.end()
    clocks = sampler.stop()   # clocks / throttle reasons over both timed regions
    assert all(np.array_equal(a, b) for a, b in zip(out, planes)), "e2e round trip is not lossless"

    # the legs below are extras (other containers, files, streams): with several ranks on one host they only add pinned
    # memory and time to a run whose purpose is the scaling of `value` and `e2e`, so they run at N = 1 only
    extras = world == 1 or bool(os.environ.get("B2K_BENCH_ALL_LEGS"))
    dt_e2e32 = dt_file = dt_e2e16 = dt_stream = 0.0
    cs_len, n_stream = 0, 0
    if extras:
        # ---------------- same call with host packing off: the int32 planes cross PCIe as they are ----------------
        G.set_host_threads(0)
        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        barrier()
        dt_e2e32 = (time.perf_counter() - t0) / args.steps
        assert all(np.array_equal(a, b) for a, b in zip(out, planes)), "e2e (no host packing) round trip is not lossless"
        G.set_host_threads(-1)

        # ---------------- files: the same calls plus the host T2 step (codestream write / parse) ----------------
        cs_buf = G.pinned_empty((int(nb) + int(nb) // 8 + (1 << 20),), np.uint8)

        def file_step():
            cs = eng.encode_codestream(cp, planes, out=cs_buf)
            eng.decode_codestream(cs, out=out)
            return len(cs)

        for _ in range(3):
            file_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cs_len = file_step()
        barrier()
        dt_file = (time.perf_counter() - t0) / args.steps
        assert all(np.array_equal(a, b) for a, b in zip(out, planes)), "codestream round trip is not lossless"

        # ---------------- same, 16-bit sample containers (b2k_encode16 / b2k_decode16) ----------------
        p16 = [G.pinned_empty((H, W), np.uint16) for _ in range(NCOMP)]
        o16 = [G.pinned_empty((H, W), np.uint16) for _ in range(NCOMP)]
        for p, q in zip(p16, img):
            p[:] = q

        def e2e16_step():
            res = eng.encode(cp, p16)
            eng.decode(cp, res.blocks, res.bytes, o16)
            res.free()

        for _ in range(2):
            e2e16_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e16_step()
        barrier()
        dt_e2e16 = time.perf_counter() - t0
        assert all(np.array_equal(a, b) for a, b in zip(o16, p16)), "16-bit e2e round trip is not lossless"

        # ---------------- streamed (SURVEY 8f N2): an encode stream feeding a decode stream, 3 frames in flight each ----------------
        # 16-bit sample containers in and out (what the reference's batch interface carries, gpup_batch_memory_submit_planes):
        # frame k+1's upload overlaps frame k's kernels and download, and the decode of frame k-1 runs beside both
        depth = int(os.environ.get("B2K_BENCH_STREAM_DEPTH", "3"))
        outs = [[G.pinned_empty((H, W), np.uint16) for _ in range(NCOMP)] for _ in range(2 * depth + 1)]
        free_outs = list(range(len(outs)))
        lock, done, live, bad, used = threading.Lock(), threading.Semaphore(0), {}, [], set()
        room = threading.Semaphore(len(outs))

        def on_decoded(tag, status):
            res, slot = live.pop(tag)
            res.free()
            if status != 0:
                bad.append(status)
            with lock:
                free_outs.append(slot)
            room.release()
            done.release()

        dec_stream = G.DecodeStream(depth=depth, sample_bytes=2, on_decoded=on_decoded, device=local)

        def on_encoded(tag, res, status):
            if status != 0 or res is None:
                bad.append(status)
                done.release()
                return
            room.acquire()
            with lock:
                slot = free_outs.pop()
                used.add(slot)
            live[tag] = (res, slot)
            dec_stream.submit(cp, res.blocks, res.bytes, outs[slot], tag)

        enc_stream = G.EncodeStream(cp, depth=depth, sample_bytes=2, on_encoded=on_encoded, device=local)

        def streamed(nframes):
            t0 = time.perf_counter()
            for i in range(nframes):
                enc_stream.submit(p16, i)
            for _ in range(nframes):
                done.acquire()
            return time.perf_counter() - t0

        streamed(3 * depth + 3)           # warm-up: every worker's engine has built its job, the pinned result arenas exist
        barrier()
        n_stream = args.steps
        dt_stream = streamed(n_stream) / n_stream
        barrier()
        enc_stream.end()
        dec_stream.end()
        assert not bad, bad
        for slot in used:
            assert all(np.array_equal(a, b) for a, b in zip(outs[slot], p16)), "streamed round trip is not lossless"

    # max over ranks
    times = torch.tensor([dt_dev, dt_e2e, dt_e2e16, dt_e2e32, dt_file, dt_enc, dt_dec, dt_stream], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        sizes = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([nb], dtype=torch.int64, device="cuda"))  # codestream segment sizes
    dt_dev, dt_e2e, dt_e2e16, dt_e2e32, dt_file, dt_enc, dt_dec, dt_stream = (float(times[i]) for i in range(8))

    if rank == 0:
        pix = W * H * world
        ms_step = dt_dev / args.steps * 1e3
        value = pix / (dt_dev / args.steps) / 1e6
        e2e_val = pix / (dt_e2e / args.steps) / 1e6
        enc_only_val = pix / (dt_enc / args.steps) / 1e6
        dec_only_val = pix / (dt_dec / args.steps) / 1e6
        peak, peak_src = peaks()
        l1_ms = float(np.mean([m for m, _ in lvl1]))
        l1_bytes = lvl1[0][1]
        achieved = l1_bytes / (l1_ms * 1e-3) / 1e9 if l1_ms > 0 else 0.0
        img_bytes = W * H * NCOMP * 4
        line = {
            "metric": METRIC, "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "i32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "timing": "CUDA events around the K queued steps, max over ranks; host wall clock of the same region incl. barriers: %.3f ms/step" % (wall_dev / args.steps * 1e3), "per_gpu": "one 8192x8192x3 image (64 tiles) per rank", "numa_node": numa, "cpus_per_rank": ncpus,
                       "l2": "inputs (805 MB of planes per step) are larger than the 126 MB L2",
                       "coded_bytes": int(nbytes), "blocks": int(nbk),
                       "ht_encode_Mblocks_s": nbk / (stage[1] / args.steps * 1e-3) / 1e6,
                       "ht_decode_Mblocks_s": nbk / (stage[2] / args.steps * 1e-3) / 1e6,
                       "stage_ms": {"fwd_mct_dwt": stage[0] / args.steps, "ht_encode": stage[1] / args.steps,
                                    "ht_decode": stage[2] / args.steps, "inv_dwt_mct": stage[3] / args.steps}},
            "e2e": {"value": e2e_val, "unit": "Mpixels/s", "ms_per_step": dt_e2e / args.steps * 1e3,
                    "h2d_bytes_per_step": int((img_bytes // 2 if pack_mode[0] == 1 else img_bytes) + nb + nbk * 64),
                    "d2h_bytes_per_step": int((img_bytes // 2 if pack_mode[1] == 1 else img_bytes) + nb + nbk * 24),
                    "encode_only": {"value": enc_only_val, "unit": "Mpixels/s", "ms": dt_enc / args.steps * 1e3},
                    "decode_only": {"value": dec_only_val, "unit": "Mpixels/s", "ms": dt_dec / args.steps * 1e3},
                    "host_threads": host_threads, "host_pack": {"encode": pack_mode[0], "decode": pack_mode[1]},
                    "api": "b2k_encode + b2k_decode (include/grok_b200.h), host int32 planes (the gpup_image layout); samples "
                           "<= 16 bit cross PCIe in 16-bit containers, narrowed/widened per chunk by host_threads host threads"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_dwt53_fwd<3> (DC shift + RCT + level-1 5/3, all 64 tiles x 3 comps)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": peak_src, "frac_of_nominal_8000_GBs": achieved / 8000.0,
                         "algorithmic_bytes_per_launch": int(l1_bytes),
                         "ms_per_launch": l1_ms, "traffic": TRAFFIC_NCU},
        }
        if pipe is not None:
            line["device_pipelined"] = pipe
        if extras:
            line.update({
                "e2e_i32_direct": {"value": pix / dt_e2e32 / 1e6, "unit": "Mpixels/s", "ms_per_step": dt_e2e32 * 1e3,
                                   "h2d_bytes_per_step": int(img_bytes + nb + nbk * 64), "d2h_bytes_per_step": int(img_bytes + nb + nbk * 24),
                                   "api": "same calls with b2k_set_host_threads(0): pinned int32 planes copied as they are"},
                "e2e_codestream": {"value": pix / dt_file / 1e6, "unit": "Mpixels/s", "ms_per_step": dt_file * 1e3,
                                   "codestream_bytes": int(cs_len),
                                   "api": "e2e plus the host T2 step: b2k_encode + b2k_codestream_write (TLM + PLT) into a pinned buffer, then "
                                          "b2k_codestream_parse + b2k_decode reading the block bytes in place from the file"},
                "e2e_u16": {"value": pix / (dt_e2e16 / args.steps) / 1e6, "unit": "Mpixels/s", "ms_per_step": dt_e2e16 / args.steps * 1e3,
                            "h2d_bytes_per_step": int(img_bytes // 2 + nb + nbk * 64), "d2h_bytes_per_step": int(img_bytes // 2 + nb + nbk * 24),
                            "api": "b2k_encode16 + b2k_decode16: same path, 16-bit sample containers (cf. gpup_batch_memory_submit_planes)"},
                "e2e_batch": {"value": pix / dt_stream / 1e6, "unit": "Mpixels/s", "ms_per_step": dt_stream * 1e3, "frames": n_stream,
                              "h2d_bytes_per_step": int(img_bytes // 2 + nb + nbk * 64), "d2h_bytes_per_step": int(img_bytes // 2 + nb + nbk * 24),
                              "api": "b2k_stream_encode_* feeding b2k_stream_decode_* (SURVEY 8f N2, cf. gpup_batch_memory_*): 3 frames in flight "
                                     "per direction on one GPU, 16-bit sample containers, host buffers pinned; wall clock from the first submit "
                                     "to the last decoded frame / frames"}
            })
        if world == 1 and not args.no_cpu_baseline:
            try:
                os.sched_setaffinity(0, range(os.cpu_count()))   # the CPU arm gets every core back
            except Exception:
                pass
            gs = grok_setup(img)
            if gs is not None:
                grok_tune_threads(gs)
                sec, info = min((grok_step(gs) for _ in range(3)), key=lambda r: r[0])           # best of 3 passes
                cb = {"value": W * H / sec / 1e6, "unit": "Mpixels/s", "cores": gs["threads"], "cpu_quota": cpu_quota(),
                      "kind": "reference", "host": cpu_model(),
                      "sample": "whole image (64 of 64 tiles), best of 3 passes: grk_compress() + grk_decompress() of the unmodified "
                                "libgrokj2k (oracle/_ref/grok) on memory streams, TLM + PLT",
                      "encode_only_Mpix_s": W * H / info["enc_s"] / 1e6, "decode_only_Mpix_s": W * H / info["dec_s"] / 1e6, **info}
                # one thread, on a 2048x2048 corner (4 of 64 tiles) so that it stays bounded
                g1 = grok_setup(img, 2048, 2048)
                g1["threads"] = 1
                sec1, info1 = min((grok_step(g1) for _ in range(2)), key=lambda r: r[0])
                cb["one_thread"] = {"value": 2048 * 2048 / sec1 / 1e6, "unit": "Mpixels/s", "cores": 1,
                                    "sample": "2048x2048 corner (4 of 64 tiles), best of 2", **info1}
                line["cpu_baseline"] = cb
                line["speedup_vs_cpu_baseline"] = {"e2e_encode_plus_decode": e2e_val / cb["value"],
                                                   "e2e_encode_only": enc_only_val / cb["encode_only_Mpix_s"],
                                                   "e2e_decode_only": dec_only_val / cb["decode_only_Mpix_s"],
                                                   "device_resident": value / cb["value"]}
            else:
                line["cpu_baseline"] = {"value": None, "unit": "Mpixels/s", "cores": 0, "kind": "reference",
                                        "sample": "oracle/_ref/grok not built"}
            st = cpu_reference_setup(img)
            if st is not None:   # round 1's figure, kept for continuity: kernels only, no T2 / streams / scheduler
                tune_reference_threads(st)
                sec, info = min((cpu_reference_step(st) for _ in range(2)), key=lambda r: r[0])
                line["cpu_kernel_composite"] = {"value": W * H / sec / 1e6, "unit": "Mpixels/s", "cores": st["threads"],
                                                "sample": "whole image, best of 2: the reference's HT coder + forward DWT kernels and its "
                                                          "grk_bench_dwt_53 hook driven by oracle/ref_shim (no T2, no streams)", **info}
        print(json.dumps(line))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


DUMP_SEED = 20261017
DUMP_SAMPLES = 1 << 21


def sample_outputs(planes, res):
    """What the device-resident round trip hands back after its last step, cut to about 42 MB: the decoded image
    and the coded bytes at fixed seeded positions, and the whole block table's lengths, bit planes and passes.
    The coded bytes are sampled from the blocks laid end to end in enumeration order, so that the arena's
    layout on the device does not matter.  float32 holds every decoded sample and byte exactly."""
    rng = np.random.default_rng(DUMP_SEED)
    pix = rng.integers(0, H * W, DUMP_SAMPLES)
    lens = res.blocks["length"].astype(np.int64)
    ends = np.cumsum(lens)
    pos = rng.integers(0, int(ends[-1]), 2 * DUMP_SAMPLES)
    blk = np.searchsorted(ends, pos, side="right")
    at = res.blocks["offset"].astype(np.int64)[blk] + pos - (ends[blk] - lens[blk])
    return {"decoded_sample": np.stack([p.reshape(-1)[pix] for p in planes]).astype(np.float32),
            "coded_bytes_sample": res.bytes[at].astype(np.float32),
            "block_table": np.stack([lens, res.blocks["numbps"], res.blocks["numpasses"]]).astype(np.float64)}


# dram__bytes_read.sum + dram__bytes_write.sum of one k_dwt53_fwd<3> launch, from the committed `ncu --set full` capture
# of THIS kernel version (profiles/r02v_dwt53_fwd_ncu_full_summary.txt, captured 2026-09-24 on the round-2 bulk-copy
# kernel: 877.08 MB read + 762.23 MB written = 1.018 x the algorithmic bytes).  A constant, not a per-run counter:
# re-capture when the kernel changes.
TRAFFIC_NCU = 1639311616

if __name__ == "__main__":
    main()
