"""bench.py -- Mpaths/s of the ReSTIR PT frame (1 spp, 1920x1080, Cornell Box) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one frame of the reference's frame graph for the emissive Cornell Box, steady state (temporal and
spatial reuse active): G-buffer -> ReSTIR DI (temporal + pairwise-MIS spatial) -> ReSTIR PT (path generation,
temporal + spatial path reuse) -> compositing + firefly filter -> TAA. Nothing is skipped or cached.

  value   frames timed with CUDA events on the launching stream, per-frame inputs already on the device
  e2e     the same frames through the C-ABI with HOST buffers in the timed region: the frame constants come from
          pinned host memory every frame and the anti-aliased RGBA16F image is read back to pinned host memory
  roofline        the judged bandwidth kernel -- the streaming merge of the spatial resample (k_spatial_merge): algorithmic
                  bytes / event-timed duration against the measured HBM peak; `dominant` names the kernel with the largest share
                  of the frame (traversal / issue bound, no bandwidth claim); `traffic` = DRAM bytes per launch from the committed
                  ncu capture, only if that capture was taken from the kernel sources that are being timed
  cpu_baseline    the CPU oracle (a port: the reference ships no CPU renderer) on a bounded sample of the workload
  c1_alias_table  config C1: alias-table build, device (zr_alias_table_build) next to the CPU reference-equivalent
  --impl reference   the same CPU path with every host core (SURVEY 8d: the only CPU arm the reference's math has); this arm
                  does not map libzetaray_b200.so (ZETARAY_B200_STRUCTS_ONLY)
  --dump-outputs DIR  after the timed frames, the image the last of them produced (what Renderer.GetOutput() hands the
                  caller: RGBA16F, 1080 x 1920 x 4) is written as DIR/image.npy in float32 (32 MB). The inputs depend only on the
                  arguments, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the source tree (it may be read-only)

W, H = 1920, 1080
METRIC = "Mpaths/s (1spp ReSTIR PT, 1080p)"
WORKLOAD = "Cornell Box 1080p ReSTIR PT 3-bounce + ReSTIR DI + firefly/TAA (cornell_emissive.gltf, static camera, 8-phase Halton jitter)"

# algorithmic bytes per pixel of each kernel (DESIGN.md "kernels"; SURVEY 8d for the reference's layout)
ALG_BYTES = {
    "k_gbuffer": 28.0,          # writes: core 16 + depth 4 + motion/emissive 8 (coat only when coated)
    "k_di_temporal": 16 + 8 + 16 + 32 + 32 + 8 + 16.0,   # core, motion, prev core, prev reservoir -> reservoir, target, final
    "k_di_spatial": 16 + 32 + 8 + 1.5 * (16 + 32) + 16.0,  # self + 1-2 neighbours -> final
    "k_pathtrace": 16 + 64 + 16.0 + 3 * 192,   # core -> reservoir + target, plus ~192 B of scene gathers per bounce (SURVEY 8d)
    "k_temporal_classify": 16 + 8 + 16 + 8 + 8 + 16 + 16 + 1 + 8.0,   # core, motion, prev core, coats, both headers -> flag byte, items
    "k_shift_temporal": 2 * (4 + 8 + 64 + 16 + 8) + 16 + 8.0,
    "k_temporal_merge": 4 + 64 + 16 + 1 + 8 + 64 + 32 + 64 + 16.0,
    "k_temporal": 16 + 8 + 64 + 16 + 16 + 64 + 64 + 16.0,   # fused CtT+TtC (SURVEY 8d 'temporal resample': 308 with 62 B planes)
    "k_spatial_search": 16 + 16 + 2.0,
    "k_sort": 16 + 2 + 4 + 2.0,
    "k_spatial": 16 + 64 + 16 + 2 + 2 + 16 + 64 + 64 + 16.0,  # fused CtS+StC (SURVEY 8d B_spatial = 294 with 62 B planes)
    # queued spatial path (rpt_spatial.cu). Per pixel with a usable neighbour (the common case; pixels without one move less, so
    # image-wide figures are upper bounds of the bytes and lower bounds of the time-per-byte):
    "k_spatial_classify": 4 + 2 + 16 + 16 + 8.0,               # flags, neighbour, own + neighbour header -> two queue items
    "k_shift": 2 * (4 + 2 + 64 + 16 + 8) + 16 + 8.0,           # per item: queue entry, neighbour map, record, G-buffer core + coat -> result
    # merge: flags 4, neighbour 2, thread map 2, own record 64 (TMA tile), target 16, neighbour record 64, both shift results 32
    # -> record 64 + colour 16
    "k_spatial_merge": 4 + 2 + 2 + 64 + 16 + 64 + 32 + 64 + 16.0,
    "k_svgf_temporal": 16 + 8 + 16 + 8 + 16 + 16 + 8 + 8.0,    # core, motion, signal, prev guide, history -> history, colour+variance, guide
    "k_svgf_atrous": 28.0,                                     # SURVEY 8d: colour 8 + depth 4 + normal 4 + variance 2 -> colour 8 + variance 2 (x passes)
    "k_firefly": 16 + 16 + 4 + 16 + 16.0,   # fused compositing + firefly: direct, indirect, depth, core(flags) -> composited
    "k_taa": 16 + 4 + 8 + 8 + 8.0,
}


def _clock_sampler(stop, out):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    dev = os.environ.get("LOCAL_RANK", "0")
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", "-i", dev, "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=5)
            parts = [p.strip() for p in r.stdout.strip().split(",")]
            if len(parts) >= 6:
                out.append(parts)
        except Exception:
            pass
        stop.wait(0.2)


def _clock_summary(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(float(s[0]) for s in samples)
    reasons = []
    for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
        if any(s[2 + i].lower().startswith("active") for s in samples):
            reasons.append(name)
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(samples[0][1]), "reasons": reasons}


def kernel_sources_hash():
    """Identifies the kernels an ncu capture belongs to: sha256 over the CUDA sources + the compile flags."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "zetaray_b200", "csrc")
    for f in sorted(os.listdir(d)) + ["../build.py", "../../include/zr_fpmath.h"]:
        p = os.path.join(d, f)
        if os.path.isfile(p):
            h.update(f.encode()); h.update(open(p, "rb").read())
    return h.hexdigest()[:16]


def alias_table_leg(st):
    """Config C1 (BASELINE.md 3): alias-table build at N = 2 / 13 107 / 10^6 emissive triangles, device vs CPU.
    The device build is normalise + partition in parallel and the pairing loop on ONE lane: Vose's LIFO pairing order defines the
    table (Math/Sampling.cpp:27-158), and `alias-table indices bit-exact` rules out the parallel constructions (they produce a
    different, equally valid table). It runs once per light-set change, not per frame."""
    import numpy as np
    import torch
    from zetaray_b200 import lib, check
    from tests import orc
    from tests.orc import ptr
    o = orc.load()
    ref = None
    try:
        ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_alias.so"))
    except OSError:
        pass
    out = []
    E16 = np.dtype([("a", "<f4"), ("b", "<f4"), ("c", "<f4"), ("d", "<u4")])
    for n in (2, 13107, 1000000):
        rng = np.random.default_rng(n)
        w = (rng.random(n, dtype=np.float32) * 100).astype(np.float32)
        d_w0 = torch.from_numpy(w).cuda()
        d_w = d_w0.clone()
        d_t = torch.zeros(n * 16, dtype=torch.uint8, device="cuda")
        d_s = torch.zeros(2 * n + 16, dtype=torch.int32, device="cuda")
        reps = 3 if n > 100000 else 20
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(reps + 1):
            if i == 1:
                e0.record(torch.cuda.current_stream())
            d_w.copy_(d_w0)                                # the build normalises the weights in place
            check(lib.zr_alias_table_build(C.c_void_p(d_w.data_ptr()), C.c_uint32(n), C.c_void_p(d_t.data_ptr()), C.c_void_p(d_s.data_ptr()), st))
        e1.record(torch.cuda.current_stream())
        torch.cuda.synchronize()
        gpu_ms = e0.elapsed_time(e1) / reps
        table = np.zeros(n, dtype=E16)
        t0 = time.perf_counter()
        for _ in range(reps):
            wc = w.copy()
            o.orc_alias_build_emissive(ptr(wc), C.c_int64(n), 0, ptr(table))
        cpu_ms = (time.perf_counter() - t0) / reps * 1e3
        same = d_t.cpu().numpy().view(E16).tobytes() == table.tobytes()
        out.append({"n": n, "gpu_ms": round(gpu_ms, 4), "cpu_port_ms": round(cpu_ms, 4), "identical": bool(same)})
    return {"what": "alias-table build (normalise + Vose), one call", "cpu": "oracle port, 1 thread (the reference's BuildAliasTable is scalar + AVX2 normalise)",
            "sizes": out}


def cpu_frames(w, h, nframes, nthreads, warm=3):
    """Times the CPU oracle on `nframes` steady-state frames of w x h (after `warm` untimed frames)."""
    from tests import scene_util, rpt_util
    import numpy as np
    R = rpt_util.OracleRenderer(scene_util.cornell(), w, h, nthreads=nthreads)
    seq = rpt_util.FrameSequence(w, h)
    taa_prev = np.zeros((w * h, 2), dtype=np.uint32)

    def frame(i):
        nonlocal taa_prev
        fc = seq.next()
        R.gbuffer(fc); R.rdi(fc); R.rpt(fc)
        _, taa_prev = R.post(fc, taa_prev, i > 0)
    for i in range(warm):
        frame(i)
    t0 = time.perf_counter()
    for i in range(nframes):
        frame(warm + i)
    dt = time.perf_counter() - t0
    return w * h * nframes / dt / 1e6, dt / nframes


def run_reference(args):
    """`--impl reference`: the reference has no CPU implementation of this path and cannot be built here (HLSL/DXR/D3D12);
    the arm is the oracle port of its math, all host cores, on a bounded sample (reduced resolution) of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["ZETARAY_B200_STRUCTS_ONLY"] = "1"      # ctypes mirrors of the ABI structs only: the product library is not mapped
    cores = os.cpu_count() or 1
    sw, sh = 960, 540
    # one renderer, `warmup` frames to reach steady state (temporal + spatial reuse on), then the timed frames
    mp, spf = cpu_frames(sw, sh, args.steps, cores, warm=max(3, args.warmup))
    per = [(mp, spf)] * args.steps
    sample = "%d steady-state frame(s) at %dx%d (1/4 of the 1080p pixels), %d threads" % (len(per), sw, sh, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": mp, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": len(per),
        "warmup": args.warmup, "ms_per_step": 1000.0 * sum(p[1] for p in per) / len(per), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "CPU port of the reference's shader math (the reference ships no CPU renderer)"},
        "cpu_baseline": {"value": mp, "unit": "Mpaths/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": mp, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--single-stream", action="store_true", help="record DirectLighting on the main stream instead of a second one")
    ap.add_argument("--schedule-by-cost", action="store_true", help="N > 1: launch the lighting kernels' blocks most-expensive-tile-first (measured cost map)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the image of the last timed frame to DIR/image.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the device path, not to --impl reference")
        run_reference(args)
        return
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist
    from zetaray_b200 import lib, check, _lib
    from zetaray_b200.passes import Scene, GBuffers, GBufferRT, DirectLighting, IndirectLighting, Compositing, TAA
    from zetaray_b200.camera import FrameSequence
    from zetaray_b200.scene import FlatScene

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # an explicit stream (not the legacy default one): the halo exchanges interleave torch / NCCL work with the passes'
    # kernels on the same stream handle
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    st = C.c_void_p(stream.cuda_stream)

    # Multi-GPU (SURVEY 8e): ONE 1080p frame is split into horizontal strips, one per GPU (strong scaling). Strip
    # boundaries come from the per-band SM-cycle cost measured during the unsharded warm-up frames; reservoir / final
    # halos move between neighbouring strips at four exchange points per frame; the finished strips are gathered on rank 0.
    from zetaray_b200.sharding import ShardedFrame, StripPlan
    flat = FlatScene.load(os.path.join(ROOT, "tests", "golden", "cornell_emissive.npz"))     # the reference's cornell_emissive.gltf, flattened
    scene = Scene(flat)
    scene.prelighting(st)
    gb = GBuffers(W, H)
    passes = dict(gbuffer=GBufferRT(), direct=DirectLighting(W, H), indirect=IndirectLighting(W, H),
                  compositing=Compositing(W, H), taa=TAA(W, H))
    taa = passes["taa"]
    seq = FrameSequence(W, H)
    fi = _lib.FrameInputs()
    fi.scene = scene.handle
    sharded = ShardedFrame(passes, gb, W, H, 0, 1)       # the stand-alone passes: per-kernel timing pass at N == 1

    # DirectLighting and IndirectLighting both depend only on the G-buffer (two independent render-graph nodes in the
    # reference, PathTracer.cpp:149-323), so DirectLighting is recorded on a second stream and joined before Compositing.
    side = None if args.single_stream else torch.cuda.Stream()
    st_side = st if side is None else C.c_void_p(side.cuda_stream)
    ev_g, ev_d = torch.cuda.Event(), torch.cuda.Event()

    # The native frame driver (zr_renderer, csrc/renderer.cu): one C-ABI call per frame, second stream inside. N > 1: the same
    # renderer strip-sharded (zr_renderer_set_shard) with the halo bands moved by zr_comm -- grouped NCCL send / recv issued from
    # C++ on the producing stream -- and the finished image gathered on rank 0.
    from zetaray_b200.passes import Renderer, Comm
    renderer = Renderer(scene, W, H, two_streams=not args.single_stream)
    comm = Comm.from_torch() if world > 1 else None

    def frame(fc):
        renderer.Render(fc, st)

    def output_image():
        return renderer.GetOutput()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up: unsharded frames bring temporal + spatial reuse to steady state (frame >= 3) and measure the cost
    # of every 32-row band; then the strips are cut and the same number of sharded warm-up frames follows ----
    plan_info = None
    plan = None
    if world > 1:
        tiles_x = (W + 31) // 32
        cost = torch.zeros(tiles_x * StripPlan.num_units(H), dtype=torch.int64, device="cuda")
        renderer.direct.SetCostMap(cost.data_ptr()); renderer.indirect.SetCostMap(cost.data_ptr())
    for _ in range(args.warmup):
        frame(seq.next())
    if world > 1:
        torch.cuda.synchronize()
        renderer.direct.SetCostMap(0); renderer.indirect.SetCostMap(0)
        c = cost.to(torch.float64)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)                       # identical plan on every rank
        tiles = [float(v) for v in c.tolist()]
        costs = [sum(tiles[b * tiles_x:(b + 1) * tiles_x]) for b in range(StripPlan.num_units(H))]
        plan = StripPlan.balanced(H, world, costs)
        renderer.SetShard(comm, plan.bounds, gather_output=True)
        if args.schedule_by_cost:       # a strip is only 2-3 waves of 1024-thread blocks: the expensive tiles first, the tail made of cheap ones
            renderer.direct.SetScheduleCosts(tiles, tiles_x, StripPlan.num_units(H))
            renderer.indirect.SetScheduleCosts(tiles, tiles_x, StripPlan.num_units(H))
        sc = plan.strip_costs(costs)
        plan_info = {"bounds": plan.bounds, "strip_cost_max_over_mean": round(max(sc) / (sum(sc) / world), 3)}
        for _ in range(args.warmup):
            frame(seq.next())
    # per-frame working set: G-buffers 2 x 36 B/px, PT reservoirs 2 x 64, DI 2 x 32, targets/finals ~ 90 B/px => ~0.8 GB
    # at 1080p, larger than the 126 MB L2, so no explicit flush between frames is needed.

    # ---- value: device-resident ----
    launches0 = lib.zr_kernel_launch_count()
    clocks, stop = [], threading.Event()
    th = threading.Thread(target=_clock_sampler, args=(stop, clocks), daemon=True)
    th.start()
    fcs = [seq.next() for _ in range(args.steps)]
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for fc in fcs:
        frame(fc)
    e1.record(stream)
    barrier()
    stop.set()
    ms = e0.elapsed_time(e1)
    launches = lib.zr_kernel_launch_count() - launches0
    dumped = None
    if args.dump_outputs and rank == 0:     # outside the timed region, before any later frame overwrites the image
        from zetaray_b200.passes import download_image
        dumped = {"image": download_image(output_image(), np.float16, 4).reshape(H, W, 4).astype(np.float32)}
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = W * H * args.steps / (ms_total * 1e-3) / 1e6

    # ---- e2e: host buffers in, host image out, every frame (rank 0 holds the host side) ----
    n_e2e = max(3, min(args.steps, 20))
    # host -> device per frame: the 544-byte cbFrameConstants block, which the C-ABI takes from host memory by value and every
    # kernel receives as launch parameters (there is no other per-frame input: scene and history stay resident)
    # the image read-back of frame i runs on a copy stream while frame i + 1 renders (TAA ping-pongs between two
    # images, so the one being copied is only read by the next frame); the host consumes frame i - 1 while i renders
    out_host = [torch.empty(W * H * 8, dtype=torch.uint8).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    st_copy = C.c_void_p(copy_stream.cuda_stream)
    ev_frame = [torch.cuda.Event(), torch.cuda.Event()]
    ev_copied = [torch.cuda.Event(), torch.cuda.Event()]
    fcs2 = [seq.next() for _ in range(n_e2e)]
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    for i, fc in enumerate(fcs2):
        frame(fc)
        if rank == 0:
            b = i & 1
            ev_frame[b].record(stream)
            copy_stream.wait_event(ev_frame[b])
            img = output_image()
            check(lib.zr_memcpy_d2h(C.c_void_p(out_host[b].data_ptr()), C.c_void_p(img.d_ptr), C.c_size_t(W * H * 8), st_copy))
            ev_copied[b].record(copy_stream)
            if i > 0:
                ev_copied[b ^ 1].synchronize()               # the caller consumes frame i - 1 here
    if rank == 0:
        ev_copied[(n_e2e - 1) & 1].synchronize()
        stream.wait_event(ev_copied[(n_e2e - 1) & 1])        # the last image is on the host before the clock stops
    e3.record(stream)
    barrier()
    t2 = torch.tensor([e2.elapsed_time(e3)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = W * H * n_e2e / (float(t2.item()) * 1e-3) / 1e6
    halo_bytes = 0
    if comm is not None:
        sent, calls = comm.stats()
        halo_bytes = sent // max(1, calls)

    # ---- config 3 of BASELINE.json: the same frame with the SVGF denoise stage between Compositing and TAA (N == 1) ----
    with_svgf = None
    if world == 1:
        renderer.SetDenoiser(True)
        for _ in range(max(3, args.warmup)):
            frame(seq.next())
        fcs3 = [seq.next() for _ in range(args.steps)]
        barrier()
        e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e4.record(stream)
        for fc in fcs3:
            frame(fc)
        e5.record(stream)
        barrier()
        ms3 = e4.elapsed_time(e5)
        with_svgf = {"value": round(W * H * args.steps / (ms3 * 1e-3) / 1e6, 3), "unit": "Mpaths/s", "ms_per_step": round(ms3 / args.steps, 4),
                     "what": "same frame + SVGF (temporal accumulation + 5 a-trous passes, 5x5 taps) between Compositing and TAA"}
        renderer.SetDenoiser(False)

    # ---- per-kernel timing (CUDA events on the launching stream around every launch) ----
    kern = {}
    nprof = 5
    if world == 1:                  # stand-alone passes on ONE stream, so a kernel's events do not include waiting for the other stream
        for _ in range(3):          # (they have not rendered yet: bring them to steady state first)
            sharded.render(fi, seq.next(), stream)
    check(lib.zr_profile_enable(1))
    for _ in range(nprof):          # N > 1: every rank renders (the frame holds collectives) and times its own launches
        if world == 1:
            sharded.render(fi, seq.next(), stream)
        else:
            frame(seq.next())
    if True:
        buf = C.create_string_buffer(8192)
        check(lib.zr_profile_collect(buf, 8192))
        check(lib.zr_profile_enable(0))
        for item in buf.value.decode().split(";"):
            if item:
                name, calls, total = item.split(":")
                kern[name] = float(total) / nprof      # ms per frame (all launches of that kernel)
    rank_kernel_ms = None
    if world > 1:
        mine = torch.tensor([sum(kern.values())], dtype=torch.float64, device="cuda")
        allv = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        rank_kernel_ms = [round(float(v.item()), 3) for v in allv]
    roofline, kernels = None, []
    if rank == 0 and kern:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        tot = sum(kern.values())
        y0, y1 = (0, H) if plan is None else plan.rows(rank)      # rank 0's strip
        own_rows = y1 - y0
        # pixels that carry a surface (the lighting kernels move only the 4-byte flag word of the others: sky, light sources)
        if world == 1:
            core = gb.download()[0]        # the per-kernel timing frames above rendered into `gb` (sharded.render)
        else:
            g = _lib.GBuffer()
            check(lib.zr_renderer_get_gbuffer(renderer.handle, 0, C.byref(g)))
            core = np.zeros((W * H, 4), dtype=np.uint32)
            check(lib.zr_memcpy_d2h(core.ctypes.data_as(C.c_void_p), C.c_void_p(g.d_core), C.c_size_t(core.nbytes), None))
            check(lib.zr_stream_synchronize(None))
        fl = core[:, 3].reshape(H, W)[y0:y1] & 0xff
        surf = int((((fl >> 2) & 1) == 0).sum() - ((((fl >> 2) & 1) == 0) & (((fl >> 1) & 1) == 1)).sum())
        px_all = W * own_rows
        PER_SURFACE_PIXEL = ("k_di_temporal", "k_di_spatial", "k_pathtrace", "k_temporal", "k_spatial", "k_spatial_classify", "k_shift",
                             "k_spatial_merge", "k_temporal_classify", "k_shift_temporal", "k_temporal_merge", "k_spatial_search", "k_sort")
        for name, msf in sorted(kern.items(), key=lambda kv: -kv[1]):
            ab = ALG_BYTES.get(name)
            nbytes = None if not ab else (ab * surf + 4.0 * (px_all - surf) if name in PER_SURFACE_PIXEL else ab * px_all)
            gbs = (nbytes / (msf * 1e-3) / 1e9) if ab else None
            kernels.append({"kernel": name, "ms_per_frame": round(msf, 4), "share": round(msf / tot, 4),
                            "alg_bytes_per_px": ab, "achieved_gbs": None if gbs is None else round(gbs, 1),
                            "frac": None if gbs is None else round(gbs / peak, 4)})
        by_name = {k["kernel"]: k for k in kernels}
        judged = by_name.get("k_spatial_merge") or by_name.get("k_spatial") or kernels[0]
        top = kernels[0]
        traffic, traffic_note = None, "no ncu capture committed for these kernel sources"
        try:        # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu --set full capture
            cap = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")))
            if cap.get("kernel_sources_sha16") == kernel_sources_hash():
                traffic = cap["kernels"][judged["kernel"]]["dram_bytes"]
                traffic_note = "profiles/r2_ncu_traffic.json (same kernel sources as timed)"
            else:
                traffic_note = "profiles/r2_ncu_traffic.json was captured from other kernel sources: not reported"
        except Exception:
            pass
        spatial_ms = sum(by_name[k]["ms_per_frame"] for k in ("k_spatial_search", "k_sort", "k_spatial_classify", "k_shift", "k_spatial_merge", "k_spatial") if k in by_name)
        roofline = {"kernel": judged["kernel"], "bound": "hbm", "achieved": judged["achieved_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": judged["frac"], "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
                    "alg_bytes_per_px": judged["alg_bytes_per_px"],
                    "spatial_resample_ms_total": round(spatial_ms, 4),
                    "dominant": {"kernel": top["kernel"], "share": top["share"], "ms_per_frame": top["ms_per_frame"],
                                 "bound": "traversal latency / instruction issue (no bandwidth claim, SURVEY 8d)"},
                    "surface_pixel_fraction": round(surf / px_all, 4),
                    "note": "algorithmic bytes = bytes/px x pixels that carry a surface + 4 B (the flag word) x the others (sky, light sources), "
                            "/ CUDA-event duration"}

    # ---- CPU baseline (rank 0, N == 1): bounded sample of the same workload ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        mp, spf = cpu_frames(960, 540, 5, cores)
        cpu = {"value": round(mp, 4), "unit": "Mpaths/s", "cores": cores, "kind": "port",
               "sample": "5 steady-state frames at 960x540 (1/4 of the 1080p pixels, same scene/params), %d threads, %.2f s/frame" % (cores, spf)}
    c1 = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            c1 = alias_table_leg(st)
        except Exception as e:      # the leg is informational; the frame numbers above do not depend on it
            c1 = {"error": str(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_total / args.steps, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "resolution": [W, H], "spp": 1, "bounces": 3, "restir_pt": "temporal + 1 spatial pass",
                       "restir_di": "temporal + pairwise-MIS spatial", "parallelism": "1 frame / %d horizontal strips (32-row halos, grouped NCCL send/recv from C++, image gathered on rank 0)" % world if world > 1 else "single GPU",
                       "strips": plan_info, "block_order": "most expensive tile first" if (world > 1 and args.schedule_by_cost) else "plain", "kernel_ms_per_frame_by_rank": rank_kernel_ms, "halo_bytes_per_exchange_per_rank": halo_bytes, "streams": 1 if side is None else 2, 
                       "l2": "per-frame working set ~0.8 GB >> 126 MB L2 (no flush needed)"},
            "e2e": {"value": round(e2e_value, 3), "unit": "Mpaths/s", "h2d_bytes_per_step": C.sizeof(_lib.FrameConstants),
                    "d2h_bytes_per_step": W * H * 8, "frames": n_e2e},
            "gpu_launches": int(launches),
            "clocks": _clock_summary(clocks),
            "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu, "c1_alias_table": c1, "with_svgf": with_svgf,
        }
        print(json.dumps(line))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
