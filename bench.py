#!/usr/bin/env python
"""bench.py — throughput of the visibility hot path on B200 (metric of BASELINE.json: meshlets culled/sec, with draws
culled/sec and the HBM-roofline fraction of the dominant kernel alongside).

    python bench.py --gpus 1 --steps 100 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the CPU restatement (oracle/, multi-threaded) on the host cores

A "step" is one frame of the hot path in the reference's order (niagara.cpp:1765-1788) over the C4 workload of
BASELINE.json (configs[3]: 10M synthetic meshlets / 1M draws): early drawcull+tasksubmit, early
clustercull+clustersubmit, depth pyramid (+ its footprint image), late drawcull+tasksubmit, late clustercull+clustersubmit.
`value` counts the meshlet instances the two cluster passes TEST per second (lanes with mgi < taskCount), inputs
resident in HBM, static camera (steady state).  Also on the line:
  e2e              the same frame driven from HOST buffers: per step H2D of the MeshDraw array + prior-frame depth and D2H
                   of the counters plus the visible command / cluster-index slabs (conservative: everything travels)
  e2e_incremental  what the reference's frame loop moves (niagara.cpp:1362-1411): CullData + the animated draws H2D
                   (scatter), counters D2H
  moving_camera    a second timed region of --steps frames with the camera yawing 0.2 degrees every step, so that the late pass
                   emits clusters and flips visibility bits (the compaction / atomics write path)
  task_shading     --steps frames with meshlet.task.glsl's submission mode (nvc_taskcull) instead of the cluster passes
  roofline         of whichever kernel dominates the step, with that pass's algorithmic bytes (SURVEY §8(d))
The CPU arms (cpu_baseline, --impl reference) run oracle/ only; they never load the product library.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

NAMES = ["drawcull_early", "clustercull_early", "pyramid", "drawcull_late", "clustercull_late"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-shaders"])
    ap.add_argument("--workload", default="C4", choices=["C4", "C2", "C3"], help="C4 = BASELINE configs[3] (default), C2 = configs[1], C3 = configs[2] stand-in: real cooked geometry, ~3M LOD-0 meshlets, the prior-frame depth is PRODUCED on the device (nvc_raster_depth) instead of synthesised")
    ap.add_argument("--draws", type=int, default=1_000_000)
    ap.add_argument("--meshlets-per-draw", type=int, default=10)
    ap.add_argument("--depth", type=int, default=4096)
    ap.add_argument("--cpu-sample-draws", type=int, default=1_000_000, help="draws in the bounded CPU-baseline sample (default: the whole C4 scene, one frame ~ 10-60 core-seconds)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the moving-camera and task-shading regions")
    ap.add_argument("--gather", default="mc", choices=["ce", "sm", "mc", "fused", "nccl", "none"], help="multi-GPU exchange of the late MeshTaskCommand slabs + counters: ce = copy-engine peer pushes over NVLink (no SMs), mc = one NVSwitch-multicast store kernel per rank (symmetric memory), fused = the late drawcull itself stores its commands through the multicast mapping, nccl = ncclAllGather, none = skip")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed (per pass: counters, task commands and clusters in a canonical order; visibility bits, depth pyramid) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_ARRAY_BYTES = 12 << 20  # per dumped array, shared by the ranks: a larger one is written as a fixed, seeded sample of its rows (a dump stays under 64 MB)


def pass_outputs(path):
    """What the path's buffers hold after a cull + cluster pass: counters, the live task commands and the (drawId, meshlet)
    pairs of the emitted clusters, both sorted — their order in the buffers depends on the scheduling of the device's atomics,
    their content does not."""
    import oracle_lib
    import torch

    torch.cuda.synchronize()
    dccb, ccb = path.read_counts()
    cmds = path.read_task_commands(int(dccb[1]) * 64)
    return {
        "dccb": dccb,
        "ccb": ccb,
        "commands": oracle_lib.sorted_commands(cmds[: min(int(dccb[0]), len(cmds))]),
        "clusters": oracle_lib.cluster_pairs(path.read_cluster_indices(min(int(ccb[0]), path.cib.numel())), cmds),
    }


def frame_state(path):
    """visibility state and depth pyramid at the end of a frame"""
    return {"dvb": path.dvb.cpu().numpy().astype(np.uint32), "mvb": path.mvb.cpu().numpy().view(np.uint32), "pyramid": path.depthPyramid.cpu().numpy()}


def dump_outputs(out_dir, passes, state, prefix="", array_bytes=DUMP_ARRAY_BYTES):
    """Writes what a caller of the frame receives over one step, as float64 (integers, exact) or float32 (depth): per pass (column
    0: 0 = early, 1 = late) the counters, task commands and clusters; the visibility bits and the pyramid at the end of the step."""

    def rows(columns_of):
        """one row per item of every pass: the pass, then the item's columns"""
        return np.concatenate([np.stack([np.full(len(cols[0]), i, np.float64)] + [c.astype(np.float64) for c in cols], 1) for i, cols in enumerate(map(columns_of, passes))])

    arrays = {
        "draw_command_count": np.stack([p["dccb"] for p in passes]).astype(np.float64),
        "cluster_count": np.stack([p["ccb"] for p in passes]).astype(np.float64),
        "task_commands": rows(lambda p: [p["commands"][f] for f in p["commands"].dtype.names]),
        "clusters": rows(lambda p: [p["clusters"] >> np.uint64(32), p["clusters"] & np.uint64(0xFFFFFFFF)]),
        "draw_visibility": state["dvb"].astype(np.float64),
        "meshlet_visibility": state["mvb"].astype(np.float64),
        "depth_pyramid": state["pyramid"].astype(np.float32),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        keep = array_bytes // max(1, a[:1].nbytes)
        if len(a) > keep:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.ascontiguousarray(a))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


KERNEL_OF_PASS = {
    "drawcull_early": "drawcull_kernel<0, 1>",
    "clustercull_early": "clustercull_filter_kernel<0",
    "pyramid": "pyramid_kernel",
    "drawcull_late": "drawcull_kernel<1, 1>",
    "clustercull_late": "clustercull_filter_kernel<1",
}


def profiled(pass_name, args, key_prefix):
    """A counter of the kernel behind `pass_name` from the committed ncu capture of THIS workload
    (profiles/r2_frame_ncu_summary.json, made by tools/ncu_summary.py from an `ncu --set full` run of this command);
    None when the capture is of another workload or missing."""
    if not (args.workload == "C4" and args.draws == 1_000_000 and args.meshlets_per_draw == 10 and args.depth == 4096):
        return None
    path = os.path.join(ROOT, "profiles", "r2_frame_ncu_summary.json")
    try:
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "inst": 1.0}
        for k in json.load(open(path)):
            if KERNEL_OF_PASS[pass_name] in k["Kernel Name"]:
                tot = 0.0
                for name, val in k.items():
                    if name.startswith(key_prefix):
                        v, unit = val.split()[:2]
                        tot += float(v) * scale.get(unit, 1.0)
                return tot or None
    except Exception:
        pass
    return None


def build_scene(args, rank, helpers=None):
    """Synthetic scene of the workload; cached under /tmp so that several bench invocations in one session (bench,
    ncu launch list, ncu full capture) do not regenerate 0.5 GB of inputs each.  helpers: host-side helper set
    (None = the product's niagara_b200.host; the CPU arms pass the checker's own)."""
    import pickle

    from niagara_b200 import scenes

    key = "%s_%d_%d_%d_%d" % (args.workload, args.draws, args.meshlets_per_draw, args.depth, rank)
    cache = os.path.join(tempfile.gettempdir(), "nvc_scene_%s.pkl" % key)
    scene = None
    if os.path.exists(cache):
        try:
            scene = pickle.load(open(cache, "rb"))
        except Exception:
            scene = None
    if scene is None:
        if args.workload == "C4":
            scene = scenes.config4_scene(args.draws, args.meshlets_per_draw, screen=(args.depth, args.depth), seed=21 + 100 * rank, helpers=helpers)
        elif args.workload == "C3":
            scene = scenes.config3_scene(os.path.join(ROOT, "tests", "golden"), screen=(args.depth, args.depth), seed=31 + 100 * rank)
        else:
            scene = scenes.config2_scene(args.draws, screen=(args.depth, args.depth), seed=11 + 100 * rank)
        try:
            tmp = cache + ".%d" % os.getpid()
            pickle.dump(scene, open(tmp, "wb"), protocol=4)
            os.replace(tmp, cache)
        except Exception:
            pass
    scene.helpers = helpers
    return scene


def workload_label(args, draws=None):
    draws = args.draws if draws is None else draws
    if args.workload == "C4":
        return "C4: %d draws x %d unique meshlets each (%d meshlet instances), all inside the frustum, %dx%d depth" % (draws, args.meshlets_per_draw, draws * args.meshlets_per_draw, args.depth, args.depth)
    if args.workload == "C3":
        return "C3 stand-in: kitten.obj cooked by the reference (309 LOD-0 meshlets, LOD chain) x 10000 draws = 3.1M LOD-0 meshlet instances, LOD selection on, two-pass Hi-Z occlusion + cone cull on depth PRODUCED on the device (nvc_raster_depth), %dx%d" % (args.depth, args.depth)
    return "C2: %d draws (reference PCG32 scene), 1024 meshes x 4 LODs, %dx%d depth" % (draws, args.depth, args.depth)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=open(self.path, "w"),
                stderr=subprocess.DEVNULL,
            )
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm))
        return out


def cpu_threads():
    """Threads of the CPU arms: one per CPU this process may run on (cgroup / affinity aware), workers pinned (ORC_PIN)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(args, scene, threads, repeats=5, shaders=False, budget_s=20.0):
    """The CPU restatement (oracle/, `kind: port` — the reference has no CPU cull path, SURVEY F2) on a bounded sample:
    the first `cpu_sample_draws` draws of the same scene, steady-state frames, all host threads (pinned, one per CPU).
    Reports the BEST and the MEDIAN frame: on a shared 128-thread host the spread between them is the scheduling noise.
    shaders=True times the reference's own GLSL compiled for the host instead (oracle/_ref/librefshader.so, `kind:
    reference`): same results bit for bit, ~4x slower than the port (64-lane workgroups with idle lanes, robust-buffer
    checks), which is why the FASTER port stays the reported baseline and this one is only attached for information.
    Nothing here touches the product library: host-side helpers come from the oracle (oracle_lib.CheckerHost)."""
    import oracle_lib

    H = oracle_lib.CheckerHost
    n = min(args.cpu_sample_draws, len(scene.draws))
    draws = scene.draws[:n].copy()
    bits, _ = H.visibility_offsets(draws, scene.meshes)
    cd = H.cull_data(scene.camera, scene.screen[0], scene.screen[1], n)
    cls = oracle_lib.OraclePath
    if shaders:
        import refshader_lib

        cls = refshader_lib.RefShaderPath
    o = cls(scene.meshes, scene.meshlets, draws, *scene.screen, threads=threads, cmd_capacity=max(64, (n * 2 + 63) // 64 * 64), helpers=H)
    o.set_visibility_bits(bits)
    o.frame(cd, scene.depth, cluster_backface=True)  # warm-up frame: establishes dvb / mvb

    def one_frame():
        t0 = time.perf_counter()
        # identical pass order; count the meshlets the two cluster passes test
        o.cull(cd, late=False)
        ncmd_e = int(o.dccb[1]) * 64
        o.render_clusters(cd, late=False, cluster_backface=True)
        o.pyramid(scene.depth)
        o.cull(cd, late=True)
        ncmd_l = int(o.dccb[1]) * 64
        o.render_clusters(cd, late=True, cluster_backface=True)
        dt = time.perf_counter() - t0
        # static scene: the late command list is also what the early pass of the next frame sees
        tested = 2 * int(o.read_task_commands(ncmd_l)["taskCount"].sum()) if ncmd_e == ncmd_l else None
        return dt, tested

    times, tested, t_begin = [], 0, time.perf_counter()
    while len(times) < repeats or (len(times) < 7 and time.perf_counter() - t_begin < budget_s):
        dt, n_tested = one_frame()
        if n_tested is not None:
            tested = n_tested
        times.append(dt)
    best, med = min(times), float(np.median(times))
    if shaders:
        return {"value": tested / best, "unit": "meshlets/s", "cores": threads, "kind": "reference", "seconds": best, "what": "the reference's own GLSL shaders compiled for the host (oracle/_ref/librefshader.so), best of %d frames" % len(times)}
    return {
        "value": tested / best,
        "value_median": tested / med,
        "unit": "meshlets/s",
        "cores": threads,
        "pinned": os.environ.get("ORC_PIN", "0") != "0",
        "kind": "port",
        "sample": "best of %d steady-state frames over the first %d draws (%d meshlet tests per frame, %dx%d depth pyramid) of the same scene, %.3f s per frame (median %.3f s)" % (len(times), n, tested, scene.screen[0], scene.screen[1], best, med),
        "draws_per_s": 2 * n / best,
        "seconds": best,
        "seconds_median": med,
    }


def run_reference(args):
    """--impl reference: the CPU restatement timed on the host cores (rank 0 only).  Never imports the product's .so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib

    threads = cpu_threads()
    # bounded sample per step so that steps + warmup end within a few minutes
    args.cpu_sample_draws = min(args.cpu_sample_draws, args.draws)
    sample_args = argparse.Namespace(**vars(args))
    sample_args.draws = args.cpu_sample_draws
    scene = build_scene(sample_args, 0, helpers=oracle_lib.CheckerHost)
    res = None
    t_steps = []
    for i in range(args.warmup + args.steps):
        r = cpu_baseline(sample_args, scene, threads, repeats=1, budget_s=0.0)
        if i >= args.warmup:
            t_steps.append(r)
        res = r
    value = float(np.mean([r["value"] for r in t_steps]))
    # informational: the reference's own shaders compiled for the host, timed in a child process so that nothing it does can
    # take this arm down (it is ~4x slower than the port, which therefore stays the reported baseline)
    shaders = None
    try:
        child = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-shaders", "--cpu-sample-draws", str(sample_args.draws), "--draws", str(sample_args.draws),
                                "--meshlets-per-draw", str(args.meshlets_per_draw), "--depth", str(args.depth)], capture_output=True, text=True, timeout=240)
        shaders = json.loads(child.stdout.strip().splitlines()[-1]) if child.returncode == 0 and child.stdout.strip() else {"unavailable": "exit %d" % child.returncode}
    except Exception as e:
        shaders = {"unavailable": str(e)[:120]}
    line = {
        "impl": "reference",
        "metric": "meshlets culled/sec",
        "value": value,
        "unit": "meshlets/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean([r["seconds"] for r in t_steps])),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_label(args, sample_args.draws), "sample": "every step = one steady-state frame of the first %d draws of that scene" % sample_args.draws, "what": "CPU restatement of the GLSL (oracle/; the reference has no CPU cull path), %d pinned threads" % threads},
        "cpu_baseline": {"value": value, "value_median": float(np.median([r["value_median"] for r in t_steps])), "unit": "meshlets/s", "cores": threads, "pinned": res["pinned"], "kind": "port", "sample": res["sample"], **({"reference_shaders": shaders} if shaders else {})},
        "e2e": {"value": value, "unit": "meshlets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "draws_per_s": float(np.mean([r["draws_per_s"] for r in t_steps])),
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    os.environ.setdefault("ORC_PIN", "1")  # the oracle's worker threads stay on one CPU each (CPU arms only)
    if args.impl == "reference":
        run_reference(args)
        return
    if args.impl == "reference-shaders":  # child of the reference arm, see run_reference
        import oracle_lib
        import refshader_lib

        if not refshader_lib.available():
            print(json.dumps({"unavailable": "oracle/_ref/librefshader.so not built"}))
            return
        print(json.dumps(cpu_baseline(args, build_scene(args, 0, helpers=oracle_lib.CheckerHost), cpu_threads(), repeats=2, shaders=True)))
        return

    import torch
    import torch.distributed as dist

    from niagara_b200 import host, layout
    from niagara_b200.lib import check
    from niagara_b200.path import VisibilityPath

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU baseline")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    peak_gbs, peak_src = load_peaks()
    scene = build_scene(args, rank)
    D = len(scene.draws)
    cd = scene.cull_data()
    path = VisibilityPath(scene.meshes, scene.meshlets, scene.draws, *scene.screen, device=dev)
    path.set_visibility_bits(scene.visibility_bits)
    depth_host = torch.from_numpy(scene.depth).pin_memory()
    draws_host = torch.from_numpy(scene.draws.view(np.uint8).reshape(-1)).pin_memory()
    depth = depth_host.to(dev)
    lib = path.lib
    launches = {"n": 0}  # kernels of OUR library launched (counted at the call sites below)
    produced = None
    if args.workload == "C3":
        produced = {
            "proj": host.projection(scene.camera, *scene.screen),
            "vertices": torch.from_numpy(scene.vertices).to(dev),
            "meshletdata": torch.from_numpy(scene.meshletdata.view(np.int32)).to(dev),
        }
        depth.zero_()
    has_fp = os.environ.get("NVC_PREPARE_HIZ", "1") != "0"

    # ---- multi-GPU: all-gather of the per-rank visible command slabs + counters (SURVEY §8(e)) ----
    gather = args.gather if world > 1 else "none"
    transport = gather  # what is reported; ce / sm / mc / fused all speak the nvc_gather_* protocol below
    slab_cmds = (D * max(1, (args.meshlets_per_draw + 63) // 64) + 63) // 64 * 64 if args.workload == "C4" else 0
    if not slab_cmds:
        gather = transport = "none"
    slab_bytes = slab_cmds * layout.MESHTASKCOMMAND_DTYPE.itemsize
    gathered = gathered_counts = None
    gather_note = None
    symm_keep = None
    if gather in ("mc", "fused"):
        # symmetric memory with an NVSwitch multicast mapping (torch owns the allocation and the handle exchange)
        err = None
        try:
            import torch.distributed._symmetric_memory as symm_mem

            region = int(lib.nvc_gather_region_bytes(slab_bytes, world))
            t = symm_mem.empty(region, dtype=torch.uint8, device=dev)
            hdl = symm_mem.rendezvous(t, dist.group.WORLD)
            mc_ptr = int(hdl.multicast_ptr) if hasattr(hdl, "multicast_ptr") else 0
            if not mc_ptr:
                raise RuntimeError("no multicast mapping on this system")
            peers = (ctypes.c_void_p * world)(*[int(p) for p in hdl.buffer_ptrs])
            check(lib.nvc_gather_attach(path.ctx, slab_bytes, rank, world, peers, ctypes.c_void_p(mc_ptr)), path.ctx, "nvc_gather_attach")
            check(lib.nvc_gather_set_mode(path.ctx, 3 if gather == "fused" else 2), path.ctx, "nvc_gather_set_mode")
            symm_keep = (t, hdl)
        except Exception as e:
            err = e
        ok = torch.tensor([0 if err else 1], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)  # every rank takes the same decision
        if not int(ok.item()):
            # no symmetric memory / multicast here: the copy-engine transport takes over on every rank
            gather_note = "%s unavailable (%s): fell back to the copy-engine transport" % (gather, str(err)[:120] if err else "another rank failed")
            gather = transport = "ce"
        dist.barrier()
    sm_push = gather == "sm"
    if gather in ("ce", "sm"):
        ticket = (ctypes.c_ubyte * 192)()
        check(lib.nvc_gather_create(path.ctx, slab_bytes, rank, world, ticket), path.ctx, "nvc_gather_create")
        mine = torch.tensor(list(ticket), dtype=torch.uint8, device=dev)
        everyone = torch.zeros(world * 192, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(everyone, mine)
        tickets = (ctypes.c_ubyte * (192 * world))(*everyone.cpu().tolist())
        check(lib.nvc_gather_connect(path.ctx, tickets), path.ctx, "nvc_gather_connect")
        check(lib.nvc_gather_set_mode(path.ctx, int(sm_push)), path.ctx, "nvc_gather_set_mode")
        dist.barrier()
    elif gather == "nccl":
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = (ctypes.c_ubyte * 128)()
            check(lib.nvc_nccl_unique_id(buf), path.ctx, "nvc_nccl_unique_id")
            uid = torch.tensor(list(buf), dtype=torch.uint8)
        uid = uid.to(dev)
        dist.broadcast(uid, 0)
        uid_host = (ctypes.c_ubyte * 128)(*uid.cpu().tolist())
        check(lib.nvc_nccl_init(path.ctx, uid_host, rank, world), path.ctx, "nvc_nccl_init")
        gathered = torch.zeros(world * slab_bytes, dtype=torch.uint8, device=dev)
        gathered_counts = torch.zeros(world * 4, dtype=torch.int32, device=dev)
        comm_stream = torch.cuda.Stream(dev, priority=-1)  # high priority: its CTAs are placed before the persistent cluster pass's
    peer = gather in ("ce", "sm", "mc", "fused")  # the nvc_gather_* protocol

    # With the copy-engine gather the late commands go to their own buffer (the C ABI takes the command buffer per
    # call): the slab pushed after drawcull(late) of frame k then stays untouched until drawcull(late) of frame k+1, so
    # the exchange has the late cluster pass AND the next frame's early passes to complete — frames in flight like the
    # reference's MAX_FRAMES = 2 (config.h:31).  The wait sits right before the slab is overwritten (and after the loop).
    dcb_early = path.dcb
    dcb_late = torch.zeros_like(path.dcb) if peer else path.dcb
    pending = {"push": False}
    xchg = {"on": True}  # the cull-only region (multi-GPU, reported beside the headline) switches the exchange off

    def frame(cull, events=None, task=None):
        """one frame; task = (payloads, emit_counts) runs meshlet.task.glsl's submission mode instead of the cluster passes"""

        def mark(i):
            if events is not None:
                events[i].record()

        def clusters(late):
            if task is None:
                path.render_clusters(cull, late=late, cluster_backface=True)
            else:
                path.task_shading(cull, late, task[0], task[1], cluster_backface=True)

        mark(0)
        path.dcb = dcb_early
        path.cull(cull, late=False)
        mark(1)
        clusters(False)
        mark(2)
        if produced is not None:
            # C3: the early pass's clusters are rasterised into a cleared depth target on the device; its pyramid is what
            # the late pass culls against (niagara.cpp:1576-1733) — no synthetic depth
            depth.zero_()
            path.raster_depth(cull, produced["proj"], produced["vertices"], produced["meshletdata"], depth)
            launches["n"] += 2
        mark(3)
        path.pyramid(depth)
        mark(4)
        path.dcb = dcb_late
        if peer and xchg["on"] and pending["push"]:
            # the previous frame's slab (and every peer's copy of it) must have landed before it is overwritten
            check(lib.nvc_gather_wait(path.ctx, path._stream()), path.ctx, "nvc_gather_wait")
            pending["push"] = False
            launches["n"] += 2
        if gather == "fused" and xchg["on"]:
            # fused compute + collective: the late drawcull stores its commands through the NVSwitch multicast mapping as it
            # writes them (this call takes the frame tag and waits for the peers' acknowledgements of that parity's buffers)
            check(lib.nvc_gather_fuse_next_drawcull(path.ctx, path._stream()), path.ctx, "nvc_gather_fuse_next_drawcull")
            launches["n"] += 1
        path.cull(cull, late=True)
        mark(5)
        launches["n"] += 5 + (1 if has_fp else 0)
        if peer and xchg["on"]:
            # the late command slab is final once drawcull(late) is done: ce = push it to every peer with the copy engines,
            # mc = one multicast store kernel, fused = only counters + flags are left; all of it overlaps the late cluster
            # pass (and the next frame's early passes)
            check(lib.nvc_gather_push(path.ctx, path._stream(), ctypes.c_void_p(path.dcb.data_ptr()), ctypes.c_void_p(path.dccb.data_ptr())), path.ctx, "nvc_gather_push")
            pending["push"] = True
            launches["n"] += 1 if gather == "ce" else 2
        elif gather == "nccl" and xchg["on"]:
            done = torch.cuda.Event()
            done.record()
            comm_stream.wait_event(done)
            check(
                lib.nvc_allgather_visible(path.ctx, ctypes.c_void_p(comm_stream.cuda_stream), ctypes.c_void_p(path.dcb.data_ptr()), slab_bytes, ctypes.c_void_p(path.dccb.data_ptr()), ctypes.c_void_p(gathered.data_ptr()), ctypes.c_void_p(gathered_counts.data_ptr())),
                path.ctx,
                "nvc_allgather_visible",
            )
        clusters(True)
        mark(6)
        if produced is not None:
            path.raster_depth(cull, produced["proj"], produced["vertices"], produced["meshletdata"], depth)
            launches["n"] += 1
        mark(7)
        if gather == "nccl" and xchg["on"]:
            torch.cuda.current_stream().wait_stream(comm_stream)

    NEV = 8  # timing marks per frame: start, cull e, clusters e, raster e, pyramid, cull l, clusters l, raster l

    def new_events(n):
        return [[torch.cuda.Event(enable_timing=True) for _ in range(NEV)] for _ in range(n)]

    def passes_of(evs):
        """[steps, 5] ms of the five cull-path passes (NAMES order) and [steps, 2] ms of the two raster passes (C3 only)"""
        idx = [(0, 1), (1, 2), (3, 4), (4, 5), (5, 6)]
        a = np.array([[e[i].elapsed_time(e[j]) for i, j in idx] for e in evs])
        r = np.array([[e[2].elapsed_time(e[3]), e[6].elapsed_time(e[7])] for e in evs])
        return a, r

    def drain():
        """end of a timed region: the last frame's exchange must be complete on every rank"""
        if peer and pending["push"]:
            check(lib.nvc_gather_wait(path.ctx, path._stream()), path.ctx, "nvc_gather_wait")
            pending["push"] = False

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, K, events=None):
        """K calls of fn(k) between barriers; device time of the region, MAX over ranks"""
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        start.record()
        for k in range(K):
            fn(k)
        drain()
        stop.record()
        sync_all()
        t = torch.tensor([start.elapsed_time(stop)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up: establishes the steady two-phase state (dvb / mvb) and warms caches / clocks ----
    for _ in range(max(3, args.warmup)):
        frame(cd)
    drain()
    torch.cuda.synchronize()

    def probe(cull, keep=None):
        """one frame with the per-pass work counts read back (untimed); keep: a list that receives pass_outputs() of both passes"""
        reached = int((path.dvb != 0).sum().item())
        mvb_set_before = None
        path.dcb = dcb_early
        path.cull(cull, late=False)
        torch.cuda.synchronize()
        dccb_e = path.dccb.cpu().numpy().astype(np.uint32)
        cmds_e = path.read_task_commands(int(dccb_e[1]) * 64)
        path.render_clusters(cull, late=False, cluster_backface=True)
        torch.cuda.synchronize()
        ccb_e = path.ccb.cpu().numpy().astype(np.uint32)
        if keep is not None:
            keep.append(pass_outputs(path))  # (the late pass overwrites cib)
        if produced is not None:
            depth.zero_()
            path.raster_depth(cull, produced["proj"], produced["vertices"], produced["meshletdata"], depth)
        path.pyramid(depth)
        path.dcb = dcb_late
        path.cull(cull, late=True)
        torch.cuda.synchronize()
        dccb_l = path.dccb.cpu().numpy().astype(np.uint32)
        cmds_l = path.read_task_commands(int(dccb_l[1]) * 64)
        path.render_clusters(cull, late=True, cluster_backface=True)
        torch.cuda.synchronize()
        ccb_l = path.ccb.cpu().numpy().astype(np.uint32)
        if keep is not None:
            keep.append(pass_outputs(path))
        if produced is not None:
            path.raster_depth(cull, produced["proj"], produced["vertices"], produced["meshletdata"], depth)
        return {
            "early_reached": reached,
            "tested_early": int(cmds_e["taskCount"].sum()),
            "tested_late": int(cmds_l["taskCount"].sum()),
            "cmds_early": int(dccb_e[0]),
            "cmds_late": int(dccb_l[0]),
            "draws_early": int(np.unique(cmds_e["drawId"][cmds_e["taskCount"] > 0]).size),
            "draws_late": int(np.unique(cmds_l["drawId"][cmds_l["taskCount"] > 0]).size),
            "emitted_early": int(ccb_e[0]),
            "emitted_late": int(ccb_l[0]),
        }

    pr = probe(cd)
    tested_per_step = pr["tested_early"] + pr["tested_late"]
    draws_per_step = pr["early_reached"] + D

    # ---- timed region: device-resident inputs, static camera ----
    filter_stats = (ctypes.c_uint64 * 2)()
    lib.nvc_filter_stats(path.ctx, filter_stats, 1)  # reset the filter's diagnostic counters
    K = args.steps
    ev = new_events(K)
    sampler = ClockSampler(local_rank)
    sync_all()
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    launches["n"] = 0
    eager_ms = timed(lambda k: frame(cd, ev[k]), K)
    gpu_launches = launches["n"]
    # the same K frames without the seven timing events per frame (each one is a stream operation between two dependent
    # launches): this is the region a multi-GPU run is judged on (no CUDA-graph replay there, see below)
    plain_ms = timed(lambda k: frame(cd), K)
    lib.nvc_filter_stats(path.ctx, filter_stats, 1)
    pass_ms, raster_ms = passes_of(ev)

    # ---- the same frames as CUDA-graph launches (SURVEY §8(d): graph replay; no per-launch host work, no timing events between
    # the passes).  Calls of the C ABI only enqueue, so a frame captures as is.
    # Multi-GPU: frames WITHOUT an exchange (--gather none) are replayed the same way.  Frames with the peer exchange are replayable
    # too (nvc_gather_graph_advance: GF = 4 frames per graph, verified at N = 2, profiles/r2_bench_n2_*.json) but that path is opt-in
    # (NVC_BENCH_GRAPH_EXCHANGE=1): it has not been run on 8 GPUs, and a capture that fails on one rank only must not be able to
    # take a scaling run down, so the default at N > 1 is the eager region above. ----
    graph_ms = None
    graph_note = None
    with_exchange = world > 1 and gather != "none"
    GF = 4 if (peer and with_exchange) else 1
    want_graph = os.environ.get("NVC_BENCH_GRAPH", "1") != "0" and K >= GF and (not with_exchange or (peer and os.environ.get("NVC_BENCH_GRAPH_EXCHANGE", "0") == "1"))
    if want_graph:
        graph = None
        try:
            drain()
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(GF):
                    frame(cd)  # warm the side stream
                drain()
            sync_all()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local" if world > 1 else "global"):  # (other threads of a multi-GPU process — the NCCL watchdog — must not invalidate the capture)
                for _ in range(GF):
                    frame(cd)
                drain()
                if with_exchange:
                    check(lib.nvc_gather_graph_advance(path.ctx, path._stream(), GF), path.ctx, "nvc_gather_graph_advance")
        except Exception as e:
            graph_note = str(e)[:200]
            graph = None
            torch.cuda.synchronize()
        # every rank takes the same decision BEFORE anything rank-divergent happens (the regions below contain collectives)
        ok_t = torch.tensor([1 if graph is not None else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
        if int(ok_t.item()):
            reps = K // GF
            for _ in range(3):
                graph.replay()
            per = []
            for rep in range(3):  # three regions of K frames: median and min reported
                per.append(timed(lambda k: graph.replay(), reps) * (K / float(reps * GF)))
            graph_ms = {"median": float(np.median(per)), "min": float(min(per))}
        elif with_exchange:
            # a failed capture has advanced this rank's frame tags without running the frames: the exchange cannot go on
            raise SystemExit("bench.py: CUDA-graph capture of the exchange failed (%s); run without NVC_BENCH_GRAPH_EXCHANGE" % graph_note)
        del graph

    # ---- multi-GPU: the same frames WITHOUT the exchange (SURVEY §8(e): cull-only and cull + gather scaling are both reported) ----
    cull_only_ms = None
    if with_exchange:
        drain()
        xchg["on"] = False
        for _ in range(2):
            frame(cd)
        cull_only_ms = timed(lambda k: frame(cd), K)
        xchg["on"] = True

    # headline = graph replay when it ran (that is how a host would drive the frame), eager otherwise
    max_ms = graph_ms["median"] if graph_ms else min(eager_ms, plain_ms)
    if args.dump_outputs:
        # The early pass's commands and clusters of the last timed step are gone (the late pass reuses the buffers): the same frame
        # runs once more, untimed, from the state the timed steps left, with both passes read back (without the multi-GPU exchange).
        # The static camera is in a steady state, so it must reproduce the last timed step exactly — which also shows that leaving the
        # exchange out did not change a rank's own outputs; every rank checks, and all of them agree before anything is written.
        # Each rank writes its own outputs, with a share of the size limit.
        last = dict(pass_outputs(path), **frame_state(path))
        passes = []
        probe(cd, passes)
        again = dict(passes[1], **frame_state(path))
        same = torch.tensor([int(all(np.array_equal(last[k], again[k]) for k in last))], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
        if not int(same.item()):
            raise SystemExit("bench.py --dump-outputs: the replayed frame differs from the last timed step (no steady state)")
        dump_outputs(args.dump_outputs, passes, again, "rank%d_" % rank if world > 1 else "", DUMP_ARRAY_BYTES // world)

    counts = torch.tensor([tested_per_step, draws_per_step], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    tested_all, draws_all = float(counts[0].item()), float(counts[1].item())

    # ---- multi-GPU: one untimed verification frame — every rank's gathered copy of every slab == its owner's slab ----
    multi_gpu_verified = None
    multi_gpu_note = None
    if world > 1 and gather != "none":
      try:
          frame(cd)
          drain()
          torch.cuda.synchronize()
          if peer:
              slabs_p, counts_p = ctypes.c_void_p(), ctypes.c_void_p()
              check(lib.nvc_gather_buffers(path.ctx, ctypes.byref(slabs_p), ctypes.byref(counts_p)), path.ctx, "nvc_gather_buffers")

              class _Raw:  # a device allocation of the library seen as a torch tensor (no copy)
                  def __init__(self, ptr, nbytes):
                      self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}

              g_slabs = torch.as_tensor(_Raw(slabs_p.value, world * slab_bytes), device=dev)
              g_counts = torch.as_tensor(_Raw(counts_p.value, world * 16), device=dev).view(torch.int32)
          else:
              g_slabs, g_counts = gathered, gathered_counts
          local_counts = path.dccb.to(torch.int32)
          all_counts = torch.empty(world * 4, dtype=torch.int32, device=dev)
          dist.all_gather_into_tensor(all_counts, local_counts.contiguous())
          ok = bool((all_counts == g_counts).all().item())
          # content: a position-weighted 64-bit checksum of each slab's valid bytes, computed by its owner and by every holder
          def checksum(buf, nbytes):
              words = buf[: (nbytes // 4) * 4].view(torch.int32).to(torch.int64)
              idx = torch.arange(1, words.numel() + 1, device=dev, dtype=torch.int64)
              return int(((words * idx) % 2147483629).sum().item() % 2147483629)

          mine_sum = torch.tensor([checksum(path.dcb, min(int(local_counts[0].item()), slab_cmds) * 20)], dtype=torch.int64, device=dev)
          all_sums = torch.empty(world, dtype=torch.int64, device=dev)
          dist.all_gather_into_tensor(all_sums, mine_sum)
          for r in range(world):
              n = min(int(all_counts[4 * r].item()), slab_cmds) * 20
              ok = ok and checksum(g_slabs[r * slab_bytes : (r + 1) * slab_bytes], n) == int(all_sums[r].item())
          flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
          dist.all_reduce(flag, op=dist.ReduceOp.MIN)
          multi_gpu_verified = bool(flag.item())
      except Exception as e:  # the verification must never take the measurement down (ranks may then disagree: report, do not hang)
        multi_gpu_note = str(e)[:160]

    exchange_timed_out = None
    if world > 1 and peer:
        flag = ctypes.c_int(0)
        if lib.nvc_gather_status(path.ctx, ctypes.byref(flag)) == 0:
            t = torch.tensor([flag.value], dtype=torch.int32, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            exchange_timed_out = bool(t.item())

    def run_moving_camera():
        """yaw 0.2 degrees per step: the late pass now emits clusters and flips visibility bits"""
        cams = [host.make_camera(orientation=host.quat_from_axis_angle((0.0, 1.0, 0.0), np.radians(0.2 * (k + 1)))) for k in range(K)]
        cds = [host.cull_data(c, scene.screen[0], scene.screen[1], D) for c in cams]
        dvb0, mvb0 = path.dvb.clone(), path.mvb.clone()
        evm = new_events(K)
        mv_ms = timed(lambda k: frame(cds[k], evm[k]), K)
        mv_pass, _ = passes_of(evm)
        # replay the same camera path from the same state, untimed, reading the work counts of every step
        path.dvb.copy_(dvb0)
        path.mvb.copy_(mvb0)
        steps = [probe(c) for c in cds]
        tested_mv = float(sum(s["tested_early"] + s["tested_late"] for s in steps))
        t2 = torch.tensor([tested_mv], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.SUM)
        lm = {k: float(np.mean([s[k] for s in steps])) for k in steps[0]}
        late_ms = float(mv_pass[:, 4].mean())
        late_bytes = lm["tested_late"] * 24 + lm["cmds_late"] * 20 + lm["draws_late"] * 48 + 2 * lm["tested_late"] / 8.0 + 4 * lm["emitted_late"]
        return {
            "what": "camera yaws 0.2 degrees per step (%d steps): draws enter / leave the frustum, occlusion changes, the late cluster pass emits clusters and rewrites visibility bits" % K,
            "value": float(t2.item()) / (mv_ms * 1e-3),
            "unit": "meshlets/s",
            "ms_per_step": mv_ms / K,
            "passes_ms": {n: float(mv_pass[:, i].mean()) for i, n in enumerate(NAMES)},
            "per_step_mean": lm,
            "late_cluster_roofline": {"algorithmic_bytes_per_launch": late_bytes, "kernel_ms": late_ms, "achieved": late_bytes / (late_ms * 1e-3) / 1e9, "peak": peak_gbs, "frac": late_bytes / (late_ms * 1e-3) / 1e9 / peak_gbs, "unit": "GB/s"},
        }

    def run_task_shading():
        """task-shading submission mode (meshlet.task.glsl): nvc_taskcull instead of the cluster passes"""
        ncmd_cap = (max(pr["cmds_early"], pr["cmds_late"]) + 63) // 64 * 64 + 64
        payloads = torch.zeros(ncmd_cap * 256, dtype=torch.uint8, device=dev)
        emit_counts = torch.zeros(ncmd_cap, dtype=torch.int32, device=dev)
        for _ in range(2):
            frame(cd, task=(payloads, emit_counts))
        evt = new_events(K)
        t_ms = timed(lambda k: frame(cd, evt[k], task=(payloads, emit_counts)), K)
        t_pass, _ = passes_of(evt)
        tk_ms = float(t_pass[:, 4].mean())
        tk_bytes = pr["tested_late"] * 24 + pr["cmds_late"] * 20 + pr["draws_late"] * 48 + 2 * pr["tested_late"] / 8.0 + 4 * pr["emitted_late"] + 4 * pr["cmds_late"]
        return {
            "what": "the frame with meshlet.task.glsl's submission mode: nvc_taskcull writes one 256-byte payload + emit count per task command instead of cib/ccb (%d steps)" % K,
            "value": tested_all * K / (t_ms * 1e-3),
            "unit": "meshlets/s",
            "ms_per_step": t_ms / K,
            "passes_ms": {n.replace("clustercull", "taskcull"): float(t_pass[:, i].mean()) for i, n in enumerate(NAMES)},
            "late_taskcull_roofline": {"algorithmic_bytes_per_launch": tk_bytes, "kernel_ms": tk_ms, "achieved": tk_bytes / (tk_ms * 1e-3) / 1e9, "peak": peak_gbs, "frac": tk_bytes / (tk_ms * 1e-3) / 1e9 / peak_gbs, "unit": "GB/s"},
        }

    extras = {}
    if not args.no_extras and args.workload == "C4" and world == 1:  # single-GPU diagnostics (write path, task-shading mode)
        for key, fn in (("moving_camera", run_moving_camera), ("task_shading", run_task_shading)):
            try:
                extras[key] = fn()
            except Exception as e:  # never let an extra take the headline down
                extras[key] = {"unavailable": str(e)[:160]}
            # back to the static camera's steady state
            path.dcb = dcb_early
            for _ in range(3):
                frame(cd)
            drain()
            torch.cuda.synchronize()

    # ---- end-to-end: host buffers in, results out, copies inside the timed region ----
    e2e = e2e_inc = None
    if not args.no_e2e:
        count_host = torch.zeros(8, dtype=torch.int32).pin_memory()
        cmd_host = torch.zeros(path.dcb.numel() if path.dcb.numel() < (1 << 26) else (1 << 26), dtype=torch.uint8).pin_memory()
        cib_host = torch.zeros(min(path.cib.numel(), 1 << 24), dtype=torch.int32).pin_memory()
        # two input buffer sets (like the reference's MAX_FRAMES = 2 frames in flight, config.h:31): the H2D copy of
        # frame k+1 runs on a copy stream while frame k computes and its results are read back
        st = {"h2d": 0, "d2h": 0}
        db_orig = path.db
        db_sets = [path.db, torch.empty_like(path.db)]
        depth_sets = [depth, torch.empty_like(depth)]
        copy_stream = torch.cuda.Stream(dev)
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        main_stream = torch.cuda.current_stream()

        def upload(k):
            with torch.cuda.stream(copy_stream):
                db_sets[k % 2].copy_(draws_host, non_blocking=True)  # MeshDraw[] (the reference's db is host-visible and rewritten when animating)
                depth_sets[k % 2].copy_(depth_host, non_blocking=True)  # prior-frame depth target stand-in
                ready[k % 2].record(copy_stream)
            st["h2d"] = draws_host.numel() + depth_host.numel() * 4 + 144

        def e2e_frame(k):
            nonlocal depth
            main_stream.wait_event(ready[k % 2])
            path.db = db_sets[k % 2]
            depth = depth_sets[k % 2]
            frame(cd)
            upload(k + 1)  # the other buffer set is free: frame k-1 was fully consumed before this call
            count_host[:4].copy_(path.dccb, non_blocking=True)
            count_host[4:].copy_(path.ccb, non_blocking=True)
            main_stream.synchronize()
            ncmd = min(int(count_host[0].item()), path.task_wglimit)
            ncl = min(int(count_host[4].item()), path.cluster_limit)
            nb = ncmd * 20
            cmd_host[:nb].copy_(path.dcb[:nb], non_blocking=True)
            cib_host[:ncl].copy_(path.cib[:ncl], non_blocking=True)
            main_stream.synchronize()
            st["d2h"] = 32 + nb + ncl * 4

        upload(0)
        for k in range(2):
            e2e_frame(k)
        # upload(2) is already in flight from the warm-up: the timed region still performs K uploads for K frames
        e_ms = timed(lambda k: e2e_frame(k + 2), K)
        copy_stream.synchronize()
        e2e = {
            "value": tested_all * K / (e_ms * 1e-3),
            "unit": "meshlets/s",
            "h2d_bytes_per_step": int(st["h2d"]),
            "d2h_bytes_per_step": int(st["d2h"]),
            "ms_per_step": e_ms / K,
            "what": "per step: H2D MeshDraw[] + depth target from pinned host memory (double-buffered: the copy for frame k+1 overlaps frame k), the frame, D2H counters then the visible MeshTaskCommand and cluster-index slabs",
        }
        path.db = db_orig
        depth = depth_sets[0]

        if world == 1:
            # incremental: what the reference's frame loop moves per frame (niagara.cpp:1362-1411, 1487-1516): the CullData push
            # constants and the MeshDraws the animation touched go up (one packed {index, MeshDraw} copy + nvc_update_draws
            # scatter), the two indirect-count words come back; depth and the visible slabs never leave the device.
            n_anim = max(1, D // 100)
            anim_idx = np.linspace(0, D - 1, n_anim).astype(np.uint32)
            idx_host = torch.from_numpy(anim_idx.view(np.int32).copy()).pin_memory()
            val_host = torch.from_numpy(np.ascontiguousarray(scene.draws[anim_idx]).view(np.uint8).reshape(-1).copy()).pin_memory()
            idx_dev = torch.empty_like(idx_host, device=dev)
            val_dev = torch.empty_like(val_host, device=dev)
            cd_host = torch.from_numpy(np.frombuffer(bytes(cd), dtype=np.uint8).copy()).pin_memory()
            cd_dev = torch.empty(cd_host.numel(), dtype=torch.uint8, device=dev)

            def inc_frame(k):
                idx_dev.copy_(idx_host, non_blocking=True)
                val_dev.copy_(val_host, non_blocking=True)
                cd_dev.copy_(cd_host, non_blocking=True)  # the push constants' bytes (the C ABI takes them by value from the host)
                check(lib.nvc_update_draws(path.ctx, path._stream(), ctypes.c_void_p(path.db.data_ptr()), D, ctypes.c_void_p(idx_dev.data_ptr()), ctypes.c_void_p(val_dev.data_ptr()), n_anim), path.ctx, "nvc_update_draws")
                frame(cd)
                count_host[:4].copy_(path.dccb, non_blocking=True)
                count_host[4:].copy_(path.ccb, non_blocking=True)
                main_stream.synchronize()

            for k in range(2):
                inc_frame(k)
            i_ms = timed(inc_frame, K)
            e2e_inc = {
                "value": tested_all * K / (i_ms * 1e-3),
                "unit": "meshlets/s",
                "h2d_bytes_per_step": int(idx_host.numel() * 4 + val_host.numel() + cd_host.numel()),
                "d2h_bytes_per_step": 32,
                "ms_per_step": i_ms / K,
                "what": "per step: H2D CullData + %d animated MeshDraws (1%% of the scene, packed {index, MeshDraw} + nvc_update_draws scatter), the frame, D2H of the two indirect-count blocks, host waits for them" % n_anim,
            }

    clocks = sampler.stop() if rank == 0 else None  # sampled across the timed regions
    if rank == 0:
        # ---- roofline of the dominant kernel, with THAT pass's algorithmic bytes (SURVEY §8(d)) ----
        W, Hh = scene.screen
        hz = path.hiz
        pyr_texels = int(hz.total_texels)
        fp_first = int(os.environ.get("NVC_FP_FIRST_LEVEL", "0"))
        fp_texels = sum((max(1, hz.width >> l) + 1) * (max(1, hz.height >> l) + 1) for l in range(min(fp_first, hz.levels - 1), hz.levels)) if has_fp else 0
        alg = {
            # per draw: 48 (MeshDraw) + 4 (dvb) + 32 (cull head, drawn from the 208-byte Mesh once per geometry upload) + 20 per command written
            "drawcull_early": pr["early_reached"] * (48 + 4 + 32) + (D - pr["early_reached"]) * (16 + 4) + pr["cmds_early"] * 20,
            "drawcull_late": D * (48 + 4 + 4 + 32) + pr["cmds_late"] * 20,
            # per meshlet tested: 24 (Meshlet) + bits; per command 20; per visible draw 48; 4 per emitted cluster
            "clustercull_early": pr["emitted_early"] * 0 + pr["tested_early"] * 24 + pr["cmds_early"] * 20 + pr["draws_early"] * 48 + pr["tested_early"] / 8.0 + 4 * pr["emitted_early"],
            "clustercull_late": pr["tested_late"] * 24 + pr["cmds_late"] * 20 + pr["draws_late"] * 48 + 2 * pr["tested_late"] / 8.0 + 4 * pr["emitted_late"],
            # depth read once, every mip written once (+ the footprint image written once)
            "pyramid": 4 * W * Hh + 4 * pyr_texels + 4 * fp_texels,
        }
        mean_ms = pass_ms.mean(axis=0)
        dom = int(np.argmax(mean_ms))
        dom_name = NAMES[dom]
        k_ms = float(mean_ms[dom])
        achieved = alg[dom_name] / (k_ms * 1e-3) / 1e9
        share = mean_ms / mean_ms.sum()
        traffic = profiled(dom_name, args, "dram__bytes_")
        line = {
            "metric": "meshlets culled/sec",
            "value": tested_all * K / (max_ms * 1e-3),
            "unit": "meshlets/s",
            "n_gpus": world,
            "steps": K,
            "warmup": max(3, args.warmup),
            "ms_per_step": max_ms / K,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f32",
            "data": "synthetic",
            "config": {
                "workload": workload_label(args),  # (per GPU: weak scaling; identical string in the reference arm)
                "per": "GPU (weak scaling: every rank culls its own scene of this size)",
                "step": "one frame: early drawcull+tasksubmit, early clustercull+clustersubmit, depth pyramid%s, late drawcull+tasksubmit, late clustercull+clustersubmit (%d launches)%s" % (" + footprint image" if has_fp else "", 6 if has_fp else 5, {"ce": "; + all-gather of the late MeshTaskCommand slabs+counters by copy-engine peer pushes over NVLink (nvc_gather_*), every frame, pipelined one frame deep: the exchange of frame k must complete before drawcull(late) of frame k+1 overwrites the slab, and the last one before the clock stops", "sm": "; + all-gather of the late MeshTaskCommand slabs+counters by a unicast peer-store kernel (nvc_gather_*), every frame, one frame deep", "mc": "; + all-gather of the late MeshTaskCommand slabs+counters by ONE NVSwitch-multicast store kernel per rank (nvc_gather_*, symmetric memory), every frame, one frame deep", "fused": "; + all-gather of the late MeshTaskCommand slabs FUSED into drawcull(late): its command write-out also goes through the NVSwitch multicast mapping (counters + flags follow), every frame, one frame deep", "nccl": "; + ncclAllGather of the late MeshTaskCommand slabs+counters on a high-priority side stream", "none": ""}[gather]),
                "counting": "value = meshlet instances TESTED by the two cluster passes per second (early %d + late %d per step per GPU); draws_per_s likewise (early %d + late %d)" % (pr["tested_early"], pr["tested_late"], pr["early_reached"], D),
                "l2": "inputs larger than L2 (Meshlet[] %d MB + MeshDraw[] %d MB + Mesh[] %d MB + depth %d MB per step vs 126 MB L2), no flush" % (scene.meshlets.nbytes >> 20, scene.draws.nbytes >> 20, scene.meshes.nbytes >> 20, scene.depth.nbytes >> 20),
                "cluster_backface": 1,
                "parallelism": "draw-sharded x%d" % world,
            },
            "draws_per_s": draws_all * K / (max_ms * 1e-3),
            **({"cull_only_value": tested_all / (mean_ms.sum() * 1e-3), "cull_only_note": "meshlets tested per second over the five cull-path passes alone (the step above also contains the two raster passes that produce the depth)"} if produced is not None else {}),
            "passes_ms": {n: float(mean_ms[i]) for i, n in enumerate(NAMES)},
            **({"raster_ms": {"early": float(raster_ms[:, 0].mean()), "late": float(raster_ms[:, 1].mean()), "what": "nvc_raster_depth (stand-in for the reference's mesh stage + rasteriser): produces the depth the late pass culls against; not part of the cull path"}} if produced is not None else {}),
            "passes_share": {n: float(share[i]) for i, n in enumerate(NAMES)},
            "passes_hbm_frac": {n: float(alg[n] / (mean_ms[i] * 1e-3) / 1e9 / peak_gbs) for i, n in enumerate(NAMES)},
            "frame_hbm_frac": float(sum(alg.values()) / (mean_ms.sum() * 1e-3) / 1e9 / peak_gbs),
            "visible": {"late_commands": pr["cmds_late"], "late_visible_draws": pr["draws_late"], "late_emitted_clusters": pr["emitted_late"], "early_commands": pr["cmds_early"], "early_emitted_clusters": pr["emitted_early"]},
            "roofline": {
                "kernel": "%s (dominant pass: %s, %.0f%% of the step)" % (KERNEL_OF_PASS[dom_name], dom_name, 100 * share[dom]),
                "bound": "hbm",
                "achieved": achieved,
                "peak": peak_gbs,
                "peak_source": peak_src,
                "unit": "GB/s",
                "frac": achieved / peak_gbs,
                "traffic": traffic,
                "traffic_source": "ncu --set full of this command, profiles/r2_frame_ncu_summary.json (dram__bytes_read.sum + dram__bytes_write.sum, per launch)" if traffic else None,
                "algorithmic_bytes_per_launch": alg[dom_name],
                "kernel_ms": k_ms,
            },
            "clocks": clocks,
            "timing": {
                "headline": ("CUDA-graph replay, %d frame(s) per graph (median of 3 regions of %d frames)" % (GF, K)) if graph_ms else "eager launches from the host (%d frames; the faster of the regions with / without per-pass timing events)" % K,
                "graph_ms_per_step": ({k: v / K for k, v in graph_ms.items()} if graph_ms else None),
                "eager_ms_per_step": eager_ms / K,
                "eager_no_events_ms_per_step": plain_ms / K,
                **({"graph_unavailable": graph_note} if graph_note else {}),
            },
            **({"without_exchange": {"value": tested_all * K / (cull_only_ms * 1e-3), "unit": "meshlets/s", "ms_per_step": cull_only_ms / K, "what": "the same frames with the all-gather switched off (--gather none), eager launches like the headline region at N > 1, same process: cull-only scaling beside cull + gather (SURVEY 8(e))"}} if cull_only_ms else {}),
            "gpu_launches": gpu_launches,
            "gather_transport": transport if not gather_note else "ce",
            **({"gather_note": gather_note} if gather_note else {}),
            "cluster_filter": {
                "enabled": os.environ.get("NVC_CLUSTER_FILTER", "1") != "0",
                "footprint_image": has_fp,
                "meshlets_filtered_per_step": int(filter_stats[0]) // max(K, 1),
                "took_exact_path_per_step": int(filter_stats[1]) // max(K, 1),
                "exact_share": (float(filter_stats[1]) / float(filter_stats[0])) if filter_stats[0] else None,
            },
        }
        inst = profiled("clustercull_late", args, "smsp__inst_executed.sum")
        if inst:
            mhz = (clocks or {}).get("sm_mhz") or 1965.0
            peak_i = 148 * 4 * mhz * 1e6
            line["issue_roofline"] = {"kernel": KERNEL_OF_PASS["clustercull_late"], "warp_instructions_per_launch": inst, "achieved_ginst_s": inst / (mean_ms[4] * 1e-3) / 1e9, "peak_ginst_s": peak_i / 1e9, "frac": inst / (mean_ms[4] * 1e-3) / peak_i}
        if multi_gpu_verified is not None:
            line["multi_gpu_verified"] = multi_gpu_verified and not exchange_timed_out
        if exchange_timed_out:
            line["exchange_timed_out"] = True  # a device-side wait of the protocol gave up (nvc_gather_status): the gathered data are void
        if multi_gpu_note:
            line["multi_gpu_verified_error"] = multi_gpu_note
        line.update(extras)
        if e2e:
            line["e2e"] = e2e
            if e2e_inc:
                line["e2e_incremental"] = e2e_inc
        if not args.no_cpu_baseline and world == 1:  # the CPU arm is timed at N = 1 only
            line["cpu_baseline"] = cpu_baseline(args, scene, cpu_threads())
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
