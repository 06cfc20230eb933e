#!/usr/bin/env python3
"""bench.py -- Louvain-phase throughput on synthetic RGGs (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path (oracle/_ref) on host cores

A "step" is one complete Louvain phase (the scope of the reference's timer, main.cpp:162-173: init +
ghost setup + all iterations until the modularity gain drops below 1e-6) over one synthetic RGG.
Workload at N GPUs: the graph `miniVite -n (16777216*N)` builds on N ranks (BASELINE.json configs[1] at
N=1; 16M vertices per GPU for N>1 => weak scaling), produced by this repo's exact fast generator.  BOTH arms run
that same graph (`config` is identical in the two JSON lines).
metric = edges/s = (directed edge count) * iterations / t_louvain, whole job.
  value : graph already resident in HBM in the reference's own array format when the clock starts
  e2e   : host (pinned) arrays -> mvgpu_upload_shard (H2D) -> mvgpu_louvain -> assignment back to host
Parity: before anything is timed, one traced run is compared with the golden trace of the UNMODIFIED reference on
the same graph (tests/golden/golden_full_<nv>_p<N>.json: iteration count, every (modularity, moved, community
hash) triple, final assignment hash); a mismatch aborts the benchmark with a non-zero exit code.
Timing: CUDA events on the library's stream (max over ranks) for `value`; inputs (3 GB/GPU) exceed L2 so
no explicit flush is needed between steps.
--dump-outputs DIR: after the timed steps, what the last timed `value` step returned to its caller is written as
DIR/<name>.npy (float64): modularity, iterations, and the final community of a fixed, seeded sample of at most 2^21
vertices (community_vertices.npy holds their global ids).  The graph is a function of the arguments, so two builds
run with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)

NV_PER_GPU = 16777216
METRIC = "louvain_phase_edges_per_sec"
DUMP_SAMPLE = 1 << 21               # --dump-outputs: vertices whose community is written (2 x 16 MB of float64)
DUMP_SEED = 20240601


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.f.name):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if c[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def host_cores():
    """(usable cores, detail): the scheduler affinity mask capped by the cgroup CPU quota -- a container that sees
    128 CPUs in its affinity mask but holds a 16-CPU quota runs 128 busy threads at 1/8 speed each."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    eff = aff if quota is None else max(1, min(aff, int(quota)))
    return eff, {"affinity": aff, "cgroup_quota": quota}


def workload_config(N, nv_total, ne_total):
    """The static description of the workload: identical in both arms' JSON lines."""
    return {"workload": f"RGG -n {nv_total} on {N} rank(s) (BASELINE.json configs[1] per GPU: {nv_total // N} vertices per "
                        f"rank), unit weights, one full Louvain phase (reference timer main.cpp:162-173)",
            "nv": nv_total, "ne": ne_total, "strips": N, "graph": "reference GenerateRGG, seed reseeder(1)",
            "l2": "inputs (3 GB per GPU) larger than L2; no flush"}


def load_golden(nv_total, N):
    p = os.path.join(ROOT, "tests", "golden", f"golden_full_{nv_total}_p{N}.json")
    return (json.load(open(p)), os.path.relpath(p, ROOT)) if os.path.exists(p) else (None, None)


def comm_hash_np(base, comm):
    """Shard-combinable hash of an assignment (SURVEY.md 8(c)): sum_i mix64((base+i)*K ^ comm[i]) mod 2^64."""
    with np.errstate(over="ignore"):
        gid = np.arange(base, base + len(comm), dtype=np.uint64)
        z = gid * np.uint64(0x9E3779B97F4A7C15) ^ comm.astype(np.uint64)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return int(z.sum(dtype=np.uint64))


def scratch_dir(need_bytes):
    """Directory for the reference's input file: RAM-backed if it has room, else the default temp dir."""
    for d in ("/dev/shm", tempfile.gettempdir()):
        try:
            if shutil.disk_usage(d).free > need_bytes * 1.2:
                return tempfile.mkdtemp(prefix="mvbench_", dir=d)
        except Exception:
            pass
    return tempfile.mkdtemp(prefix="mvbench_")


def reference_runs(nv_total, N, max_timed, budget_s, verbose=False, fallback_nv=2097152):
    """Time oracle/_ref/miniVite_ref -- the unmodified reference -- on the benchmark graph itself (N strips, read with
    -f), in its genuine MPI+OpenMP mode: N ranks x (cores/N) OpenMP threads (N=1: one rank x all cores).  One warm-up
    run, then up to `max_timed` timed runs while the time budget lasts; if a single run does not fit the budget the
    run that was made is the sample.  Only if the reference binary is missing does the C restatement stand in: on the
    benchmark graph itself up to `fallback_nv` vertices, on the 1-strip RGG of `fallback_nv` vertices above that."""
    from minivite_b200 import hostgraph as hg
    from oracle import oracle as O
    cores, cores_detail = host_cores()
    hg.set_num_threads(cores)
    t0 = time.time()
    ss = hg.generate_rgg(nv_total, N)
    ne = sum(s.lne for s in ss.shards)
    if not O.have_reference():
        same = nv_total <= fallback_nv
        if not same:
            ss.close()
            ss = hg.generate_rgg(fallback_nv, 1)
        t = time.time()
        r = O.louvain(ss.shards[0].parts, [s.rowptr for s in ss.shards], [s.edges for s in ss.shards])
        t = time.time() - t
        return {"value": sum(s.lne for s in ss.shards) * r["iters"] / t, "ms_per_step": t * 1e3, "cores": 1,
                "kind": "port", "ne": ne, "unit": "edges/s", "same_graph": same, "runs_timed": 1,
                "cores_detail": cores_detail,
                "sample": f"oracle/_ref absent: C restatement, 1 thread, RGG n={nv_total if same else fallback_nv} "
                          f"({N if same else 1} strip(s)) full Louvain phase"}
    tmp = scratch_dir(16 * ne + 8 * nv_total)
    path = os.path.join(tmp, "g.bin")
    ss.write(path)
    ss.close()
    gen_s = time.time() - t0
    thr = max(1, cores // N)
    env_bind = {"OMP_PROC_BIND": "true"} if N == 1 else {}
    os.environ.update(env_bind)
    times, iters = [], None
    t_begin = time.time()
    try:
        for k in range(1 + max_timed):
            r = O.run_reference(["-f", path], nranks=N, threads=thr, trace=False, arena_gb=max(16, (24 * ne) >> 30))
            iters = r["result"]["iters"]
            times.append(r["result"]["time"])
            if verbose:
                print(f"# reference run {k}: {r['result']['time']:.2f} s, {iters} iterations", file=sys.stderr)
            elapsed = time.time() - t_begin
            if elapsed + 1.2 * max(times) > budget_s:
                break
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    timed = times[1:] if len(times) > 1 else times          # first run = warm-up unless it is the only one
    t = statistics.mean(timed)
    return {"value": ne * iters / t, "ms_per_step": t * 1e3, "cores": cores, "kind": "reference", "ne": ne,
            "unit": "edges/s", "same_graph": True, "runs_timed": len(timed), "iters": iters,
            "cores_detail": cores_detail,
            "sample": (f"the benchmark graph itself (RGG -n {nv_total}, {N} strip(s), {ne} directed edges), full Louvain "
                       f"phase by the unmodified reference (oracle/_ref, timer main.cpp:162-173), {N} rank(s) x {thr} "
                       f"OpenMP threads on {cores} usable cores; {'1 warm-up + ' if len(times) > 1 else 'no warm-up, '}"
                       f"{len(timed)} timed run(s): " + ", ".join(f"{x:.2f} s" for x in timed) +
                       f"; graph built + written in {gen_s:.0f} s (not timed)")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nv-per-gpu", type=int, default=NV_PER_GPU, help="dev knob; the benchmark config is the default")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="dev knob: skip the golden-trace check")
    ap.add_argument("--compact-upload", type=int, default=-1, metavar="THREADS",
                    help="e2e leg: host threads that narrow unit-weight shards to 4-byte tails while the copy engine ships "
                         "them (library option compact_upload); 0 = ship the 16-byte records; default = min(32, cores/ranks)")
    ap.add_argument("--upload-mode", type=int, default=2, choices=[1, 2],
                    help="e2e leg, library option compact_upload: 1 = every chunk narrowed by host threads; 2 (default) = "
                         "the copy engine additionally takes raw chunks from the far end whenever no narrowed chunk is ready")
    ap.add_argument("--ref-budget-s", type=float, default=420.0, help="wall-clock budget of the reference arm's runs")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (modularity, iterations, sampled communities) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    N = args.gpus
    # exactly ONE JSON line may reach stdout (libraries such as NCCL print banners there): park the real stdout
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    cores, cores_detail = host_cores()
    if world > 1:   # the host-side graph generator is OpenMP code: do not oversubscribe the cores across ranks
        os.environ["OMP_NUM_THREADS"] = str(max(1, cores // world))

    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world != N and world != 1:
        raise SystemExit(f"WORLD_SIZE={world} but --gpus {N}")
    nv_total = args.nv_per_gpu * N

    import __graft_entry__ as ge

    if args.impl == "reference":
        if rank != 0:
            return 0
        ge.build_host_only()
        r = reference_runs(nv_total, N, max_timed=2, budget_s=args.ref_budget_s, verbose=args.verbose)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "edges/s",
                "n_gpus": N, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": workload_config(N, nv_total, r["ne"]),
                "reference_runs_timed": r["runs_timed"], "host_cores": dict(cores_detail, usable=r["cores"]),
                "cpu_baseline": {"value": r["value"], "unit": "edges/s", "cores": r["cores"], "kind": r["kind"],
                                 "sample": r["sample"], "same_graph_as_gpu_arm": r["same_graph"]},
                "e2e": {"value": r["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return 0

    import torch
    import torch.distributed as dist
    ge.build()
    from minivite_b200 import gpu as G
    from minivite_b200 import hostgraph as hg

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allred(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def allmax(x):
        return allred(x, dist.ReduceOp.MAX if world > 1 else None)

    def allsum(x):
        return allred(x, dist.ReduceOp.SUM if world > 1 else None)

    def allsum_u64(x):
        """sum mod 2^64 across ranks (two 32-bit halves through an int64 all-reduce)"""
        if world == 1:
            return x & 0xFFFFFFFFFFFFFFFF
        t = torch.tensor([x & 0xFFFFFFFF, (x >> 32) & 0xFFFFFFFF], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        lo, hi = int(t[0].item()), int(t[1].item())
        return (lo + (hi << 32)) & 0xFFFFFFFFFFFFFFFF

    # ---- synthetic input: this rank's strip of the N-strip RGG (exact reference graph)
    hg.set_num_threads(max(1, cores // max(world, 1)))
    t0 = time.time()
    ss = hg.generate_rgg(nv_total, N, rank, rank + 1)
    sh = ss.shards[0]
    gen_s = time.time() - t0
    ne_total = int(allsum(float(sh.lne)))
    parts = np.array([(nv_total * r) // N for r in range(N + 1)], dtype=np.int64)
    if args.verbose and rank == 0:
        print(f"# generated strip: lnv={sh.lnv} lne={sh.lne} in {gen_s:.1f}s", file=sys.stderr)

    ctx = G.LouvainGPU(local_rank, rank, N)
    if N > 1:
        idt = torch.zeros(G.UNIQUE_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(G.get_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        ctx.comm_init(bytes(idt.cpu().numpy().tobytes()))

    # ---- inputs resident in HBM (reference array format)
    h_rowptr = torch.from_numpy(np.ascontiguousarray(sh.rowptr)).pin_memory()
    h_edges = torch.from_numpy(np.ascontiguousarray(sh.edges).view(np.uint8)).pin_memory()
    d_rowptr = h_rowptr.cuda(non_blocking=True)
    d_edges = h_edges.cuda(non_blocking=True)
    torch.cuda.synchronize()
    ctx.attach_device(nv_total, parts, sh.lnv, sh.lne, d_rowptr.data_ptr(), d_edges.data_ptr(), keepalive=(d_rowptr, d_edges))

    # ---- parity gate (untimed): one traced run against the reference's golden trace of this very graph
    golden, golden_name = load_golden(nv_total, N)
    parity = {"golden": golden_name, "checked": False}
    if not args.no_parity:
        ctx.set_option("trace", 1)
        barrier()
        mod_p, iters_p = ctx.louvain()
        tr = ctx.trace()
        h_final = allsum_u64(comm_hash_np(int(parts[rank]), ctx.communities()))
        ctx.set_option("trace", 0)
        if golden is not None:
            ok_ne = golden["ne"] == ne_total
            ok_iters = golden["iters"] == iters_p
            ok_mod = float(golden["modularity"]) == mod_p
            ok_trace = ok_iters and all(float(g["modularity"]) == float(t["modularity"]) and g["moved"] == int(t["moved"])
                                        and int(g["chash"], 16) == int(t["chash"]) for g, t in zip(golden["trace"], tr))
            ok_final = int(golden["final_chash"], 16) == h_final
            parity.update(checked=True, edges_match=ok_ne, iters_match=ok_iters, modularity_match=ok_mod,
                          trace_match=bool(ok_trace), final_assignment_hash_match=ok_final, iterations=iters_p,
                          tolerance="bit-exact (unit weights): modularity compared as IEEE doubles, hashes as integers",
                          golden_source="unmodified reference (oracle/_ref) on %d rank(s), tools/make_fullsize_golden.py"
                                        % golden.get("ref_ranks", N))
            if not (ok_ne and ok_iters and ok_mod and ok_trace and ok_final):
                if rank == 0:
                    print(f"bench.py: PARITY FAILURE against {golden_name}: {parity}", file=sys.stderr)
                    emit({"metric": METRIC, "value": None, "n_gpus": N, "parity": parity, "error": "parity failure"})
                os._exit(3)
        else:
            parity.update(note="no committed golden for this size: traced run made, nothing to compare with",
                          iterations=iters_p, final_assignment_hash="%016x" % h_final)

    # ---- value: graph resident in HBM when the clock starts
    for _ in range(args.warmup):
        barrier()
        mod, iters = ctx.louvain()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    step_dev, step_wall, scan_s, scan_n, launches = [], [], 0.0, 0, 0
    phase_acc = {"setup_s": 0.0, "scan_s": 0.0, "fold_s": 0.0, "exchange_s": 0.0, "reorder_s": 0.0}
    for _ in range(args.steps):
        barrier()
        w0 = time.perf_counter()
        mod, iters = ctx.louvain()
        torch.cuda.synchronize()
        step_wall.append(time.perf_counter() - w0)
        tm = ctx.timings()
        step_dev.append(tm["total_s"])
        scan_s += tm["scan_s"]
        scan_n += tm["iters"]
        launches += tm["kernel_launches"]
        for k in phase_acc:
            phase_acc[k] += tm[k]
    barrier()
    t_dev = allmax(sum(step_dev)) / args.steps          # device-timed (CUDA events), max over ranks
    t_wall = allmax(sum(step_wall)) / args.steps
    value = ne_total * iters / t_dev
    t_scan_iter = allmax(scan_s / max(scan_n, 1))       # avg duration of one scan launch, slowest rank
    tm_last = ctx.timings()
    info = ctx.shard_info()
    if not args.no_parity:
        assert iters == iters_p and mod == mod_p, "timed runs disagree with the parity run"
    if args.dump_outputs:
        # the last timed step's assignment at a fixed, seeded sample of global vertex ids; each rank fills the entries
        # it owns and a sum over ranks (exact: every entry has one non-zero contribution) assembles the sample
        idx = (np.sort(np.random.default_rng(DUMP_SEED).choice(nv_total, DUMP_SAMPLE, replace=False))
               if nv_total > DUMP_SAMPLE else np.arange(nv_total, dtype=np.int64))
        comm = ctx.communities(out=torch.empty(sh.lnv, dtype=torch.int64).pin_memory().numpy())
        own = (idx >= parts[rank]) & (idx < parts[rank + 1])
        sampled = np.zeros(len(idx), np.float64)
        sampled[own] = comm[idx[own] - parts[rank]]
        if world > 1:
            buf = torch.from_numpy(sampled).cuda()
            dist.all_reduce(buf)
            sampled = buf.cpu().numpy()
        outputs = {"modularity": np.array([mod], np.float64), "iterations": np.array([iters], np.float64),
                   "communities": sampled, "community_vertices": idx.astype(np.float64)}
        del comm

    # ---- e2e: host arrays -> H2D -> Louvain -> assignment D2H, through the public API
    cu_threads = args.compact_upload if args.compact_upload >= 0 else max(1, min(32, cores // max(world, 1)))
    if cu_threads > 0:
        ctx.set_option("compact_upload", args.upload_mode)
        ctx.set_option("host_threads", cu_threads)
    e2e_t = []
    h_comm = torch.empty(sh.lnv, dtype=torch.int64).pin_memory().numpy()      # the user's (pinned) result buffer
    for k in range(args.warmup + args.steps):
        barrier()
        w0 = time.perf_counter()
        ctx.upload(nv_total, parts, h_rowptr.numpy(), h_edges.numpy().view(hg.EDGE_DTYPE))
        m2, it2 = ctx.louvain()
        ctx.communities(out=h_comm)
        torch.cuda.synchronize()
        if k >= args.warmup:
            e2e_t.append(time.perf_counter() - w0)
        tm_e2e = ctx.timings()
        h2d_bytes = tm_e2e["h2d_bytes"]
        assert it2 == iters and m2 == mod
    clocks = sampler.stop()                             # sampled across both timed regions (value + e2e steps)
    t_e2e = allmax(sum(e2e_t)) / args.steps
    e2e_value = ne_total * iters / t_e2e
    launches_total = int(allsum(float(launches)))
    h2d_total = int(allsum(float(h2d_bytes)))
    nsend_total = int(allsum(float(info["nsend"])))

    if rank != 0:
        ctx.close()
        if world > 1:
            dist.destroy_process_group()
        return 0

    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    peak, peak_src = load_peaks()
    lnv, lne = sh.lnv, sh.lne
    b_alg = 24.0 * lne + 56.0 * lnv            # SURVEY.md 8(d): reference element sizes, per scan launch per GPU
    b_own = 8.0 * lne + 28.0 * lnv             # this build: 4 B tail + 4 B gathered id per edge; per vertex 4 rowptr
    #                                            + 4 cur + 8 cinfo + 4 tgt write + 8 (packed delta atomics, 2 x 57% ~ 1)
    roof = {"bound": "hbm", "achieved": b_alg / t_scan_iter / 1e9, "peak": peak, "unit": "GB/s",
            "frac": b_alg / t_scan_iter / 1e9 / peak, "traffic": None,
            "kernel": "neighbour scan (k_scan_pq / k_scan_pw, chosen at run time; scan_pipe.cuh, scan_queue.cuh)", "algorithmic_bytes_per_launch": b_alg,
            "definition": "achieved = SURVEY 8(d) canonical bytes (24*ne + 56*nv, the reference's 64-bit element sizes) / "
                          "avg launch time; the kernel moves fewer bytes than that (32-bit ids, implicit unit weights, "
                          "cached gathers), so see frac_own_layout and frac_dram_traffic for what the hardware did",
            "own_layout_bytes_per_launch": b_own, "achieved_own_layout": b_own / t_scan_iter / 1e9,
            "frac_own_layout": b_own / t_scan_iter / 1e9 / peak,
            "avg_launch_ms": t_scan_iter * 1e3, "peak_source": peak_src,
            "whole_phase_gbs": b_alg * iters / t_dev / 1e9}
    prof = os.path.join(ROOT, "profiles", "scan_traffic.json")
    if N == 1 and os.path.exists(prof):            # ncu capture of THIS configuration only (N=1, config 2)
        try:
            tj = json.load(open(prof))
            roof["traffic"] = tj.get("dram_bytes_per_launch")
            roof["traffic_source"] = tj.get("source")
            if roof["traffic"]:
                roof["frac_dram_traffic"] = roof["traffic"] / t_scan_iter / 1e9 / peak
        except Exception:
            pass
    cpu = None
    if N == 1 and not args.no_cpu_baseline:
        ss.close()
        r = reference_runs(nv_total, N, max_timed=1, budget_s=240.0, verbose=args.verbose)
        cpu = {"value": r["value"], "unit": "edges/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "same_graph_as_gpu_arm": r["same_graph"]}
    steps_n = max(args.steps, 1)
    line = {"metric": METRIC, "value": value, "unit": "edges/s", "n_gpus": N,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": workload_config(N, nv_total, ne_total),
            "result": {"iterations": iters, "modularity": mod, "s_per_iter": t_dev / iters,
                       "unit_weight_path": bool(tm_last["unit_weight"]), "nghost_rank0": info["nghost"],
                       "arithmetic": "modularity gains in fp64 with the reference's rounding sequence; ids int32 on the device "
                                     "(int64 at the boundary); unit-weight degrees as exact integers",
                       "wall_ms_per_step": t_wall * 1e3, "graph_gen_s": gen_s},
            "parity": parity,
            "roofline": roof, "cpu_baseline": cpu, "host_cores": dict(cores_detail, usable=cores),
            "e2e": {"value": e2e_value, "unit": "edges/s", "ms_per_step": t_e2e * 1e3,
                    "h2d_bytes_per_step": h2d_total,
                    "path": "pinned host arrays -> mvgpu_upload_shard -> mvgpu_louvain -> mvgpu_get_communities (pinned int64 result)",
                    "compact_upload_threads": cu_threads, "compact_upload_mode": args.upload_mode if cu_threads else 0,
                    "d2h_bytes_per_step": int(nv_total * 8 + 16)},
            "gpu_launches": launches_total, "clocks": clocks,
            "nvlink": None if N == 1 else {
                "ghost_values_pushed_per_iteration": nsend_total, "bytes_per_iteration_all_gpus": nsend_total * 4,
                "note": "per iteration every boundary vertex's new community (4 B) is stored into each peer that ghosts it; "
                        "remote Comm reads / delta atomics (only for communities owned by a peer) come on top"},
            "phase_ms": {"setup": phase_acc["setup_s"] / steps_n * 1e3, "renumbering_in_setup": phase_acc["reorder_s"] / steps_n * 1e3,
                         "scan": phase_acc["scan_s"] / steps_n * 1e3, "fold": phase_acc["fold_s"] / steps_n * 1e3,
                         "exchange": phase_acc["exchange_s"] / steps_n * 1e3, "h2d_of_e2e_step": tm_e2e["h2d_s"] * 1e3}}
    emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
