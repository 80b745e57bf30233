#!/usr/bin/env python
"""Benchmark of the hot path: yk_solution::run_solution for iso3dfd (16th order, fp32).

Contract (see task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line
on rank 0.  Metric = GPoints/s (= domain points x steps / seconds inside run_solution, the reference's
"throughput (num-points/sec)", /root/reference/src/kernel/lib/soln_apis.cpp:455-461).

  value       whole-job GPoints/s with all inputs resident in HBM, device time (CUDA events on the
              launching stream), max over ranks.
  sustained   the same loop kept running for >= 2 s (power-capped clocks), with its own clock samples.
  e2e         same metric through the public C-ABI with HOST buffers: set_elements_in_slice (H2D from
              pinned memory) of p(t), p(t-1), v  ->  run_solution(K steps)  ->  get_elements_in_slice
              (D2H) of the final p.  A time-stepping job moves its state once, not every step, so the
              per-step byte counts are total/K.
  roofline    algorithmic 16 B/point-step (read p(t), p(t-1), v; write p(t+1)) x points per launch
              / mean kernel launch time, against the measured copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline the reference's own optimized CPU path (oracle/_ref, built from the unmodified
              sources) timed on this box's host cores on a bounded sample, with the reference harness's
              own defaults (warm-up, 3 trials) once with its best-known block sizes and once after its
              pre-auto-tuner; the exact command lines are recorded.
  halo_check  (N > 1) every rank recomputes the planes on both sides of its x interfaces from the same
              global hash data with a stand-alone single-rank solution and compares bit for bit.
  secondary   BASELINE.json configs 3 and 5 on the same GPUs: awp_elastic fp32 512^3 and ssg fp64 512^3
              per GPU (weak scaling over an N x 1 x 1 rank grid), each with its algorithmic-bytes roofline
              and, at N = 1, the reference's CPU harness of the same stencil beside it.

`--impl reference` times the reference's CPU implementation instead (rank 0 only).
N > 1: weak scaling, 1024^3 points per GPU, domain split along x (the outermost storage dim).
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_POINT = 16  # SURVEY.md section 8(d): 3 arrays read + 1 written, fp32
SECONDARY = (("awp_elastic", "awp_elastic fp32 (staggered-grid elastic, 2 stages)", 120, "f32"),
             ("ssg", "ssg fp64 (staggered-grid elastic, 8th order, 2 stages)", 248, "f64"))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=1024, help="points per dim per GPU")
    ap.add_argument("--size2", type=int, default=512, help="points per dim per GPU of the secondary workloads")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--no-halo-check", action="store_true")
    ap.add_argument("--replicas", action="store_true", help="diagnostic: under torchrun every rank runs an INDEPENDENT single-rank "
                    "solution (no halo exchange); shows what N busy GPUs of one box cost before any exchange")
    ap.add_argument("--opt", action="append", default=[], help="engine option key=value")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of the p(t) they computed "
                    "to DIR/p.npy (see dump_outputs), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the B200 path computed; it does not apply to --impl reference")
    return args


# --------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks DURING the timed region")
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device, period_ms=50):
        self.device, self.rows, self.proc, self.period = device, [], None, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.period)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def window(self, t0, t1):
        """Median SM clock and the throttle reasons seen between t0 and t1 (the sampler keeps running)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], None, set()
        for ts, line in list(self.rows):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            if t0 - 0.05 <= ts <= t1 + 0.15:
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}

    def stop(self):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()


# --------------------------------------------------------------------------------------------------
# reference CPU arm / cpu_baseline
# --------------------------------------------------------------------------------------------------
def host_cpu_info():
    """CPU model, flags line, hardware threads, physical cores (distinct (socket, core id) pairs), sockets."""
    model, flags, cores, sockets = "unknown", "", set(), set()
    phys = core = None
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and model == "unknown":
                model = line.split(":", 1)[1].strip()
            elif line.startswith("flags") and not flags:
                flags = line
            elif line.startswith("physical id"):
                phys = line.split(":", 1)[1].strip()
                sockets.add(phys)
            elif line.startswith("core id"):
                core = line.split(":", 1)[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    cores.add((phys, core))
                phys = core = None
    except OSError:
        pass
    threads = os.cpu_count() or 1
    try:
        threads = len(os.sched_getaffinity(0))
    except Exception:
        pass
    ncores = len(cores) if cores else threads
    return {"model": model, "flags": flags, "threads": threads, "cores": min(ncores, threads), "sockets": max(1, len(sockets))}


REF_EXE = {"iso3dfd": "yask_kernel.iso3dfd.{arch}.exe", "awp_elastic": "yask_kernel.awp_elastic.{arch}.exe", "ssg": "yask_kernel.ssg-fp64.{arch}.exe"}


def _ref_dirs():
    for sub in ("yask", "ship"):
        b = os.path.join(ROOT, "oracle", "_ref", sub, "bin")
        if os.path.isdir(b):
            yield b, os.path.join(ROOT, "oracle", "_ref", sub, "lib")


def run_reference_cpu(stencil, size, steps, budget_s=150.0, try_tuned=False):
    """Time the unmodified reference's optimized path (the reference's own harness src/kernel/yask_main.cpp, built out of
    tree by oracle/build_ref.sh) on the host cores, as its own defaults run it: warm-up on, 3 trials, `best-throughput`.
    Runs: (A) the solution's built-in best-known block sizes (-no-pre_auto_tune), threads = physical cores, one per core
    (OMP_PLACES=cores); (B) the same with every hardware thread; (C, only with try_tuned: the `--impl reference` arm) the
    harness defaults, i.e. after the reference's pre-auto-tuner -- whose warm-up alone is 1000 steps, minutes at 1024^3, so
    it is attempted within what is left of the time budget and recorded as timed out otherwise.  The largest is reported,
    all are recorded with their exact command lines.
    iso3dfd falls back to the C oracle port (oracle/yask_oracle.c, OpenMP) if the prebuilt reference cannot run here."""
    cpu = host_cpu_info()
    t_start = time.time()
    runs = []
    for bind, libd in _ref_dirs():
        for arch in [a for a in (("avx512" if "avx512f" in cpu["flags"] else None), "avx2") if a]:
            exe = os.path.join(bind, REF_EXE[stencil].format(arch=arch))
            if not os.path.exists(exe):
                continue

            def one(label, extra, nthreads, trials, nsteps, timeout):
                env = dict(os.environ, LD_LIBRARY_PATH=libd + ":" + os.environ.get("LD_LIBRARY_PATH", ""), OMP_NUM_THREADS=str(nthreads),
                           OMP_PLACES="cores" if nthreads <= cpu["cores"] else "threads", OMP_PROC_BIND="spread")
                cmd = [exe, "-g", str(size), "-num_trials", str(trials), "-trial_steps", str(nsteps), "-sleep", "0", "-no-print_suffixes"] + extra
                t0 = time.time()
                try:
                    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
                except Exception as e:
                    runs.append({"label": label, "cmd": " ".join([os.path.basename(exe)] + cmd[1:]), "error": type(e).__name__})
                    return None
                best = re.findall(r"best-throughput \(num-points/sec\):\s*([0-9.eE+]+)", r.stdout)
                mid = re.findall(r"mid-throughput \(num-points/sec\):\s*([0-9.eE+]+)", r.stdout)
                th = re.findall(r"Num OpenMP threads used:\s*(\d+)", r.stdout)
                if r.returncode != 0 or not best:
                    runs.append({"label": label, "cmd": " ".join([os.path.basename(exe)] + cmd[1:]), "error": f"rc {r.returncode}"})
                    return None
                rec = {"label": label, "cmd": " ".join([os.path.basename(exe)] + cmd[1:]), "env": f"OMP_NUM_THREADS={nthreads} OMP_PLACES={env['OMP_PLACES']} OMP_PROC_BIND=spread",
                       "best_gpts": float(best[-1]) / 1e9, "mid_gpts": float(mid[-1]) / 1e9 if mid else None,
                       "threads": int(th[-1]) if th else nthreads, "trials": trials, "steps": nsteps, "wall_s": round(time.time() - t0, 1)}
                runs.append(rec)
                return rec

            left = lambda: budget_s - (time.time() - t_start)
            a = one("bkc (built-in block sizes, -no-pre_auto_tune)", ["-no-pre_auto_tune", "-no-auto_tune"], cpu["cores"], 3, steps, max(30.0, left()))
            if a is None:
                continue
            if cpu["threads"] > cpu["cores"] and left() > a["wall_s"] + 5:
                one("bkc, all hardware threads", ["-no-pre_auto_tune", "-no-auto_tune"], cpu["threads"], 2, steps, max(30.0, left()))
            if try_tuned and left() > 3 * a["wall_s"] + 20:
                one("pre-auto-tuned (harness defaults)", [], cpu["cores"], 3, steps, max(30.0, left() - 10))
            ok = [r for r in runs if "best_gpts" in r]
            top = max(ok, key=lambda r: r["best_gpts"])
            return dict(value=top["best_gpts"], unit="GPoints/s", cores=cpu["cores"], threads=top["threads"], kind="reference",
                        sample=f"{stencil} {size}^3 x {steps} steps x {top['trials']} trials (best), reference harness {os.path.basename(exe)} "
                               f"(g++ -O3, OpenMP), warm-up on; best of {len(ok)} run(s): '{top['label']}'; CPU: {cpu['model']}, "
                               f"{cpu['sockets']} socket(s), {cpu['cores']} cores / {cpu['threads']} threads",
                        mid=top["mid_gpts"], runs=runs)
    if stencil != "iso3dfd":
        return dict(value=None, unit="GPoints/s", cores=cpu["cores"], kind="unavailable", sample=f"no prebuilt reference harness for {stencil} on this CPU", runs=runs)
    # fallback: oracle port
    from oracle import oracle as O
    from yask_b200.synth import hash_field, var_salt
    n = min(size, 256)
    p0 = hash_field(1, var_salt("p", 0), (-8, -8, -8), (n + 16,) * 3, -1, 1)
    p1 = hash_field(1, var_salt("p", 1), (-8, -8, -8), (n + 16,) * 3, -1, 1)
    v = hash_field(1, var_salt("v", 0), (0, 0, 0), (n,) * 3, 0.05, 0.3)
    t0 = time.time()
    O.iso3dfd_run(p0, p1, v, 8, steps, 2)
    dt = time.time() - t0
    return dict(value=n ** 3 * steps / dt / 1e9, unit="GPoints/s", cores=O.lib().yo_num_threads(), kind="port",
                sample=f"iso3dfd r=8 fp32 {n}^3 x {steps} steps, oracle/yask_oracle.c (OpenMP), CPU: {cpu['model']}", runs=runs)


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each "step" = one reference time-step on a bounded sample of the workload: at most 20 steps per trial
    size = args.size if args.size <= 1024 else 1024
    steps = max(1, min(args.steps, 20))
    t0 = time.time()
    cb = run_reference_cpu("iso3dfd", size, steps, budget_s=240.0, try_tuned=True)
    wall = time.time() - t0
    pts = size ** 3
    line = {"metric": f"GPoints/s, iso3dfd-16 fp32 {size}^3 per GPU", "value": cb["value"], "unit": "GPoints/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": pts / (cb["value"] * 1e9) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"iso3dfd radius 8 (16th order) fp32, {size}^3 points on the host CPU (reference OpenMP/AVX path)",
                       "steps_per_trial": steps, "wall_s": round(wall, 1)},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "GPoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
DUMP_SEED, DUMP_BYTES = 20240, 32 << 20


def dump_outputs(out_dir, p, rank, world):
    """Write what the timed run_solution() left in p at its last valid step -- the array its caller reads back -- as
    out_dir/p.npy (out_dir/p.rank<r>.npy per rank when several ranks run): float32 [plane, y, z], y-z planes at x offsets
    drawn once from DUMP_SEED within the rank's domain, as many as fit the rank's share of DUMP_BYTES (8 whole planes,
    32 MiB, at 1024^3 on one GPU); where one plane exceeds that share, seeded y rows of one plane.
    The bench's inputs are fixed hash fields, so the same arguments give the same planes and the same values."""
    import numpy as np
    tl = p.get_last_valid_step_index()
    first, last = p.domain_box(tl)
    nx, ny, nz = (b - a + 1 for a, b in zip(first[1:], last[1:]))
    share = DUMP_BYTES // world
    k = max(1, min(nx, share // (4 * ny * nz)))
    rng = np.random.default_rng(DUMP_SEED)
    xs = sorted(rng.choice(nx, size=k, replace=False).tolist())
    ys = sorted(rng.choice(ny, size=min(ny, max(1, share // (4 * nz))), replace=False).tolist())
    planes = [p.get_elements_in_slice([tl, first[1] + x] + first[2:], [tl, first[1] + x] + last[2:]).reshape(ny, nz) for x in xs]
    if len(ys) < ny:
        planes = [a[ys] for a in planes]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "p.npy" if world == 1 else f"p.rank{rank}.npy"), np.stack(planes).astype(np.float32))


def halo_check(capi, dist, rank, world, local, N, opts, seed=77, steps=3):
    """Cross-device correctness of the halo exchange at the bench's own geometry: a fresh multi-rank run of `steps`
    steps from global hash data; every rank then recomputes the 8 planes on its side of each x interface with a
    stand-alone single-rank solution over a 72-plane window of the SAME global data (shifted hash fill) and compares
    bit for bit.  After 3 steps a window plane is exact if it is >= 24 planes away from the window's ends."""
    import numpy as np
    import torch
    from yask_b200 import multi
    from yask_b200.synth import var_salt
    R, WIN, OFF = 8, 72, 32
    s = capi.Solution("iso3dfd")
    s.set_rank_domain_size_vec([N, N, N])
    s.set_num_ranks_vec([world, 1, 1])
    s.set_rank_index_vec([rank, 0, 0])
    for kv in opts:
        k, v = kv.split("=", 1)
        s.set_option(k, v)
    s.prepare_solution(local)
    multi.connect(s, dist, rank, world)
    p, v = s.get_var("p"), s.get_var("v")
    for t in (0, 1):
        p.fill_hash(t, seed, var_salt("p", t), -1.0, 1.0)
    v.fill_hash(0, seed, var_salt("v", 0), 0.05, 0.3)
    s.sync()
    dist.barrier()
    s.run_solution(0, steps - 1)
    s.sync()
    tl = p.get_last_valid_step_index()
    ok, checked = True, 0
    x0 = rank * N
    for side, present in (("lo", rank > 0), ("hi", rank < world - 1)):
        if not present:
            continue
        g_first = x0 if side == "lo" else x0 + N - R           # global index of my first compared plane
        w0 = g_first - OFF                                       # global index of the window's plane 0
        w = capi.Solution("iso3dfd")
        w.set_rank_domain_size_vec([WIN, N, N])
        for kv in opts:
            k, vv = kv.split("=", 1)
            w.set_option(k, vv)
        w.prepare_solution(local)
        wp, wv = w.get_var("p"), w.get_var("v")
        for t in (0, 1):
            wp.fill_hash(t, seed, var_salt("p", t), -1.0, 1.0, shift=[w0, 0, 0])
        wv.fill_hash(0, seed, var_salt("v", 0), 0.05, 0.3, shift=[w0, 0, 0])
        w.run_solution(0, steps - 1)
        w.sync()
        wl = wp.get_last_valid_step_index()
        ref = wp.get_elements_in_slice([wl, OFF, 0, 0], [wl, OFF + R - 1, N - 1, N - 1])
        got = p.get_elements_in_slice([tl, g_first, 0, 0], [tl, g_first + R - 1, N - 1, N - 1])
        ok = ok and bool(np.array_equal(got.view(np.uint32), ref.view(np.uint32)))
        checked += got.size
        w.close()
    s.close()
    tt = torch.tensor([1.0 if ok else 0.0, float(checked)], dtype=torch.float64, device="cuda")
    dist.all_reduce(tt[0:1], op=dist.ReduceOp.MIN)
    dist.all_reduce(tt[1:2], op=dist.ReduceOp.SUM)
    return {"result": "bit-exact" if tt[0].item() == 1.0 else "MISMATCH", "points_compared": int(tt[1].item()), "steps": steps,
            "what": "8 planes on each side of every x interface vs a stand-alone single-rank run on the same global hash data"}


def run_secondary(args, dist, rank, world, local, peak, want_cpu):
    """awp_elastic fp32 and ssg fp64 at size2^3 per GPU through the C ABI (same launcher, same ranks)."""
    import bench_stencils
    out = []
    for stencil, desc, bpp, dt in SECONDARY:
        try:
            r = bench_stencils.run(stencil, args.size2, 10, 3, 2, (), dist=dist)
        except Exception as e:
            out.append({"workload": f"{desc}, {args.size2}^3 per GPU", "error": repr(e)[:300]})
            continue
        ms = r["ms_per_step"]
        ach = bpp * args.size2 ** 3 / (ms * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "gen_traffic.json")))[stencil]["dram_bytes_per_step"]
        except Exception:
            pass
        rec = {"workload": f"{desc}, {args.size2}^3 points per GPU, rank grid {world}x1x1", "metric": "GPoints/s", "value": r["gpoints_per_s"],
               "unit": "GPoints/s", "n_gpus": world, "steps": r["steps"], "ms_per_step": ms, "dtype": dt, "scaling": "weak",
               "gpu_launches": r["kernel_launches"], "kernels": r.get("kernels"),
               "roofline": {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4), "traffic": traffic,
                            "algorithmic_bytes_per_point_step": bpp, "note": "both stages of one step; bytes = every var of each stage moved once (SURVEY.md 8d)"}}
        if want_cpu and rank == 0:
            try:
                rec["cpu_baseline"] = run_reference_cpu(stencil, args.size2, 4, budget_s=45.0)
            except Exception as e:
                rec["cpu_baseline"] = {"value": None, "kind": "unavailable", "sample": repr(e)[:200]}
        out.append(rec)
    if world == 1 and rank == 0:
        # temporal tile (north_star: "temporal tiling applies multiple time-steps inside shared memory where the radius allows"):
        # iso3dfd radius 2, one-step sweep against two steps per sweep, in a subprocess of its own
        for radius in (1, 2):
            try:
                r = subprocess.run([sys.executable, os.path.join(ROOT, "bench_temporal.py"), str(args.size), str(radius), "20"], capture_output=True, text=True, timeout=240)
                tl = json.loads(r.stdout.strip().splitlines()[-1])
                tt = tl["temporal_tile"]
                out.append({"workload": tl["workload"], "metric": "GPoints/s", "value": tt["gpoints_per_s"], "unit": "GPoints/s", "n_gpus": 1, "steps": tl["steps"],
                            "ms_per_step": tt["ms_per_step"], "dtype": "f32", "gpu_launches": tt["kernel_launches"],
                            "one_step_value": tl["one_step"]["gpoints_per_s"], "speedup_vs_one_step": tl["speedup"], "bit_identical_to_one_step": tl["bit_identical"],
                            "forms": tl.get("forms"),
                            "roofline": {"bound": "hbm", "achieved": tt["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": tt["frac"], "traffic": None,
                                         "algorithmic_bytes_per_point_step": 10, "frac_at_16B_per_point_step": tt["frac_16B"],
                                         "note": "20 B per point and PAIR of steps (p(t-1), p(t), v in; p(t+1), p(t+2) out); the one-step sweep moves 16 B per step"},
                            "one_step": tl["one_step"]})
            except Exception as e:
                out.append({"workload": f"iso3dfd radius {radius} fp32, temporal tile (2 steps per sweep)", "error": repr(e)[:300]})
    return out


def main_b200(args):
    import numpy as np
    import torch
    from yask_b200 import capi
    from yask_b200.synth import var_salt

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        # NCCL carries only the rendezvous, the barriers and the timing reductions (the data plane is peer stores over
        # NVLink, yb_halo.cu); its log level is whatever the caller set.
        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local)
    N = args.size
    K, W = args.steps, max(args.warmup, 3)

    s = capi.Solution("iso3dfd")
    s.set_rank_domain_size_vec([N, N, N])
    coupled = world > 1 and not args.replicas
    if coupled:
        s.set_num_ranks_vec([world, 1, 1])
        s.set_rank_index_vec([rank, 0, 0])
    for kv in args.opt:
        k, v = kv.split("=", 1)
        s.set_option(k, v)
    s.prepare_solution(local)
    if coupled:
        from yask_b200 import multi
        multi.connect(s, dist, rank, world)
    p, v = s.get_var("p"), s.get_var("v")
    seed = 2024
    for t in (0, 1):
        p.fill_hash(t, seed, var_salt("p", t), -1.0, 1.0)
    v.fill_hash(0, seed, var_salt("v", 0), 0.05, 0.3)
    s.sync()

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        if not dist:
            return list(vals)
        tt = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return tt.tolist()

    # ---- warm-up, then the timed region: exactly K steps --------------------------------------------
    s.run_solution(0, W - 1)
    barrier()
    s.clear_stats()
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.25)
    barrier()
    t0 = time.time()
    s.run_solution(W, W + K - 1)
    s.sync()
    barrier()
    t1 = time.time()
    st = s.get_stats()
    clk = clocks.window(t0, t1)
    own_dev_s = st.elapsed_secs
    dev_s, wall_s = max_over_ranks(own_dev_s, t1 - t0)           # CUDA events on the launching stream, max over ranks
    per_rank_ms = None
    if dist:
        tt = torch.zeros(world, dtype=torch.float64, device="cuda")
        tt[rank] = own_dev_s / K * 1e3
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        per_rank_ms = [round(x, 4) for x in tt.tolist()]
    launches = st.kernel_launches
    pts_per_gpu = N ** 3
    value = pts_per_gpu * world * K / dev_s / 1e9
    checksum = p.checksum(p.get_last_valid_step_index())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, p, rank, world)

    # ---- sustained: the same loop for >= 2 s (the part settles to its power-capped clock) ---------------
    sustained = None
    if not args.no_sustained:
        ks = max(K, int(2.2 / max(dev_s / K, 1e-6)))
        tl = p.get_last_valid_step_index()
        s.clear_stats()
        barrier()
        ts0 = time.time()
        s.run_solution(tl, tl + ks - 1)
        s.sync()
        barrier()
        ts1 = time.time()
        (sus_s,) = max_over_ranks(s.get_stats().elapsed_secs)
        sustained = {"value": round(pts_per_gpu * world * ks / sus_s / 1e9, 2), "unit": "GPoints/s", "steps": ks, "seconds": round(sus_s, 3),
                     "ms_per_step": round(sus_s / ks * 1e3, 4), "roofline_frac": None, "clocks": clocks.window(ts0, ts1)}
    clocks.stop()

    # ---- roofline of the dominant kernel (the point-update kernel: one launch per step per GPU) ------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    kern_ms = dev_s / K * 1e3                       # one sweep launch per step (multi-GPU: plus a one-thread halo wait kernel)
    achieved = BYTES_PER_POINT * pts_per_gpu / (kern_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "iso3dfd_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": traffic, "peak_source": peak_src, "kernel": "iso3dfd_tma2_kernel", "kernel_ms": round(kern_ms, 4),
                "algorithmic_bytes_per_launch": BYTES_PER_POINT * pts_per_gpu}
    if sustained:
        sustained["roofline_frac"] = round(BYTES_PER_POINT * pts_per_gpu / (sustained["ms_per_step"] * 1e-3) / 1e9 / peak, 4)

    # ---- e2e through the C ABI with host buffers ------------------------------------------------------
    e2e = None
    if not args.no_e2e:
      try:
            f0, l0 = p.halo_box(0)
            shape = [b - a + 1 for a, b in zip(f0[1:], l0[1:])]
            tl = p.get_last_valid_step_index()
            # host copies of the inputs in pinned memory (set-up, untimed): read back the synthetic fields
            hp = [torch.empty(shape, dtype=torch.float32, pin_memory=True) for _ in range(2)]
            hv = torch.empty([N, N, N], dtype=torch.float32, pin_memory=True)
            hout = torch.empty([N, N, N], dtype=torch.float32, pin_memory=True)
            import ctypes as C
            L = capi.lib()

            def get_into(var, tens, first, last):
                n = C.c_int64(0)
                capi._chk(L.yb_var_get_slice(s._h, var.index, C.c_void_p(tens.data_ptr()), capi._arr(first), capi._arr(last), C.byref(n)))

            def set_from(var, tens, first, last):
                n = C.c_int64(0)
                capi._chk(L.yb_var_set_slice(s._h, var.index, C.c_void_p(tens.data_ptr()), capi._arr(first), capi._arr(last), C.byref(n)))

            for i, t in enumerate((tl - 1, tl)):
                f, l = p.halo_box(t)
                get_into(p, hp[i], f, l)
            fv, lv = v.halo_box(0)
            get_into(v, hv, fv, lv)
            launches_before = s.get_stats().kernel_launches
            barrier()
            te0 = time.time()
            for i, t in enumerate((tl - 1, tl)):           # H2D: both step slots of p, and v
                f, l = p.halo_box(t)
                set_from(p, hp[i], f, l)
            set_from(v, hv, fv, lv)
            s.run_solution(tl, tl + K - 1)                   # K steps
            tl2 = p.get_last_valid_step_index()
            get_into(p, hout, *p.domain_box(tl2))            # D2H of the result (syncs)
            s.sync()
            barrier()
            te1 = time.time()
            (e2e_s,) = max_over_ranks(te1 - te0)
            h2d = (2 * hp[0].numel() + hv.numel()) * 4
            d2h = hout.numel() * 4
            e2e = {"value": round(pts_per_gpu * world * K / e2e_s / 1e9, 2), "unit": "GPoints/s", "h2d_bytes_per_step": h2d // K,
                   "d2h_bytes_per_step": d2h // K, "seconds": round(e2e_s, 4), "h2d_bytes_total_per_gpu": h2d, "d2h_bytes_total_per_gpu": d2h,
                   "gpu_launches": int(s.get_stats().kernel_launches - launches_before),
                   "note": "set_elements_in_slice(p t-1,t; v) from pinned host + run_solution(K) + get_elements_in_slice(p)"}
            del hp, hv, hout
      except Exception as ex:   # keep the bench line alive (e.g. pinned-memory limits on a shared host)
        e2e = {"value": None, "unit": "GPoints/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None, "error": repr(ex)[:200]}
    s.close()

    # ---- halo check (N > 1): real cross-device bit-exactness at the bench geometry -------------------------
    hc = None
    if dist and coupled and not args.no_halo_check:
        try:
            hc = halo_check(capi, dist, rank, world, local, N, args.opt)
        except Exception as ex:
            hc = {"result": "error", "error": repr(ex)[:300]}

    # ---- secondary workloads (BASELINE configs 3 and 5) -----------------------------------------------------
    secondary = None
    if not args.no_secondary:
        try:
            secondary = run_secondary(args, dist, rank, world, local, peak, want_cpu=(world == 1 and not args.no_cpu))
        except Exception as ex:
            secondary = [{"error": repr(ex)[:300]}]

    # ---- CPU baseline (rank 0, N=1 only) -----------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            cpu = run_reference_cpu("iso3dfd", 1024 if N >= 1024 else N, 10, budget_s=70.0)
        except Exception as e:  # keep the bench line alive
            cpu = {"value": None, "unit": "GPoints/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}

    if rank == 0:
        line = {"metric": f"GPoints/s, iso3dfd-16 fp32 {N}^3 per GPU", "value": round(value, 2), "unit": "GPoints/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": round(dev_s / K * 1e3, 4), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"iso3dfd radius 8 (16th order) fp32, {N}^3 points per GPU, rank grid {world}x1x1",
                           "fp_mode": "ref_gcc (bit-exact vs reference default build)", "l2": "inputs (13.5 GB/GPU) larger than L2; no flush needed",
                           "global_points": pts_per_gpu * world, "wall_ms_per_step": round(wall_s / K * 1e3, 4), "checksum": str(checksum),
                           "halo_exchange": ("none (1 rank)" if world == 1 else "none: independent replicas (diagnostic)" if not coupled else
                                             "boundary planes stored into the x neighbours' HBM by the sweep kernel's first work units, epoch "
                                             "published in-kernel, interior swept meanwhile; wait kernel in front of the next step")},
                "hbm_gbs_algorithmic": round(value * BYTES_PER_POINT, 1), "roofline": roofline, "sustained": sustained, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": int(launches), "clocks": clk}
        if per_rank_ms is not None:
            line["per_rank_ms_per_step"] = per_rank_ms
        if hc is not None:
            line["halo_check"] = hc["result"]
            line["halo_check_detail"] = hc
        if secondary is not None:
            line["secondary"] = secondary
        print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_b200(a)
