#!/usr/bin/env python
"""bench.py — particle-steps/s of the SPH step engine on synthetic Keplerian-disc ICs (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--particles P] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one body of the reference loop (SUMMER_SPH - Variable.f90:1120-1162): two full evaluations
(tree + density + EOS + gravity + sinks + SPH pairs), two half kicks, drift, dt ladder, h Newton-Raphson,
sink creation, accretion, bounds cull.  N = 1 workload: BASELINE.json configs[3] (Keplerian disc, 16M gas
particles + central sink, variable h, FP64).  Prints ONE JSON line (see README / DESIGN.md §Measurement); it is
the LAST line of stdout: with NCCL_DEBUG=VERSION in the environment (the GPU boxes set it) NCCL itself prints its
version banner on stdout once when the first communicator of a multi-rank run is created.

--impl reference times the CPU implementation of the same path (the oracle port of the Fortran loops —
no Fortran compiler exists in this image, so the reference itself cannot be built) on the host cores.

--dump-outputs DIR writes the state the last timed step handed back (what sph_download gives a caller) to DIR as
float64 .npy files: the ten gas columns on a fixed, seeded sample of rows, every sink, dt and t.  The ICs come from a
fixed seed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: the benchmark leaves nothing in it

import numpy as np  # noqa: E402

N_CONFIG5 = 64_000_000                  # BASELINE configs[4]
BYTES_PER_PARTICLE_STEP = 1960.0        # SURVEY.md §8(d): compulsory HBM bytes per particle-step
BYTES_SPH_PER_LAUNCH = 144.0            # SPH force pass, per particle per launch (SURVEY.md §8(d))
BYTES_DENSITY_PER_LAUNCH = 80.0
BYTES_GRAVITY_PER_LAUNCH = 120.0
FLOPS = {"density_candidate": 44, "sph_pair": 173, "grav_opened": 13, "grav_accepted": 35, "sink_gas": 20}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_ics(n):
    from summersph_b200 import ics
    b, s = ics.keplerian_disc(n, seed=20251018)
    return b, s


def cpu_reference_rate(n_sample, steps, warmup, threads, dump=None):
    """Oracle port timed on the host cores: particle-steps/s on a bounded disc sample."""
    from summersph_b200 import default_params, MODE_VARIABLE_H
    from oracle.oracle import Oracle
    p = default_params(MODE_VARIABLE_H)
    b, s = make_ics(n_sample)
    o = Oracle(p, threads=threads)
    o.upload(b, s)
    dt, t = 0.01, 0.0
    for _ in range(warmup):
        dt, t = o.step(dt, t)
    t0 = time.perf_counter()
    for _ in range(steps):
        dt, t = o.step(dt, t)
    el = time.perf_counter() - t0
    if dump:
        dump_outputs(dump, o, dt, t, 0)
    n, _ = o.sizes()
    return n * steps / el, el / steps


REF_THREADS = 16      # fixed, so that records taken on boxes with different core counts are comparable


def run_reference(args, rank):
    if rank != 0:
        return
    threads = min(REF_THREADS, os.cpu_count() or 1)
    n_sample = args.ref_particles
    rate, sec = cpu_reference_rate(n_sample, args.steps, args.warmup, threads, dump=args.dump_outputs)
    line = {
        "impl": "reference", "metric": "particle-steps/s", "value": rate, "unit": "particle-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"Keplerian disc {args.particles} gas + 1 sink, variable h (BASELINE configs[3]); each step timed on a {n_sample}-particle sample of it"},
        "cpu_baseline": {"value": rate, "unit": "particle-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{n_sample}-particle Keplerian disc, {args.steps} full steps, OpenMP on density/gravity/h-iteration/SPH loops; restatement, not gfortran (no Fortran compiler in the image)"},
        "e2e": {"value": rate, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def engine_for(p, local, rank, world):
    """Engine context + (world > 1) its own NCCL communicator, bootstrapped over torch.distributed."""
    from summersph_b200.engine import Engine
    e = Engine(p, device=local)
    if world > 1:
        from summersph_b200.parallel import init_comm, torch_broadcast_bytes
        init_comm(e, rank, world, torch_broadcast_bytes)
    return e


def multi_gpu_check(p, local, rank, world, dist, torch):
    """Untimed: a 60k disc with accretion and bounds removals, 3 loop bodies on all ranks (this run's multi-rank form:
    one process per GPU, NCCL, peer memory) and on a private single-rank context of rank 0; every rank compares."""
    from summersph_b200.state import GAS_FIELDS
    from summersph_b200.engine import Engine
    q = p.copy(bounding_size=95.0, sink_radius=12.0)
    res = {}
    for tag in ("multi", "single"):
        if tag == "single" and rank != 0:
            continue
        e = engine_for(q, local, rank, world) if tag == "multi" else Engine(q.copy(decomposition=0), device=local)
        e.ics_disc(60_000, seed=12)
        dt, t = 0.01, 0.0
        for _ in range(3):
            dt, t = e.step(dt, t)
        b, s = e.download()
        res[tag] = (dt, t, e.sizes(), b, s, e.state_hash()[0])
        e.close()
    out = None
    if rank == 0:
        (dt1, t1, sz1, b1, s1, h1), (dt0, t0, sz0, b0, s0, h0) = res["multi"], res["single"]
        dev = 0.0
        same = (dt1, t1, sz1) == (dt0, t0, sz0)
        if sz1 == sz0:
            for k in GAS_FIELDS:
                a, r = getattr(b1, k), getattr(b0, k)
                sc = np.maximum(np.abs(r), np.sqrt(np.mean(r * r)) + 1e-300)
                dev = max(dev, float(np.max(np.abs(a - r) / sc)))
        out = {"case": "60k disc, sink radius 12, bounding 95, 3 steps, ranks vs a private 1-rank context on rank 0",
               "bit_identical": bool(h1 == h0), "dt_t_sizes_equal": bool(same), "max_rel_dev": dev,
               "state_hash": f"{h1:016x}", "state_hash_1rank": f"{h0:016x}"}
    return out


def timed_run(e, n, steps, warmup, barrier, sampler=None, before=None):
    """warmup untimed steps, then `steps` timed steps on the engine's stream (CUDA events inside the engine)."""
    dt, t = 0.01, 0.0
    for _ in range(warmup):
        dt, t = e.step(dt, t)
    if before:
        before()                                 # untimed hook between warm-up and the timed region (--drift)
    stage_acc = {}
    barrier()
    if sampler:
        sampler.start()
    l0 = e.launch_count(); f0 = e.far_reuse_count()
    e.timer_start()
    for _ in range(steps):
        dt, t = e.step(dt, t)
        for k, v in e.stage_times().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
    ms = e.timer_stop()
    barrier()
    clocks = sampler.stop() if sampler else None
    stage_acc["_gravity_near_launches"] = e.far_reuse_count() - f0       # evaluations that kept the stored far sums (k_gravity_near instead of the full walk)
    return ms, stage_acc, e.launch_count() - l0, clocks, (dt, t)


DUMP_ROWS = 1 << 19          # sampled gas rows: 10 FP64 columns of them (40 MB) + their row numbers + the sinks stay under 64 MB
DUMP_SEED = 20251018


def dump_outputs(directory, e, dt, t, rank):
    """--dump-outputs: the state after the last timed step as float64 DIR/<name>.npy.  Gas columns on DUMP_ROWS rows drawn
    with a fixed seed (all rows when there are fewer; `rows` holds the row numbers), sink_<column> for every sink, dt_t."""
    from summersph_b200.state import GAS_FIELDS, SINK_FIELDS
    b, s = e.download()                          # under the domain decomposition a collective: every rank takes part
    if rank != 0:
        return
    n = len(b)
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))
    out = {"rows": rows, "dt_t": np.array([dt, t])}
    out.update({k: getattr(b, k)[rows] for k in GAS_FIELDS})
    out.update({"sink_" + k: getattr(s, k) for k in SINK_FIELDS})
    os.makedirs(directory, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(directory, k + ".npy"), np.asarray(v, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--particles", type=int, default=16_000_000)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--decomposition", type=int, default=None, help="multi-rank form: 1 = Morton domains + halo exchange (default for --gpus > 1), "
                    "0 = replicated state with Morton-sliced walks (bit-identical to one rank)")
    ap.add_argument("--ref-particles", type=int, default=1_000_000)
    ap.add_argument("--cpu-baseline-particles", type=int, default=100_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (large multi-GPU sizing runs)")
    ap.add_argument("--no-config5", action="store_true", help="skip the short 64M-particle sub-run (BASELINE configs[4])")
    ap.add_argument("--no-check", action="store_true", help="skip the untimed multi-rank vs single-rank comparison")
    ap.add_argument("--drift", action="store_true", help="add the energy / momentum / angular-momentum drift over the timed steps "
                    "(sph_conserved before and after them, outside the timed region) as a \"drift\" key (single rank / replicated form)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the state after the last timed step to DIR/<name>.npy (float64; gas rows sampled with a fixed seed)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from summersph_b200 import default_params, MODE_VARIABLE_H, Bodies, Sinks
    from summersph_b200.state import GAS_FIELDS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the SPH step)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    decomp = (1 if world > 1 else 0) if args.decomposition is None else (args.decomposition if world > 1 else 0)

    p = default_params(MODE_VARIABLE_H)
    p.n_ranks = world
    p.decomposition = decomp
    n = args.particles

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(v):
        tv = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        return float(tv.item())

    def allgather(v):
        tv = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world == 1:
            return [float(v)]
        out = [torch.zeros_like(tv) for _ in range(world)]
        dist.all_gather(out, tv)
        return [float(x.item()) for x in out]

    # ---- device-resident throughput ("value") ---------------------------------------------------------
    # The domain form stops collectively (same error on every rank from the same call) when a rank runs out of room or the
    # GPUs cannot map each other's memory; the line is then measured with the replicated form and says so ("fallback").
    cons = {}
    sampler = ClockSampler(local)                # every rank samples its own GPU; rank 0's record is the line's "clocks", the others' medians are listed beside it
    fallback = None
    for form in ([decomp, 0] if decomp == 1 else [decomp]):
        p.decomposition = form
        e = None; err = None
        try:
            check = multi_gpu_check(p, local, rank, world, dist, torch) if (world > 1 and not args.no_check) else None
            e = engine_for(p, local, rank, world)
            e.ics_disc(n, seed=20251018)         # generated on the device: every rank its own rows under the decomposition
            want_drift = args.drift and form == 0      # sph_conserved walks the single-rank / replicated tree
            ms, stage_acc, launches, clocks, (dt, t) = timed_run(e, n, args.steps, args.warmup, barrier, sampler,
                                                                 before=(lambda: cons.update(first=e.conserved())) if want_drift else None)
            near_launches = int(stage_acc.pop("_gravity_near_launches", 0))
        except Exception as ex:                  # noqa: BLE001 - reported in the line
            err = f"{type(ex).__name__}: {ex}"[:300]
        if allmax(1.0 if err else 0.0) == 0.0:
            decomp = form
            break
        if e is not None:
            e.close()
        if form == 0 or decomp == 0:
            raise SystemExit(f"bench: the engine failed: {err}")
        fallback = {"from": "Morton-ordered domains", "to": "replicated state", "reason": err or "a peer rank failed"}
        sampler = ClockSampler(local)
    per_rank = allgather(ms)
    per_rank_sm_mhz = allgather(float(clocks["sm_mhz"] or 0.0)) if clocks else None
    per_rank_walk = [v / args.steps for v in allgather(stage_acc.get("density", 0) + stage_acc.get("gravity", 0) + stage_acc.get("sph", 0))]
    per_rank_comm = [v / args.steps for v in allgather(sum(stage_acc.get(k, 0) for k in ("comm", "halo", "let", "migrate")))]
    per_rank_build = [v / args.steps for v in allgather(stage_acc.get("keys", 0) + stage_acc.get("sort", 0) + stage_acc.get("tree", 0))]
    ms = allmax(ms)
    value = n * args.steps / (ms * 1e-3)
    counters_exec = e.counters()                 # what the last timed step actually tested (exact-zero pairs culled before counting)
    dstats = e.domain_stats()
    dstats_all = {k: [int(x) for x in allgather(float(dstats[k]))] for k in ("own", "halo", "let_nodes")} if decomp else None
    state_hash, state_sums = e.state_hash()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, e, dt, t, rank)
    drift = None
    if want_drift:
        from summersph_b200._abi import drift_report
        drift = drift_report(cons["first"], e.conserved())
    # interaction counts of the reference algorithm (every leaf-box candidate): one untimed evaluation with exact
    # counters on the state the timed steps ended in
    e.set_exact_counters(True); e.evaluate(); counters = e.counters(); e.set_exact_counters(False)
    n_now, ns_now = e.sizes()

    # ---- end to end through the C-ABI with host buffers ("e2e") -----------------------------------------
    # The host owns the state between steps (what the Fortran loop does): every step uploads the state it got back from
    # the previous step, advances it and downloads the result.  Under the decomposition each rank moves only the rows it
    # owns (sph_upload_local / sph_download_local); in the replicated form every rank moves all rows.
    e2e_steps = 0 if args.no_e2e else args.steps
    e2e_value = None; h2d = d2h = 0; e2e_cold = None; resident_hits = None
    if e2e_steps:
        n_loc = e.local_size() if decomp else n_now
        capn = int(n_loc * 1.25) + 4096
        pin = {k: torch.empty(capn, dtype=torch.float64).pin_memory() for k in GAS_FIELDS}
        num = torch.empty(capn, dtype=torch.int32).pin_memory()
        hs = Sinks.empty(ns_now)
        def views(m):
            return Bodies(*[pin[k].numpy()[:m] for k in GAS_FIELDS])
        numbers = None
        if decomp:
            numbers, _ = e.download_local(into=views(n_loc)); num.numpy()[:n_loc] = numbers
            hs = e.sinks_only()
        else:
            e.download(into=(views(n_loc), hs))
        dt2, t2 = dt, t
        moved = 0
        # One host round trip per step.  1 rank: sph_step_host (upload + loop body + download in one call, copies under the
        # compute).  N ranks: sph_upload_local + sph_step + sph_download_local, every rank its own rows.  Two legs, each one
        # untimed round trip then e2e_steps timed ones: "cold" = every upload is taken as a new state
        # (sph_set_resident_check off); default = the context compares what it is handed with what it holds (bitwise, on the
        # device; domains agree through one all-reduce) and, when the host passes the state through unchanged, keeps its
        # tree and stored far-field sums.  The line's e2e is the default leg; the cold leg is in e2e.cold.
        def round_trip():
            nonlocal dt2, t2, n_loc, hs, numbers
            if world == 1:
                so = Sinks.empty(len(hs) + 8)
                dt2, t2, n_loc, ns2 = e.step_host(views(n_loc), hs, dt2, t2, into=(views(capn), so))
                hs = Sinks(*[getattr(so, k)[:ns2] for k in ("x", "y", "z", "vx", "vy", "vz", "m", "radius")])
                return
            if decomp:
                e.upload_local(n, views(n_loc), hs, numbers=num.numpy()[:n_loc])
            else:
                e.upload(views(n_loc), hs)
            dt2, t2 = e.step(dt2, t2)
            if decomp:
                n_loc = e.local_size()
                if n_loc > capn:
                    raise SystemExit("e2e: pinned buffers too small for this rank's rows")
                numbers, _ = e.download_local(into=views(n_loc)); num.numpy()[:n_loc] = numbers
                hs = e.sinks_only()
            else:
                n_loc = e.sizes()[0]
                hs = Sinks.empty(e.sizes()[1])
                e.download(into=(views(n_loc), hs))
        for leg in ("cold", "default"):
            e.set_resident_check(leg == "default")
            round_trip()
            h0 = e.resident_hits()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                round_trip()
                moved += n_loc if leg == "default" else 0
            barrier()
            sec = allmax(time.perf_counter() - t0)
            if leg == "cold":
                e2e_cold = {"value": n * e2e_steps / sec, "unit": "particle-steps/s", "ms_per_step": 1e3 * sec / e2e_steps,
                            "what": "the same calls with sph_set_resident_check(ctx, 0): every upload is a new state (tree rebuilt, both gravity evaluations walk the whole tree)"}
            else:
                resident_hits = e.resident_hits() - h0
        e2e_sec = sec                                 # the default leg
        e2e_value = n * e2e_steps / e2e_sec
        rows = sum(allgather(float(moved))) / e2e_steps            # rows moved per step, all ranks
        h2d = int(rows * (10 * 8 + (4 if decomp else 0)) + world * 8 * 8 * len(hs))
        d2h = h2d

    # ---- BASELINE configs[4]: the 64M-particle disc, a short run of the same engine (sub-record) ----------------
    config5 = None
    if not args.no_config5 and n != N_CONFIG5:
        e.close(); e = None
        torch.cuda.empty_cache()
        try:
            e5 = engine_for(p, local, rank, world)
            e5.ics_disc(N_CONFIG5, seed=20251018)
            ms5, st5, _, _, _ = timed_run(e5, N_CONFIG5, 2, 2, barrier)
            st5.pop("_gravity_near_launches", None)
            ms5 = allmax(ms5)
            h5, sums5 = e5.state_hash()
            config5 = {"workload": f"Keplerian disc {N_CONFIG5} gas + 1 sink (BASELINE configs[4])", "particles": N_CONFIG5, "n_gpus": world, "steps": 2, "warmup": 2,
                       "ms_per_step": ms5 / 2, "value": N_CONFIG5 * 2 / (ms5 * 1e-3), "unit": "particle-steps/s",
                       "stage_ms_per_step": {k: v / 2 for k, v in st5.items()}, "state_sums": sums5,
                       "domain_stats": e5.domain_stats() if decomp else None}
            e5.close()
        except Exception as ex:                  # never lose the main line to the sub-run
            config5 = {"error": str(ex)[:300]}

    if rank == 0:
        peaks, peak_src = measured_peaks()
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        per_launch = {"sph": (BYTES_SPH_PER_LAUNCH, "k_force"), "density": (BYTES_DENSITY_PER_LAUNCH, "k_density"), "gravity": (BYTES_GRAVITY_PER_LAUNCH, "k_gravity")}
        dom = max(per_launch, key=lambda k: stage_acc.get(k, 0.0))
        # launches of the dominant kernel in the timed region: two per step, except that a gravity evaluation on the stored
        # far sums (evaluation A of a step that follows a step without removals) is k_gravity_near, timed apart ("gravity_near")
        dom_launches = 2 * args.steps - (near_launches if dom == "gravity" else 0)
        dom_ms = stage_acc[dom] / max(dom_launches, 1)
        achieved = per_launch[dom][0] * (n / world) / (dom_ms * 1e-3) / 1e9       # one rank's launch processes n / world targets
        traffic = None; traffic_note = "no ncu capture at this particle count in profiles/"
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2b_traffic.json")))
            if int(tr["particles"]) == n and world == 1:
                traffic = tr["dram_bytes_per_launch"][per_launch[dom][1]]; traffic_note = tr.get("note", "")
        except Exception:
            pass
        if e is None:
            from summersph_b200.engine import Engine
            e = Engine(p.copy(decomposition=0), device=local)
        fp64_one = e.fp64_peak()
        fp64_peak = fp64_one * world
        def flops(c):
            return (c["density_candidates"] * FLOPS["density_candidate"] + c["sph_pairs"] * FLOPS["sph_pair"]
                    + c["grav_opened"] * FLOPS["grav_opened"] + c["grav_accepted"] * FLOPS["grav_accepted"] + n * ns_now * FLOPS["sink_gas"])
        step_flops = 2.0 * flops(counters)
        grav_flops_exec = counters_exec["grav_opened"] * FLOPS["grav_opened"] + counters_exec["grav_accepted"] * FLOPS["grav_accepted"] + n * ns_now * FLOPS["sink_gas"]
        step_flops_exec = 2.0 * flops(counters_exec) - grav_flops_exec * near_launches / args.steps      # evaluations on the stored far sums execute only the near pairs (not counted)
        dom_flops = {"gravity": counters["grav_opened"] * FLOPS["grav_opened"] + counters["grav_accepted"] * FLOPS["grav_accepted"] + n * ns_now * FLOPS["sink_gas"],
                     "sph": counters["sph_pairs"] * FLOPS["sph_pair"], "density": counters["density_candidates"] * FLOPS["density_candidate"]}[dom]
        dom_tflops = dom_flops / world / (dom_ms * 1e-3) / 1e12
        sec = ms / args.steps * 1e-3
        line = {
            "metric": "particle-steps/s", "value": value, "unit": "particle-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"Keplerian disc {n} gas + 1 central sink, variable h, eta 1.2, theta 0.5 (BASELINE configs[3])",
                       "particles": n, "mode": "variable_h",
                       "parallelism": f"{world} rank(s)" + ("" if world == 1 else (", Morton-ordered domains + halo exchange + top-tree all-gather" if decomp else ", replicated state + Morton-sliced walks")),
                       "ics": "generated on the device (sph_ics_disc, counter-based, seed 20251018)",
                       "l2": "inputs (>=1.3 GB state + tree) exceed the 126 MB L2; no flush needed"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "particle-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "resident_hits": resident_hits, "cold": e2e_cold, "what": ("sph_upload_local + sph_step + sph_download_local per step: every rank moves the rows it owns (pinned host SoA + their numbers); the ranks recognise the state they are handed back (bitwise comparison on the device, one all-reduce) and keep tree, halo selection and far-field sums; one untimed round trip before the timed ones" if decomp else
                                                 ("sph_step_host per step: upload (pinned host SoA) + one loop body + download (ascending number order) in one call, the copies under the compute; the context recognises the state it is handed back (bitwise comparison on the device) and keeps its tree and far-field sums; one untimed call before the timed ones" if world == 1 else
                                                  "sph_upload (pinned host SoA) + sph_step + sph_download (ascending number order) per step"))},
            "gpu_launches": launches,
            "gravity_far_reuse": {"near_only_evaluations": near_launches, "of": 2 * args.steps,
                                  "what": "evaluation A of a step sees the positions, tree and sinks of the step before (F:894 after F:905-912): it keeps that evaluation's far-field sums "
                                          "and re-evaluates the recorded near pairs with the new h (k_gravity_near, stage gravity_near); same terms as a full walk, summed in another order"},
            "roofline": {"bound": "fp64", "kernel": per_launch[dom][1], "achieved": dom_tflops, "peak": fp64_one, "unit": "TFLOP/s", "frac": dom_tflops / fp64_one,
                         "peak_source": "in-library FP64 FMA probe (sph_fp64_peak) run at the end of this process; MEASURED_PEAKS.json holds no FP64 figure",
                         "launch_ms": dom_ms, "launches": dom_launches, "algorithmic_flops_per_launch": dom_flops / world,
                         "hbm": {"achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "peak_source": peak_src,
                                 "algorithmic_bytes_per_particle_per_launch": per_launch[dom][0]},
                         "traffic": traffic, "traffic_note": traffic_note,
                         "note": "the walk kernels re-read their sources from L1 / L2 / shared memory: the FP64 pipe binds, the HBM fraction is given beside it (SURVEY.md 8(d))"},
            "fp64": {"achieved_tflops": step_flops / sec / 1e12, "peak_tflops": fp64_peak, "frac": step_flops / sec / 1e12 / fp64_peak,
                     "algorithmic_flops_per_step": step_flops,
                     "executed": {"flops_per_step": step_flops_exec, "achieved_tflops": step_flops_exec / sec / 1e12, "frac": step_flops_exec / sec / 1e12 / fp64_peak,
                                  "what": "the same per-interaction flop counts on the pairs the timed kernels actually tested (exact-zero pairs are culled before any FP64 work; a gravity evaluation that kept the stored far sums counts as zero)"},
                     "how": "reference-expression flop counts x interaction counters (SURVEY.md 8(d)): 44 per density candidate, 173 per unordered pair, 13 / 35 per opened / accepted node, 20 per sink-gas pair"},
            "hbm_step": {"achieved": BYTES_PER_PARTICLE_STEP * n / sec / 1e9, "peak": hbm_peak * world,
                         "frac": BYTES_PER_PARTICLE_STEP * n / sec / 1e9 / (hbm_peak * world), "unit": "GB/s"},
            "stage_ms_per_step": {k: v / args.steps for k, v in stage_acc.items()},
            "per_rank_ms_per_step": [v / args.steps for v in per_rank],
            "counters": counters, "counters_executed": counters_exec,
            "state_hash": f"{state_hash:016x}", "state_sums": state_sums,
        }
        if world > 1:
            line["per_rank_sm_mhz"] = per_rank_sm_mhz
            line["per_rank_walk_ms_per_step"] = per_rank_walk
            line["per_rank_comm_ms_per_step"] = per_rank_comm
            line["per_rank_build_ms_per_step"] = per_rank_build
            line["multi_gpu_check"] = check
            if fallback:
                line["fallback"] = fallback
            if dstats_all:
                line["domain_stats"] = dstats_all
        if drift is not None:
            line["drift"] = dict(drift, over_steps=args.steps)
        if config5 is not None:
            line["config5"] = config5
        if not args.no_cpu_baseline and world == 1:
            threads = min(REF_THREADS, os.cpu_count() or 1)
            nb = args.cpu_baseline_particles
            rate, sec_c = cpu_reference_rate(nb, 1, 0, threads)
            line["cpu_baseline"] = {"value": rate, "unit": "particle-steps/s", "cores": threads, "kind": "port",
                                    "sample": f"{nb}-particle Keplerian disc (same parameters), 1 full step, oracle port with OpenMP; restatement, not gfortran (no Fortran compiler on the box: profiles/r2_fortran_probe_gpubox.log)"}
        print(json.dumps(line), flush=True)
    if e is not None:
        e.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
