#!/usr/bin/env python
"""bench.py — dispatch decisions/sec (policy-eval + route), BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)

Workload (config.workload): BASELINE config 3 — 1,000,000 jobs x 4,096 rules x 65,536 workers
(seeded synthetic, cordum_b200/synth.py "c3").  At N > 1 the same 1M jobs are sharded
contiguously by job index across the N ranks (config 4, strong scaling); every rank holds the
full rule / routing / worker tables.

One step = one pass of the hot path over the rank's job shard:
    ingest the heartbeat load deltas of this rank's W/N worker slice (pinned host -> HBM)
    [N > 1]  one NCCL all-gather of the per-rank 16 B/worker load slices   (SURVEY §8e)
    worker_chunk_kernel + worker_merge_kernel   (load score / overload / per-pool sorted views, label bitmaps and
                                                 single-label answers over the 64k workers)
    policy_kernel        (first-match over the rule set + decision mapping; overlaps the two lines above)
    route_kernel         (pool filter + least-loaded pick for the jobs that may dispatch)
`value`  : job columns already resident in HBM; K steps bracketed by barrier + synchronize on
           both sides, max over ranks.  Successive steps rotate over enough distinct resident
           copies of the shard that the working set exceeds 2 x L2 (no step re-reads L2-hot columns).
`e2e`    : the same decisions produced through the public C ABI from HOST buffers: string-level
           job envelopes (per-job strings, nothing interned) in page-locked memory -> H2D of the envelope
           bytes -> cordum_encode_device (dictionary coding + topic sort on the GPU) -> kernels ->
           D2H of the decision records, every step, two batches in flight.  `e2e.host_encoder` reports
           the same path through cordum_encode (host threads) beside it.
`roofline`: policy_kernel's (the dominant kernel) algorithmic bytes per launch / its CUDA-event duration, against the
           measured HBM copy bandwidth in MEASURED_PEAKS.json.
`cpu_baseline` / --impl reference: the oracle (C++ port of the reference's Go path, oracle/oracle.cpp)
           timed on the box's usable host cores (affinity and cgroup quota, cordum_b200/hostinfo.py).
`parity_check`: untimed; every record of every rank's shard against the oracle, mismatches all-reduced.

--dump-outputs DIR: after the timed steps, the decision records of the last timed step (what a caller of
           cordum_batch_fetch receives for that batch) are written as DIR/<field>.npy, one array per record field in job
           order (DIR/<field>.rank<r>.npy per rank at N > 1).  The inputs are seeded, so two builds run with the same
           arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # a benchmark run leaves the source tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "dispatch decisions/sec (policy-eval+route)"
UNIT = "decisions/s"
L2_BYTES = 126 << 20
DECISION_FIELDS = ("decision", "sched_decision", "flags", "route_status", "reason_code", "rule_idx", "worker_slot")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump_outputs(out_dir: str, rec: np.ndarray, rank: int, world: int):
    """One .npy per decision-record field.  The u8 fields are exact in float32; rule_idx and worker_slot (int32) go out
    as float64 so that no value is rounded.  At 1M jobs: 5 x 4 MB + 2 x 8 MB."""
    os.makedirs(out_dir, exist_ok=True)
    suffix = ".rank%d" % rank if world > 1 else ""
    for f in DECISION_FIELDS:
        a = rec[f]
        np.save(os.path.join(out_dir, f + suffix + ".npy"), a.astype(np.float32 if a.dtype.itemsize == 1 else np.float64))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 50 ms from the start of the timed region to the end of the
    measurement loops (throughput, per-kernel, end-to-end)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)   # no sampler outlives the run: --value-only and failed checks never reach stop()
        except OSError:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU path (oracle)
def cpu_reference_rate(cfg, threads: int, target_s: float, first: int = 0):
    """Times the oracle on a bounded, contiguous sample of cfg.jobs.  Returns (decisions/s, sample, seconds)."""
    import oracle_lib
    from cordum_b200 import wire

    o = oracle_lib.Oracle(cfg.policy, cfg.routing, cfg.workers)
    n = cfg.jobs.n_jobs
    probe = min(n, max(4096, 64 * threads))   # large enough that thread start-up does not skew the estimate
    t0 = time.perf_counter()
    o.eval(cfg.jobs, wire.MODE_POLICY_AND_ROUTE, threads=threads, first=first % max(1, n - probe), count=probe)
    dt = max(time.perf_counter() - t0, 1e-6)
    sample = int(min(n, max(probe, probe / dt * target_s)))
    start = first % max(1, n - sample + 1)
    t0 = time.perf_counter()
    o.eval(cfg.jobs, wire.MODE_POLICY_AND_ROUTE, threads=threads, first=start, count=sample)
    dt = time.perf_counter() - t0
    o.close()
    return sample / dt, sample, dt


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    from cordum_b200 import synth

    from cordum_b200 import hostinfo

    threads = hostinfo.usable_cores()   # affinity and cgroup quota, not os.cpu_count()
    cfg = synth.make_config("c3")
    per_step_s = max(0.5, min(6.0, 150.0 / max(1, args.steps + args.warmup)))
    for w in range(args.warmup):
        cpu_reference_rate(cfg, threads, per_step_s, first=w * 50_000)
    total_jobs, total_s, sample = 0, 0.0, 0
    for k in range(args.steps):
        rate, sample, dt = cpu_reference_rate(cfg, threads, per_step_s, first=(args.warmup + k) * 50_000)
        total_jobs += sample
        total_s += dt
    value = total_jobs / total_s
    desc = "%d steps x ~%d contiguous jobs of the 1M-job c3 batch (about %.1f s each); full 4096-rule set and 65536-worker table" % (
        args.steps, sample, per_step_s)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * total_s / max(1, args.steps), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64 bitmask + f32 score", "data": "synthetic",
        "config": {"workload": "c3: 1,000,000 jobs x 4096 rules x 65536 workers (seed 3), policy+route",
                   "note": "reference CPU path = oracle/oracle.cpp (C++ restatement of the Go evaluator; the Go "
                           "toolchain and the CAP module are absent), one std::thread per host core"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc,
                         "host": hostinfo.describe()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- CUDA path
def run_cuda(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist

    from cordum_b200 import engine, shard, synth, wire

    torch.cuda.set_device(local_rank)
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"   # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = synth.make_config("c3")
    J, W = cfg.jobs.n_jobs, cfg.workers.n_workers
    j0, j1 = shard.job_range(rank, world, J)
    my_jobs = cfg.jobs.slice(j0, j1 - j0) if world > 1 else cfg.jobs
    n_shard = my_jobs.n_jobs
    w0, w1 = shard.worker_range(rank, world, W)
    assert shard.padded_workers(world, W) == W, "worker count must divide evenly for the all-gather"

    eng = engine.Engine(device=local_rank)
    eng.load_policy(cfg.policy, "bench")
    eng.load_routing(cfg.routing)
    eng.load_workers(cfg.workers)
    st = eng.stats()
    in_b, out_b = st.job_in_bytes, st.job_out_bytes
    table_bytes = int(st.passrow_bytes + st.rulecol_bytes + st.routing_bytes + st.worker_bytes)

    # resident copies of the shard: enough distinct addresses that successive steps cannot hit L2
    shard_bytes = n_shard * (in_b + out_b)
    n_rot = max(2, int(np.ceil(2.0 * L2_BYTES / max(1, shard_bytes))) + 1)
    if args.step == "tick":
        n_rot = (n_rot + 5) // 6 * 6   # tick graphs are cached per (batch pair, tick phase of 6): a multiple of 6 keeps them to n_rot
    batches = [eng.batch(n_shard) for _ in range(n_rot)]
    t_enc0 = time.perf_counter()
    for b in batches:
        b.encode(my_jobs)
        b.dispatch(wire.MODE_POLICY_AND_ROUTE)   # makes the columns resident (and warms the dictionaries)
    enc_s = (time.perf_counter() - t_enc0) / n_rot
    ref_result = batches[0].results().copy()

    # per-step heartbeat deltas for this rank's worker slice (synthetic, seeded per step)
    base = cfg.workers.loads()
    n_delta_sets = 8
    rng = np.random.default_rng(1000 + rank)
    delta_sets = []
    for s in range(n_delta_sets):
        d = base[w0:w1].copy()
        d["active_jobs"] = rng.integers(0, 9, w1 - w0)
        d["cpu_load"] = (rng.random(w1 - w0) * 100).astype(np.float32)
        d["gpu_utilization"] = (rng.random(w1 - w0) * 100).astype(np.float32)
        delta_sets.append(torch.from_numpy(d.view(np.uint8).reshape(-1, 16).copy()).pin_memory())
    stream = torch.cuda.current_stream()
    if world > 1 and args.exchange == "peer":
        # peer-memory heartbeat exchange: every rank maps every other rank's slice buffer (CUDA IPC over NVLink); both
        # cordum_workers_ingest and cordum_tick_async gather through it, no collective library on the path
        handles = [None] * world
        dist.all_gather_object(handles, eng.peer_export(rank, world))
        eng.peer_import(handles)
        dist.barrier()
    if args.exchange == "nccl":
        # the engine's own NCCL communicator (cordum_exchange_init): all-gather of the slices in cordum_workers_ingest
        if world > 1:
            ok = 1
            try:
                box = [engine.Engine.exchange_unique_id() if rank == 0 else None]
            except Exception as ex:   # libnccl not loadable from the engine: every rank falls back together
                print("engine exchange unavailable (%s): using torch.distributed" % ex, file=sys.stderr)
                box, ok = [None], 0
            flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
            dist.broadcast(flag, src=0)
            if int(flag.item()):
                dist.broadcast_object_list(box, src=0)
                eng.exchange_init(box[0], rank, world)
            else:
                args.exchange = "torch"
    if args.exchange == "torch":
        send = torch.empty((w1 - w0, 16), dtype=torch.uint8, device="cuda")
        recv = [torch.empty((W, 16), dtype=torch.uint8, device="cuda") for _ in range(2)]

    use_ticks = args.step == "tick"
    if use_ticks and world > 1:
        assert args.exchange == "peer", "ticks gather over peer memory"

    def step(k: int, batch, resident: bool):
        if use_ticks and resident:
            # one graph launch: heartbeat epoch k (peer gather + refresh) || policy of this batch || route of the previous one
            batch.tick(delta_sets[k % n_delta_sets].data_ptr(), w0, w1 - w0)
            return
        if args.exchange in ("peer", "nccl"):
            # heartbeat ingest: pinned host -> HBM, gather of the per-rank slices (peer memory / NCCL, SURVEY §8e), refresh
            eng.ingest(delta_sets[k % n_delta_sets].data_ptr(), w0, w1 - w0)
        else:
            send.copy_(delta_sets[k % n_delta_sets], non_blocking=True)
            buf = shard.gather_loads(send, out=recv[k % 2]) if world > 1 else send   # torch.distributed all-gather
            eng.set_loads_device(buf.data_ptr(), W, stream.cuda_stream)
        if resident:
            batch.dispatch_resident_async(wire.MODE_POLICY_AND_ROUTE | wire.FLAG_NO_TIMING)
        else:
            batch.dispatch_async(wire.MODE_POLICY_AND_ROUTE)

    def sync_all():
        for b in batches:
            b.wait()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------------------------------------------------------- device-resident: `value`
    if use_ticks:
        for k in range(n_rot + 6):      # untimed: every (batch pair, phase) tick graph is captured here
            step(k, batches[k % n_rot], True)
        sync_all()
    for k in range(args.warmup):
        step(k, batches[k % n_rot], True)
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count()
    # Device time: a CUDA event on the ingest stream before the first step and one after every batch stream has been
    # joined into it (the kernels run on per-batch streams); the wall clock between the synchronizes is kept beside it.
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ext = [torch.cuda.ExternalStream(b.stream, device=torch.device("cuda", local_rank)) for b in batches]
    t0 = time.perf_counter()
    if use_ticks:
        # every tick is one graph launch on the engine's tick stream: the events go on that stream
        tstream = torch.cuda.ExternalStream(eng.tick_stream, device=torch.device("cuda", local_rank))
        ev_a.record(tstream)
        for k in range(args.steps):
            step(args.warmup + k, batches[(args.warmup + k) % n_rot], True)
        eng.tick_flush()             # the route of the last batch
        ev_b.record(tstream)
    else:
        ev_a.record(stream)
        for k in range(args.steps):
            step(args.warmup + k, batches[(args.warmup + k) % n_rot], True)
        for x in ext:
            stream.wait_stream(x)
        ev_b.record(stream)
    sync_all()
    wall = time.perf_counter() - t0
    elapsed = ev_a.elapsed_time(ev_b) * 1e-3
    launches = eng.launch_count() - launches0
    if world > 1:
        t = torch.tensor([elapsed, wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed, wall = (float(x) for x in t.tolist())
    value = J * args.steps / elapsed

    # parity spot check inside the bench: the last resident run must equal the first copy run's records
    # (same jobs; only the load table changed, so compare policy fields)
    chk = batches[(args.warmup + args.steps - 1) % n_rot].fetch()
    assert np.array_equal(chk["decision"], ref_result["decision"]) and np.array_equal(chk["rule_idx"], ref_result["rule_idx"])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, chk, rank, world)   # before the parity epoch below overwrites batches[0]'s records

    # parity of the sharded path, exchange included: one more epoch with a known delta set, then EVERY rank compares
    # EVERY record of its shard with the oracle evaluated on the table all ranks' slices add up to (checker only,
    # untimed; the mismatch count is summed over ranks into the JSON line).  At N=1 the same oracle pass over the full
    # 1M-job batch is also the cpu_baseline measurement.
    from cordum_b200 import hostinfo
    import oracle_lib

    k_chk = 3
    step(k_chk, batches[0], True)
    sync_all()
    full = base.copy()
    for r in range(world):
        r0, r1 = shard.worker_range(r, world, W)
        rr = np.random.default_rng(1000 + r)
        for s_ in range(k_chk % n_delta_sets + 1):   # replay rank r's generator up to the set in use
            act = rr.integers(0, 9, r1 - r0)
            cpu_ = (rr.random(r1 - r0) * 100).astype(np.float32)
            gpu_ = (rr.random(r1 - r0) * 100).astype(np.float32)
        full["active_jobs"][r0:r1] = act
        full["cpu_load"][r0:r1] = cpu_
        full["gpu_utilization"][r0:r1] = gpu_
    cores = hostinfo.usable_cores()
    o_threads = max(1, cores // world)
    n_chk = n_shard if not args.parity_sample else min(args.parity_sample, n_shard)
    o = oracle_lib.Oracle(cfg.policy, cfg.routing, cfg.workers)
    o.update_workers(np.arange(W, dtype=np.uint32), full)
    t_or = time.perf_counter()
    want = o.eval(my_jobs, wire.MODE_POLICY_AND_ROUTE, threads=o_threads, first=0, count=n_chk)
    oracle_s = time.perf_counter() - t_or
    o.close()
    got = batches[0].fetch()[:n_chk]
    fields = DECISION_FIELDS
    bad_rows = np.zeros(n_chk, dtype=bool)
    for f in fields:
        bad_rows |= got[f] != want[f]
    counts = torch.tensor([int(bad_rows.sum()), int(n_chk)], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    n_bad, n_checked = (int(x) for x in counts.tolist())
    parity = {"jobs_checked": n_checked, "mismatches": n_bad, "fields": list(fields), "ok": n_bad == 0,
              "ranks_checked": world, "oracle_threads_per_rank": o_threads, "oracle_s": oracle_s}
    assert n_bad == 0, "sharded path differs from the oracle on %d of %d jobs" % (n_bad, n_checked)

    if args.value_only:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "ms_per_step": 1000.0 * elapsed / args.steps,
                              "wall_ms_per_step": 1000.0 * wall / args.steps, "step_mode": "tick" if use_ticks else "streams", "parity_check": parity,
                              "gpu_launches": int(launches)}), flush=True)
        for b in batches:
            b.free()
        eng.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------------------------------------------------------- per-kernel durations for the roofline
    # Serialized launches (wait after every step) so the CUDA-event span of a kernel contains that kernel only;
    # in the throughput loop above policy_kernel overlaps the previous step's route_kernel / worker_chunk_kernel + worker_merge_kernel.
    pol_ms, rte_ms = [], []
    step(0, batches[0], True)          # one more heartbeat epoch, then hold the worker tables still so that
    sync_all()                         # route_kernel's event span does not contain a wait for worker_chunk_kernel + worker_merge_kernel
    for k in range(max(8, min(args.steps, 16))):
        b = batches[k % n_rot]
        b.dispatch_resident(wire.MODE_POLICY_AND_ROUTE)
        if k >= 2:
            p_, r_ = b.kernel_times()
            pol_ms.append(p_)
            rte_ms.append(r_)
    sync_all()

    # ---------------------------------------------------------------- end to end: `e2e`
    # Input = string-level envelopes in host memory where NOTHING is shared between jobs: every job's strings are laid out
    # contiguously, job after job, as a shim unpacking protobuf JobRequests would leave them (wire.EnvelopeBatch.deinterned).
    # The variant with an interned arena (equal strings share one span, which lets the encoder resolve values by address)
    # is measured beside it and reported as `interned_arena`.
    e2e_steps = max(4, min(args.steps, 12))
    plain_jobs = my_jobs.deinterned()
    pinned = [eng.pinned_envelopes(plain_jobs) for _ in range(2)]   # what a shim would unpack its requests into
    env_bytes = int(len(plain_jobs.arena) + sum(v.nbytes for v in plain_jobs.cols.values()))

    def e2e_run(jobs_in, device: bool):
        """jobs_in: one envelope set per in-flight batch.  device: cordum_encode_device (envelope bytes -> GPU, encoded
        there) or cordum_encode (host threads) + H2D of the records."""
        def enc(b, k):
            if device:
                b.encode_device(jobs_in[k % 2])
            else:
                b.encode(jobs_in[k % 2])
        for k in range(2):
            enc(batches[k % 2], k)
            step(k, batches[k % 2], False)
        sync_all()
        t0 = time.perf_counter()
        enc_t = []
        for k in range(e2e_steps):
            b = batches[k % 2]
            te = time.perf_counter()
            enc(b, k)                          # waits for this batch's previous run first
            enc_t.append((time.perf_counter() - te) * 1e3)
            step(k, b, False)                  # [H2D records +] kernels + D2H decisions, async
        sync_all()
        return time.perf_counter() - t0, enc_t

    def same_decisions(b):
        r = b.results()
        return np.array_equal(r["decision"], ref_result["decision"]) and np.array_equal(r["rule_idx"], ref_result["rule_idx"])

    fb0 = eng.host_fallbacks()
    e2e_elapsed, enc_ms = e2e_run(pinned, True)
    assert same_decisions(batches[(e2e_steps - 1) % 2]), "device-encoded envelopes give different decisions"
    e2e_fallbacks = eng.host_fallbacks() - fb0
    log("e2e per-step encode_device enqueue(+wait) ms:", " ".join("%.1f" % x for x in enc_ms))
    e2e_host_elapsed, enc_host_ms = e2e_run([plain_jobs, plain_jobs], False)
    assert same_decisions(batches[(e2e_steps - 1) % 2]), "the de-interned envelopes encode to different decisions"
    log("e2e per-step host encode(+wait) ms, de-interned arena:", " ".join("%.1f" % x for x in enc_host_ms))
    e2e_int_elapsed, enc_int_ms = e2e_run([my_jobs, my_jobs], False)
    log("e2e per-step host encode(+wait) ms, interned arena:   ", " ".join("%.1f" % x for x in enc_int_ms))
    for b in batches[:2]:
        b.encode(my_jobs)                      # leave host-encoded records behind for the records-only loop below
    # from already-encoded pinned records (copies + kernels only)
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        step(k, batches[k % 2], False)
    sync_all()
    e2e_cols_elapsed = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_elapsed, e2e_cols_elapsed, e2e_int_elapsed, e2e_host_elapsed], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_elapsed, e2e_cols_elapsed, e2e_int_elapsed, e2e_host_elapsed = (float(x) for x in t.tolist())
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        return

    peak, peak_src = measured_peaks()
    # Dominant kernel = policy_kernel.  Its algorithmic bytes per job: the 64 B policy record it reads + the 16 B decision
    # record it writes + 8 B per dispatchable job into the route list (counted as 8 B for every job: an upper bound on
    # what it may write), plus the policy tables once per launch.
    pol_job_bytes = 64 + out_b + 8
    pol_tables = int(st.passrow_bytes + st.rulecol_bytes)
    algo_bytes = n_shard * pol_job_bytes + pol_tables
    k_ms = float(np.mean(pol_ms))
    r_ms = float(np.mean(rte_ms))
    achieved = algo_bytes / (k_ms * 1e-3) / 1e9
    # whole path: 96 B of records in (64 B policy + 32 B routing), 16 B out, the 8 B route-list entry written and read
    path_bytes = n_shard * (in_b + out_b + 16) + table_bytes
    path_gbs = path_bytes / ((k_ms + r_ms) * 1e-3) / 1e9
    # SURVEY.md §8(d) fixes 100 B per decision (84 B of attribute columns + the 16 B record) + the tables once per batch
    s8d_bytes = n_shard * 100 + table_bytes
    s8d_gbs = s8d_bytes / ((k_ms + r_ms) * 1e-3) / 1e9
    traffic = None
    traffic_note = None
    tp = os.path.join(ROOT, "profiles", "policy_kernel_traffic.json")
    if os.path.exists(tp) and world == 1:   # from the ncu --set full capture of this kernel (tools/ncu_metrics.py); the
        with open(tp) as f:                  # file names the commit it was taken at, so a stale number is visible
            tj = json.load(f)
        traffic, traffic_note = tj.get("dram_bytes_per_launch"), tj.get("source")

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        # the parity pass above ran the oracle over the whole 1M-job batch on all usable host cores: that IS the CPU
        # path on this workload (no sampling, no extrapolation)
        cpu = {"value": n_chk / oracle_s, "unit": UNIT, "cores": o_threads, "kind": "port",
               "sample": "all %d jobs of the c3 batch in %.1f s, full rule set and worker table; oracle/oracle.cpp, "
                         "one std::thread per usable host core" % (n_chk, oracle_s),
               "host": hostinfo.describe()}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * elapsed / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64 bitmask + f32 score", "data": "synthetic",
        "timing": {"clock": "CUDA events (first ingest -> all batch streams joined), max over ranks",
                   "wall_ms_per_step": 1000.0 * wall / args.steps},
        "config": {"workload": "c3: 1,000,000 jobs x 4096 rules x 65536 workers (seed 3), policy+route",
                   "jobs_per_rank": n_shard, "parallelism": "jobs sharded by index x%d, tables replicated" % world,
                   "l2": "inputs larger than L2: steps rotate over %d resident copies of the shard (%.0f MB total)" % (
                       n_rot, n_rot * shard_bytes / 1e6),
                   "step": ("one CUDA-graph tick: [heartbeat-slice H2D + %sworker_chunk/merge] || policy_kernel(batch k) || route_kernel(batch k-1)" % (
                       "peer-memory gather over NVLink + " if world > 1 else "")) if use_ticks else (
                       "one graph launch [heartbeat-slice H2D + %sworker_chunk/merge] (overlapped with policy_kernel) + route_kernel" % (
                           ("peer-memory gather + " if args.exchange == "peer" else "all-gather + ") if world > 1 else "")),
                   "step_mode": args.step,
                   "layout": "jobs as topic-sorted 64 B + 32 B records (host encoder), bulk-async tile loads",
                   "exchange": ("peer memory (CUDA IPC over NVLink, push kernel inside the ingest graph)" if args.exchange == "peer" else
                                ("engine-owned NCCL all-gather" if args.exchange == "nccl" else args.exchange)) if world > 1 else "none"},
        "clocks": clocks,
        "e2e": {"value": J * e2e_steps / e2e_elapsed, "unit": UNIT,
                "h2d_bytes_per_step": int(env_bytes + (w1 - w0) * 16), "d2h_bytes_per_step": int(n_shard * out_b),
                "includes": "string-level envelopes in page-locked host memory (per-job strings, nothing interned) -> H2D of the "
                            "envelope bytes -> cordum_encode_device (dictionary coding + topic sort on the GPU) -> kernels -> D2H of "
                            "the decision records, 2 batches in flight",
                "input": "de-interned arena: %.0f MB of strings + %.0f MB of spans for %d jobs" % (
                    len(plain_jobs.arena) / 1e6, (env_bytes - len(plain_jobs.arena)) / 1e6, n_shard),
                "host_fallbacks": int(e2e_fallbacks),
                "host_encoder": {"value": J * e2e_steps / e2e_host_elapsed, "interned_arena": J * e2e_steps / e2e_int_elapsed,
                                 "encode_ms_per_batch": float(np.median(enc_host_ms)), "encode_ms_per_batch_interned": float(np.median(enc_int_ms)),
                                 "what": "cordum_encode on the host threads + H2D of the 96 B records instead of the device encoder"},
                "from_encoded_records": J * e2e_steps / e2e_cols_elapsed,
                "host": hostinfo.describe()},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_note, "kernel": "policy_kernel", "kernel_ms": k_ms,
                     "algorithmic_bytes": int(algo_bytes), "peak_source": peak_src,
                     "other_kernels": {"route_kernel_ms": r_ms},
                     "whole_path": {"algorithmic_bytes": int(path_bytes), "kernels_ms": k_ms + r_ms, "achieved": path_gbs,
                                    "frac": path_gbs / peak},
                     "whole_path_survey_8d": {"bytes_per_decision": 100, "algorithmic_bytes": int(s8d_bytes),
                                              "kernels_ms": k_ms + r_ms, "achieved": s8d_gbs, "frac": s8d_gbs / peak}},
        "cpu_baseline": cpu,
        "parity_check": parity,
    }
    print(json.dumps(line), flush=True)
    for b in batches:
        b.free()
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="cordum_b200", choices=["cordum_b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the decision records of the last timed step as DIR/<field>.npy (float32 / float64)")
    ap.add_argument("--value-only", action="store_true", help="diagnostic runs: skip the end-to-end and per-kernel sections")
    ap.add_argument("--parity-sample", type=int, default=0,
                    help="check only the first N jobs of each rank's shard against the oracle (0 = every job; for quick runs)")
    ap.add_argument("--step", default="streams", choices=["tick", "streams"],
                    help="device-resident step: the multi-stream path (cordum_workers_ingest as one graph launch + "
                         "cordum_dispatch_resident_async; measured faster at 1-8 GPUs) or one CUDA-graph scheduler tick per step")
    ap.add_argument("--exchange", default="nccl", choices=["peer", "nccl", "torch"],
                    help="heartbeat exchange at N > 1: the engine's NCCL communicator (all-gather of the slices; measured fastest at "
                         "2-8 GPUs), peer memory over NVLink (CUDA IPC, push kernel inside the ingest graph), or torch.distributed "
                         "all_gather + cordum_workers_set_loads_device")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (the reference leg times a sample sized by its own speed)")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_cuda(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
