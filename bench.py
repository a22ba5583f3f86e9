#!/usr/bin/env python
"""bench.py — composed-GPU probes/sec for the post-attach probe + spec path.

A "step" is one pass of the hot path for one freshly composed GPU: the attach
reconcile step (enumerate -> HBM probe -> visibility decision -> status / CDI
JSON emit), BASELINE.json config 2 ("1xB200 attach: sm_100a HBM probe + CDI
emit").  One probe = 1 fill + 5 copy sweeps + 5 read sweeps over S = 4 GiB
(algorithmic bytes 16*S, DESIGN.md "Measurement"); the copies run ping-pong and
fold their source out of shared memory, so every byte a sweep writes is
re-read and compared with the closed form by the sweep after it.

  e2e        THE throughput: probes/s through the public C-ABI call
             (cro_reconcile_attach): host JSON in, host JSON out, the node's
             inventory re-read, host<->device copies inside, wall clock
             bracketed by barrier + synchronize.
  value      the same K probes divided by the CUDA-event time of their kernels
             (events recorded by libcroprobe on the stream the kernels run on),
             max over ranks: what the device itself needs, no host time.
  roofline   the kernel with the largest share of the step (hbm_copy_fused)
             against MEASURED_PEAKS.json; roofline_kernels lists all of them.
  cpu_baseline / --impl reference
             the reference's CPU path for the same step (exec nvidia-smi,
             parse, decide, emit) from the oracle port, timed on this host.
  cold       (N = 1) the hot-plug path: a fresh helper process per attach
             (croprobe-cli), process start to first verdict.
  fullbox    (N > 1) BASELINE config 3 under the same clock: ONE process,
             cro_probe_all over the N GPUs — concurrent HBM probes, NVLink read /
             push / latency rounds chained by events, the in-library
             ncclAllGather of the device-written 512-byte structs.
  storm / churn  (N > 1) BASELINE configs 4 and 5 on the same context.

N > 1 (torchrun): one rank per GPU, each probes its own device (weak scaling,
no data-path collective) and the 512-byte result structs are all-gathered over
NCCL — the one exchange step the path has; then rank 0 alone runs the
single-process legs while the other ranks wait on a CPU (gloo) barrier.

--dump-outputs DIR writes what the last probe of the `value` loop handed its
caller (the device-written verdict and checksums) and a fixed sample of the
region it left in HBM, as DIR/<name>.npy.  The pattern seed does not depend on
which GPU of the box the run lands on, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import random
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: nothing is cached beside the sources

SWEEP_BYTES = 4 << 30
READ_SWEEPS = COPY_SWEEPS = 5
# The library seeds a device's pattern with seed_base | device minor; with the low 16 bits set the minor drops out, so
# the bytes a run probes do not depend on which GPU it was given.  Ranks are kept apart above those bits.
SEED_BASE = 0x00C0FFEE0000FFFF
DUMP_BLOCKS, DUMP_BLOCK_WORDS = 64, 1024     # region sample: 64 seeded blocks of 1024 words (1 MiB as float64 halves)
METRIC = "composed-GPU probes/sec"
UNIT = "probes/s"
WORKLOAD = "configs[1]: 1xB200 attach — HBM probe (fill + 5 read + 5 copy sweeps, S=4 GiB) + CDI/status JSON emit"
CANNED_UUID = "GPU-device00-uuid-temp-0000-000000000000"


def workload_config(sweep_bytes: int, world: int):
    """The `config` object: the workload and nothing else, so both arms print the same one."""
    return {"workload": WORKLOAD, "sweep_bytes": sweep_bytes, "read_sweeps": READ_SWEEPS, "copy_sweeps": COPY_SWEEPS,
            "algorithmic_bytes_per_probe": 16 * sweep_bytes,
            "l2": "inputs (4 GiB per sweep) are larger than the 126 MB L2; no flush needed",
            "parallelism": "1 rank per GPU, independent devices, one 512 B all-gather per step" if world > 1 else "1 GPU"}


_REAL_STDOUT = None


def emit(line) -> None:
    """Writes the one JSON line to the process's real stdout (see main())."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        smi = shutil.which("nvidia-smi")
        if not smi:
            return
        try:
            self.proc = subprocess.Popen([smi, "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for k, name in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's CPU path
# ---------------------------------------------------------------------------
def reference_step_factory(spawn: bool = True):
    """Returns (step_fn, description, oracle).  One step = what handleAttachingState does on the CPU for one CR:
    exec `nvidia-smi --query-gpu=gpu_uuid` (internal/utils/gpus.go:886), parse (:896-916), decide (:73-84),
    emit status JSON + the FM scale-up body.  The SPDY/kubelet hop of the reference is NOT included, so this
    is a lower bound on the reference's latency.  spawn=False replaces the exec by an in-process NVML enumeration
    (the best a CPU path could do; not something the reference does)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    co = oracle.COracle()
    smi = shutil.which("nvidia-smi")
    canned = CANNED_UUID + "\n"
    nvml = None
    if not spawn:
        try:
            import pynvml
            pynvml.nvmlInit()
            nvml = pynvml
        except Exception:
            nvml = None
    if smi:
        first = subprocess.run([smi, "--query-gpu=gpu_uuid", "--format=csv,noheader,nounits"], capture_output=True, text=True)
        dev = first.stdout.strip().split("\n")[0].strip() if first.returncode == 0 and first.stdout.strip() else CANNED_UUID
    else:
        dev = CANNED_UUID

    fm_reply = json.dumps({"data": {"machines": [{"resources": [{"res_uuid": "res-0-0", "res_type": "gpu", "res_op_status": "0",
                                                                  "res_serial_num": dev, "res_spec": {"condition": [
                                                                      {"column": "model", "operator": "eq", "value": "NVIDIA-B200"}]}}]}]}})

    def enumerate_text():
        if not spawn:
            if nvml is not None:
                uuids = []
                for i in range(nvml.nvmlDeviceGetCount()):
                    u = nvml.nvmlDeviceGetUUID(nvml.nvmlDeviceGetHandleByIndex(i))
                    uuids.append(u.decode() if isinstance(u, bytes) else u)
                return "\n".join(uuids) + "\n", "", None
            return canned, "", None
        if smi:
            p = subprocess.run([smi, "--query-gpu=gpu_uuid", "--format=csv,noheader,nounits"], capture_output=True, text=True)
            return p.stdout, p.stderr, (None if p.returncode == 0 else "exit status %d" % p.returncode)
        return canned, "", None

    def step():
        so, se, ee = enumerate_text()
        inp = oracle.AttachInput(name="cr", target_node="worker-0", device_resource_type="DEVICE_PLUGIN",
                                 provider_device_id=dev, provider_cdi_device_id="res-0-0", std_out=so, std_err=se, exec_err=ee)
        st, rq, err, _n = co.attach_step(inp, oracle.Status("Attaching"))
        js = co.emit_status(st.state, st.error, st.device_id, st.cdi_device_id)
        body = co.emit_fm_scale_up("tenant", "machine", "gpu", "NVIDIA-B200")
        ids = oracle.fm_scale_up_response_to_ids(fm_reply, "cr", "gpu", "NVIDIA-B200")   # the provider's half of the step
        return st.state, len(js) + len(body) + len(ids[0])

    if not spawn:
        how = ("NVML in process (pynvml) + oracle parse/decide/emit, no process spawn" if nvml is not None else
               "canned enumeration text + oracle parse/decide/emit, no process spawn")
    else:
        how = ("exec nvidia-smi --query-gpu=gpu_uuid per step + oracle parse/decide/emit" if smi else
               "nvidia-smi absent: canned enumeration text + oracle parse/decide/emit (process spawn NOT included)")
    return step, how, co


def cpu_best_case(budget_s: float = 3.0):
    """The CPU path with its dominant cost (the nvidia-smi spawn) taken away: NVML in process + parse / decide / emit.
    Not a configuration the reference has — it shows where a CPU-only rewrite of the UUID check would land."""
    step, how, _co = reference_step_factory(spawn=False)
    step()
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s and n < 200000:
        step()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": 1, "sample": "%d steps in %.1f s; %s" % (n, dt, how),
            "note": "checks that a UUID is listed; moves no bytes through the device"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    step, how, _co = reference_step_factory()
    # The unmodified reference reconciles ONE ComposableResource at a time: SetupWithManager sets no
    # MaxConcurrentReconciles (internal/controller/composableresource_controller.go:444-448), so
    # controller-runtime runs a single worker.  One host thread (plus the nvidia-smi child it execs) is
    # therefore every thread this path can use; `value` is that.  For transparency the same run also times
    # a hypothetical 32-worker build ("all_threads") — not a configuration the reference ships.
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()                         # a step is ONE reconcile, as in our arm
    dt = time.perf_counter() - t0
    value = args.steps / dt
    cores = 1
    wide = min(os.cpu_count() or 1, 32)
    t1 = time.perf_counter()
    with ThreadPoolExecutor(wide) as ex:
        list(ex.map(lambda _i: step(), range(2 * wide)))
    all_threads = {"value": 2 * wide / (time.perf_counter() - t1), "unit": UNIT, "cores": wide,
                   "note": "hypothetical MaxConcurrentReconciles=%d; the reference ships 1" % wide}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args.sweep_bytes, world),
        "reference_path": "oracle port (the Go reference cannot be compiled here: no Go toolchain); one reconcile worker",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": how},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "all_threads": all_threads, "cpu_best_case": cpu_best_case(),
        "what_it_checks": "a UUID string is listed by nvidia-smi (gpus.go:73-84); ~99 % of a step is the process spawn",
        "gpu_launches": 0,
    }
    emit(line)


def cpu_baseline(budget_s: float = 12.0):
    step, how, co = reference_step_factory()
    step()
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s and n < 2000:
        step()
        n += 1
    dt = time.perf_counter() - t0
    # context: what the same integer sweep costs on the host (closed form, all cores), bounded to 256 MiB
    cores = os.cpu_count() or 1
    words = (256 << 20) // 8
    t1 = time.perf_counter()
    co.checksum(0x00C0FFEE00000000, 0, words, threads=cores)
    sweep_s = time.perf_counter() - t1
    return {"value": n / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d sequential steps in %.1f s; %s" % (n, dt, how),
            "enumerate_ms": cpu_enumerate_ms(), "best_case_no_spawn": cpu_best_case(),
            "host_pattern_checksum_gbs_all_cores": (256 << 20) / sweep_s / 1e9, "host_cores": cores}


def cpu_enumerate_ms():
    """Best-case CPU enumeration next to the reference's exec of nvidia-smi (SURVEY.md §8d config 1): NVML in
    process, and the /proc scan the RKE2 branch scripts (internal/utils/gpus.go:1017-1037).  Median of 10, ms."""
    out = {}

    def med(fn, n=10):
        ts = []
        for _ in range(n):
            t = time.perf_counter()
            fn()
            ts.append((time.perf_counter() - t) * 1e3)
        ts.sort()
        return round(ts[len(ts) // 2], 3)
    smi = shutil.which("nvidia-smi")
    if smi:
        out["nvidia_smi_exec"] = med(lambda: subprocess.run([smi, "--query-gpu=gpu_uuid", "--format=csv,noheader,nounits"],
                                                            capture_output=True), 5)
    try:
        import pynvml

        def nvml():
            pynvml.nvmlInit()
            for i in range(pynvml.nvmlDeviceGetCount()):
                h = pynvml.nvmlDeviceGetHandleByIndex(i)
                pynvml.nvmlDeviceGetUUID(h), pynvml.nvmlDeviceGetMinorNumber(h), pynvml.nvmlDeviceGetPciInfo(h)
            pynvml.nvmlShutdown()
        out["nvml_in_process"] = med(nvml)
    except Exception as e:   # noqa: BLE001
        out["nvml_in_process"] = "unavailable: %s" % type(e).__name__
    base = "/proc/driver/nvidia/gpus"
    if os.path.isdir(base):
        def proc():
            for name in sorted(os.listdir(base)):
                p = os.path.join(base, name, "information")
                if os.path.isfile(p):
                    open(p).read()
        out["proc_scan"] = med(proc)
    return out


# ---------------------------------------------------------------------------
# the hot-plug path: a fresh helper process per attach
# ---------------------------------------------------------------------------
def cold_leg(uuid: str, runs: int = 4):
    """A GPU composed after the agent's cuInit is invisible to its CUDA contexts; libcroprobe then probes it through
    `croprobe-cli probe-raw` (its own cuInit, CUDA_VISIBLE_DEVICES=<uuid>).  This times that helper from process start
    to first verdict, K times: the first run also pays the page-in of the driver stack."""
    cli = os.path.join(ROOT, "composable-resource-operator_b200", "croprobe-cli")
    if not os.path.exists(cli):
        return {"unavailable": "croprobe-cli not built"}
    rows = []
    for sweep_mib, nvml in ((1024, False),) * runs + ((4096, False), (1024, True)):
        t0 = time.perf_counter()
        p = subprocess.run([cli, "cold", uuid, str(sweep_mib)] + (["nvml"] if nvml else []), capture_output=True, text=True, timeout=120)
        wall = time.perf_counter() - t0
        if p.returncode != 0:
            return {"error": (p.stdout + p.stderr)[-300:]}
        d = json.loads(p.stdout.strip().split("\n")[-1])
        d["process_wall_s"] = round(wall, 4)
        rows.append(d)
    hot = rows[1:runs]           # helper default (1 GiB, identity from /proc), driver stack paged in
    best = min(hot, key=lambda d: d["cold_total_s"])
    return {"helper": "croprobe-cli cold <uuid> 1024 (one device, CUDA_VISIBLE_DEVICES=<uuid>, identity from /proc, lazy region)",
            "init_s": best["init_s"], "first_probe_ms": round(best["cold_probe_s"] * 1e3, 3), "warm_probe_ms": round(best["warm_probe_s"] * 1e3, 3),
            "start_to_first_verdict_s": best["cold_total_s"], "probes_per_s": round(1.0 / best["cold_total_s"], 2),
            "first_run_of_the_box_s": rows[0]["cold_total_s"], "runs": [r["cold_total_s"] for r in rows[:runs]],
            "with_4gib_sweep_s": rows[runs]["cold_total_s"], "with_nvml_identity_s": rows[runs + 1]["cold_total_s"],
            "status": max(r["status"] for r in rows)}


# ---------------------------------------------------------------------------
# single-process legs (BASELINE configs 3, 4, 5): what a Go operator calls
# ---------------------------------------------------------------------------
def gbs(b, ns):
    return round(b / ns, 1) if ns else None


def stats(vals):
    vals = [v for v in vals if v]
    if not vals:
        return None
    return {"min": min(vals), "mean": round(sum(vals) / len(vals), 1), "max": max(vals), "n": len(vals)}


def fullbox_leg(cro, ctx, S, steps, warmup, coracle):
    """BASELINE config 3: cro_probe_all — concurrent HBM probes, NVLink rounds, in-library ncclAllGather."""
    n = ctx.device_count()
    t0 = time.perf_counter()
    res = ctx.probe_all()            # first call: peer mappings, latency tables, ncclCommInitAll
    first_s = time.perf_counter() - t0
    for _ in range(max(1, warmup)):
        res = ctx.probe_all()
    walls, fts = [], []
    ok = True
    for _ in range(steps):
        t0 = time.perf_counter()
        res = ctx.probe_all()
        walls.append(time.perf_counter() - t0)
        fts.append(ctx.fullbox_times())
        ok = ok and all(r.status == 0 and r.fail_code == 0 for r in res)
    P = int(res[0].p2p_bytes)
    full = (1 << n) - 1
    ok = ok and all((r.p2p_ok | (1 << i)) & full == full for i, r in enumerate(res) if n <= 8)
    # parity against the oracle: two devices' HBM closed forms at full size, and every NVLink leg of device 0
    cores = os.cpu_count() or 1
    for r in res[:2]:
        ok = ok and r.checksum == r.expect == coracle.checksum(r.seed, 0, S // 8, threads=cores)
    devs = ctx.own_devices()
    for j in range(1, n):
        d = ctx.p2p_detail(0, j)
        want = coracle.checksum(res[j].seed, 0, P // 8, threads=cores)
        ok = ok and (d.read_xor, d.read_sum, d.read_wsum) == want
        ok = ok and (d.landed_xor, d.landed_sum, d.landed_wsum) == coracle.checksum(res[0].seed, 0, P // 8, threads=cores)
        ok = ok and d.chase_end == coracle.chase_end(max(devs[0].device_minor, 0), max(devs[j].device_minor, 0), d.hops)
    mean_wall = sum(walls) / len(walls)
    med = lambda xs: sorted(xs)[len(xs) // 2]   # noqa: E731
    read = [gbs(P, r.p2p_read_ns[j]) for i, r in enumerate(res) for j in range(min(n, 8)) if j != i]
    push = [gbs(P, r.p2p_write_ns[j]) for i, r in enumerate(res) for j in range(min(n, 8)) if j != i]
    lat = [r.p2p_latency_ns_x16[j] / 16.0 for i, r in enumerate(res) for j in range(min(n, 8)) if j != i and r.p2p_latency_ns_x16[j]]
    rs, ps = stats(read), stats(push)
    out = {
        "call": "cro_probe_all (one process, %d GPUs)" % n, "n_gpus": n, "steps": steps, "p2p_bytes": P,
        "latency_hops": int(ctx.p2p_detail(0, 1).hops) if n > 1 else 0,
        "probes_per_s": round(n / mean_wall, 1), "ms_per_call": round(mean_wall * 1e3, 3), "ms_per_call_median": round(med(walls) * 1e3, 3),
        "first_call_s": round(first_s, 3),
        "phases_ms": {"hbm": round(med([f.hbm_ns for f in fts]) / 1e6, 3), "nvlink_bandwidth_rounds": round(med([f.p2p_ns for f in fts]) / 1e6, 3),
                      "latency_chase": round(med([f.chase_ns for f in fts]) / 1e6, 3), "allgather": round(med([f.gather_ns for f in fts]) / 1e6, 4),
                      "host_enqueue": round(med([f.enqueue_ns for f in fts]) / 1e6, 3)},
        "allgather_us": round(med([f.gather_ns for f in fts]) / 1e3, 1),
        "host_syncs_per_call": int(fts[-1].host_syncs), "rounds": int(fts[-1].rounds),
        "gather": {0: "host", 1: "ncclAllGather (in library)", 2: "host (degraded: no usable libnccl — replicas only)"}[int(fts[-1].gather)],
        "hbm_read_gbs": stats([gbs(S, r.read_best_ns) for r in res]), "hbm_copy_gbs": stats([gbs(2 * S, r.copy_best_ns) for r in res]),
        "nvlink_read_gbs": rs, "nvlink_push_gbs": ps, "latency_ns": stats([round(x, 1) for x in lat]),
        "matrix_flat": bool(rs and (rs["max"] - rs["min"]) <= 0.05 * rs["mean"]),
        "nvlink_frac_of_900_nominal": {"read": round(rs["mean"] / 900.0, 3) if rs else None, "push": round(ps["mean"] / 900.0, 3) if ps else None},
        "nvlink_frac_of_770_measured_peer_copy": {"read": round(rs["mean"] / 770.0, 3) if rs else None,
                                                   "push": round(ps["mean"] / 770.0, 3) if ps else None},
        "gathered_identical_on_all_ranks": True,     # asserted inside cro_probe_all (it fails with CRO_ERR_NCCL otherwise)
        "copies_verified": [int(r.copy_verified) for r in res], "parity_ok": bool(ok),
    }
    # how many hops does the latency figure need?  (SURVEY.md §8d asks for 64 Ki; the default is 1 Ki)
    if n > 1:
        conv = {}
        default_hops = out["latency_hops"]
        for hops in (1024, 4096, 16384, 65536):
            ctx.set_latency_hops(hops)
            r2 = ctx.probe_all()
            ft = ctx.fullbox_times()
            l2 = [r.p2p_latency_ns_x16[j] / 16.0 for i, r in enumerate(r2) for j in range(min(n, 8)) if j != i and r.p2p_latency_ns_x16[j]]
            conv[str(hops)] = {"mean_ns": round(sum(l2) / len(l2), 1), "min_ns": round(min(l2), 1), "max_ns": round(max(l2), 1),
                               "chase_ms": round(ft.chase_ns / 1e6, 3), "status": max(r.status for r in r2)}
            ok = ok and all(r.status == 0 for r in r2)
        ctx.set_latency_hops(default_hops)
        out["latency_vs_hops"] = conv
        out["parity_ok"] = bool(ok)
    return out


def storm_leg(cro, ctx, n_req, probe=True):
    """BASELINE config 4: n_req synthetic ComposabilityRequests over the box's GPUs, warm probe contexts."""
    n = ctx.device_count()
    nodes = ["worker-%d" % i for i in range(n)]
    rng = random.Random(20260921)
    with cro.Cluster({"nodes": nodes, "probe": probe, "device_resource_type": "DEVICE_PLUGIN"}, ctx) as c:
        sizes = []
        for i in range(n_req):
            size = rng.randint(1, 4)
            sizes.append(size)
            err = c.apply("req-%04d" % i, {"type": "gpu", "model": "NVIDIA-B200-%d" % (i // n), "size": size,
                                           "allocation_policy": "samenode", "target_node": "worker-%d" % (i % n)})
            assert err == "", err
        t0 = time.perf_counter()
        st = c.run()
        wall = time.perf_counter() - t0
        per_node = [0] * n
        for i, s in enumerate(sizes):
            per_node[i % n] += s
        return {"config": 4, "probe": probe, "n_gpus": n, "requests": n_req, "children": sum(sizes), "wall_s": round(wall, 3),
                "requests_running": st["requests_running"], "resources_online": st["resources_online"],
                "requests_per_s": round(st["requests_running"] / wall, 1), "child_probes_per_s": round(st["probes"] / wall, 1) if probe else None,
                "specs_per_s": round(st["status_updates"] / wall, 1), "status_updates": st["status_updates"], "spec_bytes": st["spec_bytes"],
                "reconciles": st["request_reconciles"] + st["resource_reconciles"], "reconcile_p50_us": st["reconcile_p50_ns"] / 1e3,
                "reconcile_p99_us": st["reconcile_p99_ns"] / 1e3, "errors": st["reconcile_errors"], "probe_failures": st["probe_failures"],
                "busiest_gpu_children": max(per_node),
                # per GPU: probes, device time busy (its own %globaltimer), first probe start .. last probe end
                "gpus": st.get("gpus"), "gpu_busy_frac_of_span": [round(g["busy_us"] / max(1, g["span_us"]), 4) for g in st.get("gpus", [])],
                "bound_s_busiest_gpu": round(max((g["busy_us"] for g in st.get("gpus", [])), default=0) / 1e6, 3),
                "note": "single reconcile worker per controller (reference default), physical GPUs multiplexed across CRs, timers immediate"}


def churn_leg(cro, ctx, cycles, probe=True):
    """BASELINE config 5: attach/detach churn, 4-GPU compose -> Online -> decompose per cycle."""
    n = ctx.device_count()
    width = min(4, n)
    with cro.Cluster({"nodes": ["worker-%d" % i for i in range(n)], "probe": probe}, ctx) as c:
        t0 = time.perf_counter()
        probes = 0
        st = {"reconcile_errors": 0, "probe_failures": 0}
        for cyc in range(cycles):
            names = []
            for j in range(width):
                name = "churn-%d-%d" % (cyc, j)
                names.append(name)
                assert c.apply(name, {"type": "gpu", "model": "NVIDIA-B200", "size": 1, "target_node": "worker-%d" % ((width * cyc + j) % n)}) == ""
            st = c.run()
            assert st["requests_running"] == width, st
            for x in names:
                c.delete(x)
            st = c.run()
            probes = st["probes"]
        wall = time.perf_counter() - t0
        d = c.dump()
        return {"config": 5, "probe": probe, "n_gpus": n, "cycles": cycles, "width": width, "attaches": cycles * width, "wall_s": round(wall, 3),
                "probes": probes, "probes_per_s": round(probes / wall, 1) if probe else None, "attach_detach_cycles_per_s": round(cycles / wall, 2),
                "left_over_objects": len(d["requests"]) + len(d["resources"]), "errors": st["reconcile_errors"], "probe_failures": st["probe_failures"],
                "note": "logical attach/detach (CUDA cannot hot-plug inside one process); warm probe contexts"}


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
def dump_outputs(out_dir, ctx, r, S):
    """What the last timed probe computed, as float64 arrays; 64-bit words are split into exact (high, low) 32-bit halves.
    The struct's times are left out: they are measurements, not results."""
    import numpy as np

    def halves(words):
        w = np.asarray(words, dtype=np.uint64)
        return np.stack([w >> np.uint64(32), w & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    # (checksum, closed form, copy checksum) x (xor, sum, position-weighted sum) x (high, low)
    np.save(os.path.join(out_dir, "probe_checksums.npy"), halves([r.checksum, r.expect, r.copy_checksum]))
    np.save(os.path.join(out_dir, "probe_seed.npy"), halves([r.seed]))
    np.save(os.path.join(out_dir, "probe_verdict.npy"), np.array(
        [r.status, r.fail_code, r.fail_index, r.copy_verified, r.read_sweeps, r.copy_sweeps, r.nonce, r.sweep_bytes], dtype=np.float64))
    words = 2 * S // 8                     # both halves of the ping-pong region, as the last sweeps left them
    n = min(DUMP_BLOCK_WORDS, words)
    firsts = np.random.default_rng(0).integers(0, words - n + 1, DUMP_BLOCKS)
    np.save(os.path.join(out_dir, "region_sample.npy"), halves([ctx.read_words(0, int(f), n) for f in firsts]))


def run_ours(args, rank, local_rank, world):
    import torch
    cro = importlib.import_module("composable-resource-operator_b200")
    multirank = importlib.import_module("composable-resource-operator_b200.multirank")
    dist = cpu_group = None
    if world > 1:
        import datetime
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # a CPU-side group for the waits that must not touch a GPU (an NCCL barrier parks a kernel on every rank's device)
        cpu_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(minutes=30))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    S = args.sweep_bytes

    t_init = time.perf_counter()
    ctx = cro.ProbeContext(sweep_bytes=S, devices=[local_rank], read_variant=args.read_variant,
                           copy_variant=args.copy_variant, rank_base=rank, world=world, read_sweeps=READ_SWEEPS, copy_sweeps=COPY_SWEEPS,
                           seed_base=SEED_BASE + (rank << 16))
    info = ctx.own_devices()[0]
    uuid = info.gpu_uuid.decode()
    ctx_create_s = time.perf_counter() - t_init

    send = gathered = None
    if world > 1:
        send = torch.as_tensor(multirank.DevBuf(ctx.result_device_ptr(0), 512), device=dev)
        gathered = torch.empty(world * 512, dtype=torch.uint8, device=dev)

    # The attach reconcile with the FM provider client in the loop (csrc/provider.cpp): metal3 walk ->
    # PATCH ScaleUpBody (emitted) -> ScaleUpResponse (parsed, op-status gate) -> probe -> status JSON.
    # The fabric's reply is scripted: the appliance is not part of the box.
    node, machine = "worker-%d" % rank, "machine-%d" % rank
    fm_reply = json.dumps({"data": {"machines": [{"fabric_uuid": "", "fabric_id": 0, "mach_uuid": machine, "mach_id": 0,
                                                  "mach_name": "", "tenant_uuid": "tenant", "resources": [{
                                                      "res_uuid": "res-%d-0" % rank, "res_name": "", "res_type": "gpu", "res_status": 0,
                                                      "res_op_status": "0", "res_serial_num": uuid,
                                                      "res_spec": {"condition": [{"column": "model", "operator": "eq",
                                                                                  "value": "NVIDIA-B200"}]}}]}]}},
                          separators=(",", ":"))
    request = {"name": "cr-%d" % rank, "spec": {"type": "gpu", "model": "NVIDIA-B200", "target_node": node},
               "status": {"state": "Attaching"}, "probe": True,
               "env": {"DEVICE_RESOURCE_TYPE": "DEVICE_PLUGIN", "CDI_PROVIDER_TYPE": "FTI_CDI", "FTI_CDI_API_TYPE": "FM",
                       "FTI_CDI_TENANT_ID": "tenant", "FTI_CDI_CLUSTER_ID": "cluster"},
               "fabric": {"http": [{"method": "PATCH", "path": "fabric_manager/api/v1/machines/%s/update" % machine,
                                    "status": 200, "body": fm_reply}],
                          "objects": {"nodes": {node: {"annotations": {"machine.openshift.io/machine": "ns/m"}}},
                                      "metal3machines": {"ns/m": {"annotations": {"metal3.io/BareMetalHost": "ns/b"}}},
                                      "baremetalhosts": {"ns/b": {"annotations": {"cluster-manager.cdi.io/machine": machine}}}}}}
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    coracle = oracle.COracle()

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    ag_start, ag_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def all_gather_results():
        """The path's one exchange step: 512-byte result structs over NCCL; returns its device time in ns."""
        if not dist:
            return 0
        ag_start.record()
        dist.all_gather_into_tensor(gathered, send)
        ag_end.record()
        ag_end.synchronize()
        return int(ag_start.elapsed_time(ag_end) * 1e6)

    # ---- warm-up -----------------------------------------------------------
    for _ in range(max(3, args.warmup)):
        ctx.probe_device(0)
        all_gather_results()
        cro.reconcile_attach(ctx, request)

    # ---- device-resident timing: `value` ------------------------------------
    sampler = ClockSampler(info.cuda_ordinal)
    sampler.start()
    time.sleep(0.25)
    launches0 = ctx.launch_count()
    barrier()
    dev_ns = 0
    ev = {0: [], 1: [], 2: []}          # CUDA-event ns per sweep kind: fill / copy / read
    tm = {0: [], 1: [], 2: []}          # the kernels' own %globaltimer windows
    results = []
    for _ in range(args.steps):
        r = ctx.probe_device(0)
        ts = ctx.sweep_times(0)
        dev_ns += sum(t.event_ns for t in ts) + all_gather_results()
        for t in ts:
            ev[t.kind].append(t.event_ns)
            tm[t.kind].append(t.timer_ns)
        results.append(r)
    barrier()
    launches = ctx.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, results[-1], S)

    # ---- end to end through the reference-facing call: `e2e` ----------------
    barrier()
    t0 = time.perf_counter()
    specs = 0
    last = None
    rec_s = ag_s = 0.0
    for _ in range(args.steps):
        ta = time.perf_counter()
        last = cro.reconcile_attach(ctx, request)       # host JSON in -> fresh inventory -> probe -> host JSON out
        tb = time.perf_counter()
        all_gather_results()
        ag_s += time.perf_counter() - tb
        rec_s += tb - ta
        specs += 1
    barrier()
    e2e_s = time.perf_counter() - t0
    sampler.stop()
    time.sleep(0.05)
    clocks = sampler.summary()

    # max over ranks
    if dist:
        t = torch.tensor([float(dev_ns), e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ns, e2e_s = float(t[0]), float(t[1])
        gl = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(gl)
        launches = int(gl[0])

    # parity: every probe's device-written verdict is clean AND equals the CPU oracle's closed form for ITS seed
    cores = os.cpu_count() or 1
    ok = all(r.status == 0 and r.fail_code == 0 and r.copy_verified == r.copy_sweeps == COPY_SWEEPS and r.read_sweeps == READ_SWEEPS
             for r in results)
    ok = ok and len({r.nonce for r in results}) == len(results)               # every probe wrote a fresh pattern
    for r in (results[0], results[-1]):
        ok = ok and r.checksum == r.expect == r.copy_checksum == coracle.checksum(r.seed, 0, S // 8, threads=max(1, cores // max(1, world)))
    ok = ok and (last["status"]["state"] == "Online" and last["status"].get("device_id") == uuid and
                 len(last.get("fabric_requests", [])) == 1)
    if world > 1:
        # every rank must hold the same gathered array: one struct per rank, distinct devices, all ok
        everyone = multirank.results_from_bytes(bytes(gathered.cpu().numpy().tobytes()))
        problem = multirank.check_gathered(everyone, world)
        if problem or everyone[rank].gpu_uuid != info.gpu_uuid or [r.rank for r in everyone] != list(range(world)):
            print("rank %d: bad all-gather: %s" % (rank, problem), file=sys.stderr)
            ok = False
    if dist:
        okt = torch.tensor([1 if ok else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        ok = bool(int(okt[0]))

    line = None
    if rank == 0:
        peak, peak_src = load_peaks()
        value = world * args.steps / (dev_ns * 1e-9)
        e2e = world * args.steps / e2e_s
        avg = lambda xs: sum(xs) / max(1, len(xs))   # noqa: E731
        step_ns = sum(ev[0]) + sum(ev[1]) + sum(ev[2])

        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except Exception:
            ncu = None

        def roof(name, kind, alg_bytes):
            avg_ns = avg(ev[kind])
            ach = alg_bytes / avg_ns   # bytes per ns == GB/s
            traffic = None
            if ncu and name in ncu:    # dram bytes per launch from the committed ncu --set full capture, scaled to S
                traffic = (ncu[name]["dram_read"] + ncu[name]["dram_write"]) * (S / ncu["sweep_bytes"])
            return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "frac_of_nominal_8000": ach / 8000.0,
                    # 60 of 64 channel-equivalents carry a uniformly addressed sweep on the 180 GB part
                    # (profiles/r01_channel_balance.md): 8184 GB/s pin bandwidth * 60/64
                    "frac_of_channel_limited_7670": ach / 7670.0, "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
                    "avg_launch_ms": avg_ns * 1e-6, "avg_launch_ms_globaltimer": avg(tm[kind]) * 1e-6,
                    "share_of_step": sum(ev[kind]) / step_ns, "launches_per_step": len(ev[kind]) // args.steps, "peak_source": peak_src}
        kernels = [roof("hbm_fill", 0, S), roof("hbm_copy_fused", 1, 2 * S), roof("hbm_read_checksum", 2, S)]
        dominant = max(kernels, key=lambda k: k["share_of_step"])
        best_read = min(ev[2])
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": dev_ns * 1e-6 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": workload_config(S, world),
            "impl_details": {"read_variant": int(results[-1].read_variant), "copy_variant": int(results[-1].copy_variant),
                             "sweep_order": "fill, 5 x checksumming copy (ping-pong A->B, B->A, ...), 5 x read (the first one reads the last copy's destination)",
                             "verdict": "written on the device by the finalize kernel (512-byte cro_probe_result, ABI 2)"},
            # what actually crosses PCIe per step: 16 bytes of probe parameters go up; the 512-byte device-written result
            # struct and the first 64 sweep slots (64 B each) come down; the probe's inputs are options, not tensors
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 16, "d2h_bytes_per_step": 512 + 64 * 64,
                    "host_json_in_bytes": len(json.dumps(request)), "host_json_out_bytes": len(last["_raw"]),
                    "ms_per_step": e2e_s * 1e3 / args.steps,
                    "reconcile_ms": rec_s * 1e3 / args.steps, "allgather_wall_ms": ag_s * 1e3 / args.steps,   # rank 0's split of a step
                    "call": "cro_reconcile_attach (C ABI) with host JSON buffers: FM client (walk, ScaleUpBody emit, response "
                            "parse) + fresh node inventory (/proc re-read) + probe + status emit",
                    "fabric_request_bytes": len(last["fabric_requests"][0]["body"]) if last.get("fabric_requests") else 0},
            "specs_per_s": world * specs / e2e_s,
            "probe_gbs_best_read": S / best_read, "probe_frac_of_8000": S / best_read / 8000.0,
            "roofline": dominant, "roofline_kernels": kernels,
            "gpu_launches": launches, "clocks": clocks, "parity_ok": bool(ok),
            "copy_verified": bool(all(r.copy_verified == r.copy_sweeps for r in results)),
            "checks_per_probe": {"copy_destinations_reread_and_compared": COPY_SWEEPS, "read_sweeps_compared": READ_SWEEPS,
                                 "checksum": "xor + wrapping sum + position-weighted sum of every 64-bit word",
                                 "fresh_pattern_per_probe": True, "oracle_recheck": "first and last probe, full 4 GiB, on the host"},
            "ctx_create_s_after_torch_init": ctx_create_s, "device": uuid,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
    ctx.close()

    if world == 1:
        if rank == 0 and not args.no_cold:
            torch.cuda.empty_cache()
            try:
                line["cold"] = cold_leg(uuid)
            except Exception as e:   # noqa: BLE001  (a helper that cannot start is reported, it does not void the step's numbers)
                line["cold"] = {"error": repr(e)}
            if "status" in line["cold"]:          # a probe verdict came back: it must be clean
                ok = ok and line["cold"]["status"] == 0
            line["parity_ok"] = bool(ok)
    else:
        # ---- single-process legs: rank 0 alone, the other ranks wait on the CPU ---------------------------------
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)
        if rank == 0 and not args.no_fullbox:
            n = min(world, torch.cuda.device_count())
            try:
                with cro.ProbeContext(sweep_bytes=S, devices=list(range(n)), p2p_bytes=min(1 << 30, S),
                                      read_sweeps=READ_SWEEPS, copy_sweeps=COPY_SWEEPS) as box:
                    line["fullbox"] = fullbox_leg(cro, box, S, max(3, min(args.steps, 20)), 2, coracle)
                    ok = ok and line["fullbox"]["parity_ok"]
                    P = line["fullbox"]["p2p_bytes"]
                    for name, key in (("p2p_read (hbm_read_tma on a peer-mapped address)", "nvlink_read_gbs"),
                                      ("p2p_push (hbm_copy_fused into a peer-mapped address)", "nvlink_push_gbs")):
                        st = line["fullbox"][key]
                        if st:
                            line["roofline_kernels"].append({
                                "kernel": name, "bound": "nvlink", "achieved": st["mean"], "peak": 770.0, "unit": "GB/s", "frac": st["mean"] / 770.0,
                                "frac_of_nominal_900": st["mean"] / 900.0, "algorithmic_bytes_per_launch": P, "traffic": None,
                                "peak_source": "B200_PROFILING.md: measured peer copy 770 GB/s per direction (900 nominal); both directions of every pair loaded",
                                "min": st["min"], "max": st["max"], "pairs": st["n"]})
                    if not args.no_storm:
                        line["storm"] = storm_leg(cro, box, args.storm)
                        line["churn"] = churn_leg(cro, box, args.cycles)
                        ok = ok and line["storm"]["errors"] == 0 and line["storm"]["probe_failures"] == 0 and \
                            line["storm"]["requests_running"] == args.storm and line["churn"]["left_over_objects"] == 0 and \
                            line["churn"]["probe_failures"] == 0
            except Exception as e:   # noqa: BLE001
                print("single-process legs failed: %r" % (e,), file=sys.stderr)
                line["fullbox"] = {"error": repr(e)}
                ok = False
            line["parity_ok"] = bool(ok)
        dist.barrier(group=cpu_group)
    if rank == 0:
        emit(line)
    if dist:
        dist.barrier(group=cpu_group)
        dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sweep-bytes", type=int, default=SWEEP_BYTES)
    ap.add_argument("--read-variant", type=int, default=0)
    ap.add_argument("--copy-variant", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cold", action="store_true")
    ap.add_argument("--no-fullbox", action="store_true")
    ap.add_argument("--no-storm", action="store_true")
    ap.add_argument("--storm", type=int, default=1000)
    ap.add_argument("--cycles", type=int, default=100)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed probe computed as DIR/<name>.npy")
    args = ap.parse_args()
    # stdout must carry the ONE JSON line and nothing else, but libraries print there too (NCCL writes
    # "NCCL version ..." with printf at init).  Keep the real stdout aside and point fd 1 at stderr for
    # everything else; emit() writes the JSON line to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import __graft_entry__ as g
    if args.impl == "reference":
        # the reference arm maps the CHECKER only: libcroprobe.so is neither built nor imported in this process
        if rank == 0:
            try:
                g.build_oracle()
            except Exception as e:   # noqa: BLE001
                print("build_oracle() failed: %s" % e, file=sys.stderr)
        run_reference(args, rank, world)
        return
    run_ours(args, rank, local_rank, world)     # runs what build() left in the tree; the import fails loudly without it


if __name__ == "__main__":
    main()
