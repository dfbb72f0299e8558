"""bench.py -- pods scheduled/sec (and consolidation candidates/sec) of the B200 solver on BASELINE.json's configs.

A step == one Scheduler.Solve over the whole synthetic batch.
  N = 1  headline = configs[2] (C3), the largest single-GPU configuration: 1 000 000 pods = 1 000 apps x 1 000 replicas,
         zonal topology spread (maxSkew 1) + hostname anti-affinity per app, first 1 000 AWS-KWOK instance types.
           value  pods/s with the problem resident in HBM (kp_upload once, kp_solve_resident per step; device time from
                  CUDA events recorded by the library on its own stream)
           e2e    the same metric through the reference-facing call kp_solve() with HOST buffers: encode-to-tables
                  prep, H2D, kernels and D2H of the result all inside the timed region
         secondary keys: "c2" (configs[1], 100k pods with selectors + tolerations x 500 types), "consolidation"
         (configs[3], 10k nodes / 200k running pods / 166 750 removal subsets), "c5_one_gpu" (configs[4]'s 8 NodePool
         shards as ONE kp_solve_batch on this GPU, one CTA per shard).
  N > 1  headline = configs[4] (C5): 10 000 000 pods, 8 NodePools, C2 + C3 constraint mix, 1 000 types; NodePool p lives
         on rank p mod N, a rank solves its pools as one batch (one CTA per pool) and the step ends with the ONE
         collective of the job -- the library's ncclAllReduce of the global topology-domain counter table -- inside
         the CUDA-event window.  Total work is fixed: "scaling": "strong".
`--impl reference` times the CPU restatement of the reference algorithm (oracle/, kind "port": the Go reference
cannot be built in this image) on the box's host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C3_APPS, C3_REPLICAS, C3_ITS = 1000, 1000, 1000
C2_PODS, C2_ITS = 100_000, 500
C5_PODS, C5_POOLS, C5_ITS = 10_000_000, 8, 1000
# packed row sizes of SURVEY.md section 8(d)
B_POD, B_CLAIM, B_IT = 128, 256, 192
C3_NAME = ("C3: 1M pods = 1000 apps x 1000 replicas, topologySpread(zone, maxSkew 1) + required pod anti-affinity "
           "(hostname) per app, first 1000 AWS-KWOK instance types, 1 NodePool over 3 zones")
C2_NAME = "C2: 100k pods with zone/arch nodeSelector + tolerations, first 500 AWS-KWOK instance types, 1 tainted NodePool"
C5_NAME = ("C5: 10M pods, 8 NodePools (pods pinned by nodeSelector + toleration), half C2 mix / half C3 mix (apps of "
           "1000 replicas, never across pools), first 1000 AWS-KWOK instance types; NodePool p on rank p mod N")
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much in all


def exact_f64(v):
    """float64 copy of an integer result array that keeps every value exact: a 64-bit word becomes its (high, low)
    32-bit halves along a new last axis."""
    a = np.asarray(v)
    if a.dtype.itemsize == 8 and a.dtype.kind in "iu":
        a = np.stack([a >> 32, a & 0xFFFFFFFF], axis=-1)
    return a.astype(np.float64)


def dump_outputs(out_dir, res, keys, limit=DUMP_BYTES):
    """Writes res[k] as out_dir/<k>.npy (float64, see exact_f64) for every k in keys.  When the arrays exceed `limit`
    bytes, every array keeps the same fraction of its rows, sorted, drawn with the array's length as the seed: arrays of
    one length (all the per-pod ones) keep the same rows, and two runs of the same workload keep the same rows."""
    arrays = {k: exact_f64(res[k]) for k in keys}
    budget = limit - 4096 * len(arrays)  # room for the .npy headers
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        if total > budget and a.ndim > 0 and len(a) > 1:
            n = len(a)
            rows = np.random.default_rng(n).choice(n, max(1, n * budget // total), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def algorithmic_bytes(res, n_pods, n_its, n_groups=0, domains=4):
    """B_alg of SURVEY.md section 8(d): the traffic of the REFERENCE algorithm on this input (every CanAdd it would run
    reads one claim row, every commit writes one)."""
    ev = res["n_existing_evals"] + res["n_inflight_evals"] + res["n_template_evals"]
    return n_pods * B_POD + ev * B_CLAIM + res["n_commits"] * B_CLAIM + n_its * B_IT + 2 * n_groups * domains * 4


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum of one solver launch on this workload, from the tracked ncu capture
    (profiles/r2_ncu_traffic.json; a number measured under a profiler is evidence, not a bench value); None if absent."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json"))).get(key)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons while the timed region runs (B200_PROFILING.md).  Sampled through NVML in-process:
    spawning `nvidia-smi` five times a second stalls a one-warp kernel for hundreds of milliseconds at a time (measured:
    individual steps went from 189 ms to 0.5 - 1.4 s), an NVML query does not.  Falls back to nvidia-smi at 1 Hz."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        bits = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        for name, bit in (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown),
                          ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                          ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown),
                          ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap)):
            if bits & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                              str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
        f = [x.strip() for x in out.split(",")]
        self.samples.append(float(f[0]))
        self.max_mhz = float(f[1])
        for n, v in zip(names, f[2:]):
            if v.lower().startswith("active"):
                self.reasons.add(n)

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            time.sleep(float(os.environ.get("KP_SAMPLE_S", "0.2")) if self.nvml is not None else 1.0)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "sm_min_mhz": float(np.min(self.samples)) if self.samples else None,
                "reasons": sorted(self.reasons), "source": "nvml" if self.nvml is not None else "nvidia-smi",
                "samples": len(self.samples)}


def oracle_threads():
    """The reference evaluates candidates with parallelizeUntil (scheduler.go:757-779); the oracle does the same with a
    worker pool.  Use the thread count that is fastest on this host (calibrated on a 25k-pod C2 prefix)."""
    from karpenter_b200 import workloads
    from tests import oracle_lib
    cal = workloads.config_c2(n_pods=25_000, n_its=C2_ITS)
    best_w, best_t = 1, None
    for w in sorted({1, min(os.cpu_count() or 1, 8), min(os.cpu_count() or 1, 16)}):
        dt = None
        for _ in range(2):  # best of two: the first multi-threaded run pays thread start-up and frequency ramp
            t0 = time.perf_counter()
            oracle_lib.solve(cal.problem, threads=w)
            d1 = time.perf_counter() - t0
            dt = d1 if dt is None else min(dt, d1)
        if best_t is None or dt < best_t:
            best_w, best_t = w, dt
    return best_w


def c3_sample(apps):
    """Bounded sample of C3 for the CPU arm: the first `apps` apps with all their 1000 replicas (same generator, same
    seed: pods 0 .. apps*1000-1 of the workload)."""
    from karpenter_b200 import workloads
    return workloads.config_c3(n_apps=apps, replicas=C3_REPLICAS, n_its=C3_ITS)


def run_reference(args, rank, world):
    """The reference's own algorithm (oracle port) on the host cores, on the config the GPU arm reports at this N."""
    from karpenter_b200 import workloads
    from tests import oracle_lib
    if rank != 0:
        return
    oracle_lib.build()
    threads = oracle_threads()
    total = args.steps + args.warmup
    if world == 1:
        # the oracle needs ~0.2 ms per pod on this shape: size the sample so that K + W solves end within a few minutes
        apps = int(max(8, min(60, 480 // max(total, 1))))
        enc = c3_sample(apps)
        n = apps * C3_REPLICAS
        name, cfg = C3_NAME, {"n_pods": C3_APPS * C3_REPLICAS, "n_instance_types": C3_ITS}
        sample = (f"the first {apps} of the {C3_APPS} apps with all their {C3_REPLICAS} replicas ({n} pods; same "
                  f"generator and seed), one full Solve per step")
    else:
        scale = 64 if total <= 8 else 160
        n_total = C5_PODS // scale
        enc = workloads.config_c5(n_pods=n_total, n_pools=C5_POOLS, n_its=C5_ITS, app_replicas=1000, pools_subset=[0])
        n = int(enc.problem.n_pods)
        name, cfg = C5_NAME, {"n_pods": C5_PODS, "n_instance_types": C5_ITS, "n_nodepools": C5_POOLS}
        sample = (f"NodePool 0's shard of the workload generated at 1/{scale} size ({n} pods, same constraint mix), one "
                  f"full Solve per step")
    times, res = [], None
    for i in range(total):
        t0 = time.perf_counter()
        res = oracle_lib.solve(enc.problem, threads=threads)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    ms = 1000 * sum(times) / len(times)
    value = n / (ms / 1000)
    line = {
        "impl": "reference", "metric": "pods scheduled/sec", "value": value, "unit": "pods/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": dict(cfg, workload=name),
        "cpu_baseline": {"value": value, "unit": "pods/s", "cores": threads, "kind": "port",
                         "sample": sample + f"; candidates evaluated by {threads} thread(s) like the reference's "
                                            f"parallelizeUntil (fastest of 1/8/16 on this host, {os.cpu_count()} cores)"},
        "e2e": {"value": value, "unit": "pods/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "unscheduled": int((res["pod_target"] == -1).sum()), "node_claims": int(res["n_claims"]),
    }
    print(json.dumps(line))


def cached_cpu_baseline(oracle_lib, problem, n_pods, gpu_res):
    """oracle/orc_cached.cpp: the solver's OWN algorithm (failure bits, accepted-signature fast path, threshold bitmaps, scan
    bounds, incremental Go sort) as scalar C++ on ONE host core, over the same prepared tables -- what separates the algorithm's
    share of a speed-up from the hardware's.  New-NodeClaim provisioning shapes (C2, C3); never fatal for the bench."""
    try:
        best = None
        for _ in range(3):
            got = oracle_lib.cached_solve(problem)
            if got is None:
                return {"unavailable": "shape outside what oracle/orc_cached.cpp serves"}
            res, ms, prep = got
            best = ms if best is None else min(best, ms)
        same = all(np.array_equal(np.asarray(res[k]), np.asarray(gpu_res[k])) for k in oracle_lib.CACHED_KEYS)
        return {"value": n_pods / (best / 1000), "unit": "pods/s", "ms": best, "host_prep_ms": prep, "cores": 1, "kind": "cached port",
                "identical_to_the_gpu_result": bool(same),
                "sample": "the full workload, the CUDA solver's algorithm as scalar C++ on one host core, tables prepared before the "
                          "clock starts (best of 3)"}
    except Exception as e:  # noqa: BLE001 -- a baseline leg must not take the bench line down
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}


def time_encoder(n_pods_headline, e2e_ms):
    """The Python mirror's encoder on real Pod objects (the headline feeds class ids, as the cgo shim would after interning):
    200 apps x 1 000 replicas of C3's shape as `Pod` objects carrying their owner's template key, Scheduler.encode timed."""
    from karpenter_b200 import workloads
    from karpenter_b200.model import HOSTNAME_LABEL, ZONE_LABEL, LabelSelector, Pod, PodAffinityTerm, TopologySpreadConstraint
    from karpenter_b200.scheduler import Scheduler
    apps, reps = 200, 1000
    its = workloads.kwok.aws_instance_types(C3_ITS)
    pool = workloads.default_nodepool(zones=workloads.kwok.AWS_ZONES[:3])
    pods = []
    for a in range(apps):
        labels = {"app": f"app-{a:05d}"}
        sel = LabelSelector.of(labels)
        tsc = [TopologySpreadConstraint(1, ZONE_LABEL, sel)]
        anti = [PodAffinityTerm(sel, HOSTNAME_LABEL)]
        req = {"cpu": f"{250 * (1 + a % 4)}m", "memory": f"{256 * (1 + a % 6)}Mi"}
        for r in range(reps):
            pods.append(Pod(name=f"p{a}-{r}", uid=(a << 32) | r, labels=labels, requests=req, topology_spread_constraints=tsc,
                            pod_anti_affinity=anti, template=a))
    s = Scheduler([pool], {pool.name: its}, backend=lambda p: None)
    t0 = time.perf_counter()
    s.encode(pods)
    with_t = time.perf_counter() - t0
    for p in pods:
        p.template = None
    t0 = time.perf_counter()
    s.encode(pods[:50_000])
    without_t = (time.perf_counter() - t0) * len(pods) / 50_000
    rate = len(pods) / with_t
    return {"pods_per_s": rate, "pods_per_s_without_template_keys": len(pods) / without_t,
            "sample": f"{len(pods)} Pod objects ({apps} apps x {reps} replicas, C3's shape, {C3_ITS} instance types), "
                      "Scheduler.encode: catalog + NodePool + pods -> kp_problem; Pod.template = the owner's pod-template key",
            "e2e_with_encode_ms_extrapolated": e2e_ms + 1000.0 * n_pods_headline / rate,
            "note": "extrapolated to the headline's pod count from the sample's rate; the headline e2e starts from class ids"}


def peak_gbs():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0), "measured"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def time_provisioning(h, problem, n_pods, steps, warmup, torch, flush, barrier, sampler=None, e2e_steps=None):
    """W + K resident solves (device time from the library's CUDA events), then the same through kp_solve with host
    buffers.  Returns a dict of measurements + the last result."""
    h.upload(problem)
    dev_ms, wsolve_share, res, wall = [], None, None, None
    for i in range(warmup + steps):
        flush.zero_()  # evict the previous step's working set from L2
        torch.cuda.synchronize()  # the solve runs on the library's own stream: nothing of torch's may overlap it
        if i == warmup:
            barrier()
            if sampler is not None and not os.environ.get("KP_NO_SAMPLER"):
                sampler.start()
            wall = time.perf_counter()
        res = h.solve_resident()
        if i >= warmup:
            dev_ms.append(h.stats()["solve_ms"])
    barrier()
    wall = time.perf_counter() - wall
    if sampler is not None:
        sampler.stop_flag = True
    launches = h.stats()["kernel_launches"]
    e2e_t = []
    n_e2e = min(steps, 3) if e2e_steps is None else e2e_steps
    for i in range(1 + n_e2e):
        barrier()
        t0 = time.perf_counter()
        h.solve(problem)
        torch.cuda.synchronize()
        if i >= 1:
            e2e_t.append(time.perf_counter() - t0)
    st = h.stats()
    return {"ms": float(np.mean(dev_ms)), "ms_all": [round(float(x), 3) for x in dev_ms], "wall": wall,
            "launches_per_step": int(launches), "e2e_ms": 1000 * float(np.mean(e2e_t)), "stats": st, "res": res}


def roofline_block(res, n_pods, n_its, ms, key):
    peak, src = peak_gbs()
    balg = algorithmic_bytes(res, n_pods, n_its, res["n_groups"])
    achieved = balg / (ms / 1000) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": ncu_traffic(key), "kernel": "k_wsolve", "peak_source": src, "algorithmic_bytes": int(balg),
            "note": "B_alg = bytes the REFERENCE algorithm moves on this input (SURVEY 8d); k_wsolve is a latency-bound "
                    "serial first-fit chain (one warp per Scheduler) that skips provably failing candidates, so its "
                    "DRAM traffic is a few MB and the fraction measures chain speed, not bandwidth use; see DESIGN.md"}


def run_consolidation(args, h, rank, world, dist, torch):
    """C4: every <=3-node removal subset of the 100 cheapest-to-disrupt nodes of a 10k-node cluster holding 200k running
    pods (166 750 computeConsolidation calls).  Each rank evaluates the subsets s with s % world == rank; no collective
    on the data path, decisions would be gathered on rank 0."""
    from karpenter_b200 import _abi, sharding, workloads
    enc, consol = workloads.config_c4(n_nodes=args.consol_nodes, n_pods=args.consol_pods)
    S = consol["n_subsets"]
    off, nodes = consol["subset_off"], consol["subset_nodes"]
    ci = _abi.ConsolInput(**sharding.shard_subsets(consol, rank, world))
    dev_ms, e2e_ms = [], []
    res = None
    for i in range(1 + max(1, min(args.steps, 3))):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        res = h.consolidate(enc.problem, ci)  # host buffers in, decisions out: upload + kernels + download
        torch.cuda.synchronize()
        if i >= 1:
            e2e_ms.append(1000 * (time.perf_counter() - t0))
            dev_ms.append(res["solve_ms"])
    ms, e2e = float(np.mean(dev_ms)), float(np.mean(e2e_ms))
    decisions = np.bincount(res["decision"], minlength=3).astype(np.int64)
    if dist is not None:
        t = torch.tensor([ms, e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e = t.tolist()
        dt = torch.from_numpy(decisions).cuda()
        dist.all_reduce(dt)
        decisions = dt.cpu().numpy()
    if rank != 0:
        return None
    E = args.consol_nodes
    pods_per = (consol["node_pod_off"][1:] - consol["node_pod_off"][:-1])
    pods_sub = np.add.reduceat(pods_per[nodes], off[:-1])
    balg = int(pods_sub.sum()) * B_POD + int(((E - (off[1:] - off[:-1])) * pods_sub).sum()) * B_CLAIM  # SURVEY.md 8(d)
    peak, src = peak_gbs()
    traffic = ncu_traffic("c4_k_consolidate")
    roof = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": src, "kernel": "k_consolidate",
            "traffic": traffic, "reference_algorithm_bytes": int(balg),
            "note": "the reference re-reads every node row per pod per subset (reference_algorithm_bytes); "
                    "k_consolidate reads per-class candidate bitmaps and keeps per-subset state on chip, so the honest "
                    "roofline is its own DRAM traffic (ncu dram__bytes, profiles/) over its device time"}
    if traffic:
        roof["achieved"] = traffic / (ms / 1000) / 1e9
        roof["frac"] = roof["achieved"] / peak
    out = {"metric": "consolidation candidates/sec", "value": S / (ms / 1000), "unit": "subsets/s", "ms": ms,
           "workload": "C4: 10 000 existing KWOK nodes holding 200 000 running pods (bin-packed, 99 % of vCPU requested), "
                       "every <=3-node subset of the 100 nodes with the lowest disruption cost",
           "n_subsets": int(S), "nodes": int(E), "running_pods": int(enc.problem.get("n_pods")),
           "pods_per_subset": {"min": int(pods_sub.min()), "mean": float(pods_sub.mean()), "max": int(pods_sub.max())},
           "decisions": {"noop": int(decisions[0]), "delete": int(decisions[1]), "replace": int(decisions[2])},
           "e2e": {"value": S / (e2e / 1000), "unit": "subsets/s", "ms": e2e}, "roofline": roof}
    if not args.no_cpu_baseline and world == 1:
        from tests import oracle_lib
        threads = min(os.cpu_count() or 1, 32)
        n = min(S, 100 * threads)
        pick = np.linspace(0, S - 1, n).astype(np.int64)  # spread over singles, pairs and triples
        sizes = (off[1:] - off[:-1])[pick]
        smp = dict(consol, n_subsets=n, subset_off=np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32),
                   subset_nodes=np.concatenate([nodes[off[i]:off[i + 1]] for i in pick]).astype(np.int32))
        t0 = time.perf_counter()
        oracle_lib.consolidate(enc.problem, _abi.ConsolInput(**smp), threads=threads)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n / dt, "unit": "subsets/s", "cores": threads, "kind": "port",
                               "sample": f"{n} of the {S} subsets, evenly spaced (independent simulations, one per thread "
                                         f"at a time), {threads} of {os.cpu_count()} host cores"}
        try:  # the solver's own algorithm on ONE host core (oracle/orc_cached.cpp); never fatal for the bench
            got = oracle_lib.cached_consolidate(enc.problem, _abi.ConsolInput(**consol))
            if got is None:
                out["cpu_baseline_cached"] = {"unavailable": "shape outside what oracle/orc_cached.cpp serves"}
            else:
                cres, cms, cprep = got
                same = all(np.array_equal(np.asarray(cres[k]), np.asarray(res[k]))
                           for k in ("decision", "replacement_its", "n_new_claims", "n_unscheduled"))
                out["cpu_baseline_cached"] = {
                    "value": S / (cms / 1000), "unit": "subsets/s", "ms": cms, "host_prep_ms": cprep, "cores": 1, "kind": "cached port",
                    "identical_to_the_gpu_result": bool(same),
                    "sample": "all subsets, the CUDA path's algorithm (candidate bitmaps, failure bits, fast path, price lists) as "
                              "scalar C++ on one host core, one simulation after the other"}
        except Exception as e:  # noqa: BLE001
            out["cpu_baseline_cached"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    return out


def c5_shards(rank, world):
    """This rank's NodePool shards of C5: one kp_problem per pool (pool p lives on rank p mod N)."""
    from karpenter_b200 import sharding, workloads
    pools = sharding.pools_of_rank(C5_POOLS, rank, world)
    n_pods = int(os.environ.get("KP_C5_PODS", C5_PODS))
    return pools, workloads.config_c5_shards(n_pods=n_pods, n_pools=C5_POOLS, n_its=C5_ITS, app_replicas=1000,
                                             pool_groups=[[p] for p in pools]), n_pods


def time_c5(h, rank, world, steps, warmup, torch, dist, flush, barrier, sampler=None):
    """C5 on `world` GPUs: every rank solves its pools as one batch; the step ends with the library's all-reduce of the
    global domain-counter table.  Device time = the library's CUDA events around sort + solve + scatter + all-reduce."""
    from karpenter_b200 import _native, sharding
    pools, shards, n_total = c5_shards(rank, world)
    problems = [e.problem for e in shards]
    if world > 1:
        uid = [_native.Handle.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        h.comm_init(uid[0], rank, world)

    def upload():
        h.upload_batch(problems)
        slots = [h.counter_slots(i) for i in range(len(problems))]
        offs, total = sharding.instance_offsets(slots, rank, world, dist if world > 1 else None, device="cuda")
        h.set_counter_layout(total, offs)
        return total
    total_slots = upload()
    dev_ms, ar_ms, outs, wall = [], [], None, None
    for i in range(warmup + steps):
        flush.zero_()
        torch.cuda.synchronize()
        if i == warmup:
            barrier()
            if sampler is not None and not os.environ.get("KP_NO_SAMPLER"):
                sampler.start()
            wall = time.perf_counter()
        outs = h.solve_batch_resident()
        if i >= warmup:
            dev_ms.append(h.stats()["solve_ms"])
            ar_ms.append(h.last_allreduce_ms())
    barrier()
    wall = time.perf_counter() - wall
    if sampler is not None:
        sampler.stop_flag = True
    launches = h.stats()["kernel_launches"]
    table = h.global_counts()
    e2e_t = []
    for i in range(1 + (1 if world == 1 else max(1, min(steps, 2)))):
        barrier()
        t0 = time.perf_counter()
        upload()
        h.solve_batch_resident()
        torch.cuda.synchronize()
        if i >= 1:
            e2e_t.append(time.perf_counter() - t0)
    st = h.stats()
    return {"ms": float(np.mean(dev_ms)), "ms_all": [round(float(x), 3) for x in dev_ms], "allreduce_ms": float(np.mean(ar_ms)),
            "wall": wall, "launches_per_step": int(launches), "e2e_ms": 1000 * float(np.mean(e2e_t)), "stats": st,
            "outs": outs, "n_total": n_total, "pools": pools, "counter_slots": int(total_slots),
            "counter_sum": int(table.sum()), "n_mine": int(sum(int(p.n_pods) for p in problems)), "problems": problems}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="karpsolve")
    ap.add_argument("--apps", type=int, default=C3_APPS, help="C3 apps (1000 = BASELINE size; smaller only for quick checks)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-consolidation", action="store_true")
    ap.add_argument("--no-c2", action="store_true")
    ap.add_argument("--no-deployments", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--consol-nodes", type=int, default=10_000)
    ap.add_argument("--consol-pods", type=int, default=200_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's result of its last timed step as DIR/<name>.npy (float64, one file per "
                         "result array of the C ABI), so that two builds can be compared output for output")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (world > 1 or args.impl != "karpsolve"):
        ap.error("--dump-outputs writes the one-GPU headline (C3) of --impl karpsolve")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    from karpenter_b200 import _abi, _native, workloads
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    h = _native.Handle(local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    timing = ("CUDA events on the library stream around NewQueue sort + candidate bitmaps + solver kernel"
              " (+ counter scatter + ncclAllReduce when sharded), max over ranks")
    line = None
    if world == 1:
        # ---------------- headline: C3 at BASELINE size on one B200
        enc = workloads.config_c3(n_apps=args.apps, replicas=C3_REPLICAS, n_its=C3_ITS)
        n_pods = args.apps * C3_REPLICAS
        m = time_provisioning(h, enc.problem, n_pods, args.steps, args.warmup, torch, flush, barrier, sampler)
        res, st = m["res"], m["stats"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, res, _abi.PARITY_KEYS)
        name = C3_NAME if args.apps == C3_APPS else C3_NAME.replace("1M pods = 1000 apps", f"{n_pods} pods = {args.apps} apps")
        line = {
            "metric": "pods scheduled/sec", "value": n_pods / (m["ms"] / 1000), "unit": "pods/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": name, "n_pods": n_pods, "n_instance_types": C3_ITS, "parallelism": "1 Scheduler instance, 1 GPU",
                       "l2": "flushed between steps (256 MiB memset)", "timing": timing},
            "e2e": {"value": n_pods / (m["e2e_ms"] / 1000), "unit": "pods/s", "ms_per_step": m["e2e_ms"],
                    "h2d_bytes_per_step": int(st["bytes_h2d"]), "d2h_bytes_per_step": int(st["bytes_d2h"]),
                    "host_prep_ms": st["prep_ms"], "upload_ms": st["upload_ms"], "kernels_ms": st["solve_ms"],
                    "download_ms": st["download_ms"]},
            "gpu_launches": m["launches_per_step"] * args.steps,
            "roofline": roofline_block(res, n_pods, C3_ITS, m["ms"], "c3_k_wsolve"),
            "clocks": sampler.summary(),
            "unscheduled": int((res["pod_target"] == -1).sum()), "node_claims": int(res["n_claims"]),
            "us_per_pod": 1000 * m["ms"] / n_pods, "wall_s_timed_region": m["wall"], "ms_per_step_all": m["ms_all"],
        }
        if not args.no_cpu_baseline:
            from tests import oracle_lib
            oracle_lib.build()
            threads = oracle_threads()
            apps = min(60, args.apps)
            smp = c3_sample(apps)
            t0 = time.perf_counter()
            oracle_lib.solve(smp.problem, threads=threads)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": apps * C3_REPLICAS / dt, "unit": "pods/s", "cores": threads, "kind": "port",
                                    "sample": f"the first {apps} of the {args.apps} apps with all their {C3_REPLICAS} replicas "
                                              f"({apps * C3_REPLICAS} pods), one Solve, {threads} thread(s) (fastest of 1/8/16) "
                                              f"of {os.cpu_count()} host cores"}
            line["cpu_baseline_cached"] = cached_cpu_baseline(oracle_lib, enc.problem, n_pods, res)
        # ---------------- secondary: C2
        if not args.no_c2:
            enc2 = workloads.config_c2(n_pods=C2_PODS, n_its=C2_ITS)
            m2 = time_provisioning(h, enc2.problem, C2_PODS, args.steps, args.warmup, torch, flush, barrier)
            st2 = m2["stats"]
            c2 = {"workload": C2_NAME, "value": C2_PODS / (m2["ms"] / 1000), "unit": "pods/s", "ms_per_step": m2["ms"],
                  "us_per_pod": 1000 * m2["ms"] / C2_PODS, "ms_per_step_all": m2["ms_all"],
                  "e2e": {"value": C2_PODS / (m2["e2e_ms"] / 1000), "unit": "pods/s", "ms_per_step": m2["e2e_ms"],
                          "h2d_bytes_per_step": int(st2["bytes_h2d"]), "d2h_bytes_per_step": int(st2["bytes_d2h"])},
                  "roofline": roofline_block(m2["res"], C2_PODS, C2_ITS, m2["ms"], "c2_k_wsolve"),
                  "unscheduled": int((m2["res"]["pod_target"] == -1).sum()), "node_claims": int(m2["res"]["n_claims"])}
            if not args.no_cpu_baseline:
                t0 = time.perf_counter()
                oracle_lib.solve(enc2.problem, threads=threads)
                dt = time.perf_counter() - t0
                c2["cpu_baseline"] = {"value": C2_PODS / dt, "unit": "pods/s", "cores": threads, "kind": "port",
                                      "sample": f"the full workload ({C2_PODS} pods), one Solve, {threads} thread(s)"}
                c2["cpu_baseline_cached"] = cached_cpu_baseline(oracle_lib, enc2.problem, C2_PODS, m2["res"])
            line["c2"] = c2
        # ---------------- secondary: a Deployment-shaped queue (cohort commits) and the Python encoder on Pod objects
        if not args.no_deployments:
            encd = workloads.config_deployments(C3_APPS, C3_REPLICAS, n_its=C3_ITS, topology=True)
            md = time_provisioning(h, encd.problem, n_pods_dep := C3_APPS * C3_REPLICAS, 2, 1, torch, flush, barrier, e2e_steps=1)
            line["deployments"] = {
                "workload": "NOT a BASELINE config: 1 000 Deployments x 1 000 identical replicas with C3's constraints (zonal spread + "
                            "hostname anti-affinity), every Deployment with its own CPU request so that its pods stand together in the "
                            "queue; the solver's cohort instantiation commits runs of identical pods in one step",
                "value": n_pods_dep / (md["ms"] / 1000), "unit": "pods/s", "ms_per_step": md["ms"], "us_per_pod": 1000 * md["ms"] / n_pods_dep,
                "cohort_pods": int(md["stats"].get("cohort_pods", 0)), "node_claims": int(md["res"]["n_claims"]),
                "unscheduled": int((md["res"]["pod_target"] == -1).sum())}
            line["encoder"] = time_encoder(n_pods, m["e2e_ms"])
        # ---------------- secondary: C5's 8 NodePool shards as one batch on this GPU
        if not args.no_c5:
            m5 = time_c5(h, 0, 1, 1, 1, torch, None, flush, barrier)
            line["c5_one_gpu"] = {
                "workload": C5_NAME.replace("NodePool p on rank p mod N", "all 8 NodePool shards as ONE kp_solve_batch on this GPU, one CTA each"),
                "value": m5["n_total"] / (m5["ms"] / 1000), "unit": "pods/s", "ms_per_step": m5["ms"], "n_pods": m5["n_total"],
                "ms_per_step_all": m5["ms_all"], "counter_scatter_ms": m5["allreduce_ms"],
                "e2e": {"value": m5["n_total"] / (m5["e2e_ms"] / 1000), "unit": "pods/s", "ms_per_step": m5["e2e_ms"]},
                "counter_table_slots": m5["counter_slots"], "counter_table_sum": m5["counter_sum"],
                "node_claims": int(sum(int(o["n_claims"]) for o in m5["outs"])),
                "unscheduled": int(sum(int((o["pod_target"] == -1).sum()) for o in m5["outs"]))}
            if not args.no_cpu_baseline:
                try:  # the solver's own algorithm on ONE host core, pool after pool (oracle/orc_cached.cpp); never fatal
                    from tests import oracle_lib
                    tot_ms, same, per_pool = 0.0, True, []
                    for prob, gpu_out in zip(m5["problems"], m5["outs"]):
                        got = oracle_lib.cached_solve(prob)
                        if got is None:
                            raise RuntimeError("shape outside what oracle/orc_cached.cpp serves")
                        cres, cms, _ = got
                        tot_ms += cms
                        per_pool.append(round(cms, 1))
                        same = same and all(np.array_equal(np.asarray(cres[k]), np.asarray(gpu_out[k])) for k in oracle_lib.CACHED_KEYS)
                    line["c5_one_gpu"]["cpu_baseline_cached"] = {
                        "value": m5["n_total"] / (tot_ms / 1000), "unit": "pods/s", "ms": tot_ms, "ms_per_pool": per_pool, "cores": 1,
                        "kind": "cached port", "identical_to_the_gpu_result": bool(same),
                        "sample": "all 8 NodePool shards, one after the other on one host core (they are independent: 8 cores would "
                                  "take the time of the slowest pool)"}
                except Exception as e:  # noqa: BLE001
                    line["c5_one_gpu"]["cpu_baseline_cached"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    else:
        # ---------------- headline at N > 1: C5, NodePool -> rank, library-side all-reduce inside the timed step
        m5 = time_c5(h, rank, world, args.steps, args.warmup, torch, dist, flush, barrier, sampler)
        t = torch.tensor([m5["ms"], m5["e2e_ms"], m5["allreduce_ms"]], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms, ar_ms = t.tolist()
        agg = torch.tensor([sum(int(o["n_claims"]) for o in m5["outs"]),
                            sum(int((o["pod_target"] == -1).sum()) for o in m5["outs"]), m5["n_mine"],
                            int(m5["stats"]["bytes_h2d"]), int(m5["stats"]["bytes_d2h"]),
                            sum(int(o["n_existing_evals"] + o["n_inflight_evals"] + o["n_template_evals"]) for o in m5["outs"]),
                            sum(int(o["n_commits"]) for o in m5["outs"]), sum(int(o["n_groups"]) for o in m5["outs"])],
                           device="cuda", dtype=torch.int64)
        dist.all_reduce(agg)
        claims, unsched, n_all, h2d, d2h, evs, commits, ngroups = [int(x) for x in agg.tolist()]
        if rank == 0:
            assert n_all == m5["n_total"], (n_all, m5["n_total"])
            peak, src = peak_gbs()
            balg = n_all * B_POD + evs * B_CLAIM + commits * B_CLAIM + C5_ITS * B_IT * world + 2 * ngroups * 4 * 4
            achieved = balg / (ms / 1000) / 1e9
            line = {
                "metric": "pods scheduled/sec", "value": n_all / (ms / 1000), "unit": "pods/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": {"workload": C5_NAME, "n_pods": n_all, "n_instance_types": C5_ITS, "n_nodepools": C5_POOLS,
                           "parallelism": f"nodepool-shard: {C5_POOLS} pools over {world} ranks, one CTA per pool",
                           "collective": f"library ncclAllReduce(sum, int32) of the global topology-domain counter table, "
                                         f"{m5['counter_slots']} slots = {4 * m5['counter_slots']} bytes, inside the timed step",
                           "l2": "flushed between steps (256 MiB memset)", "timing": timing},
                "e2e": {"value": n_all / (e2e_ms / 1000), "unit": "pods/s", "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "note": "kp_upload_batch (host prep + H2D) + kp_solve_batch_resident (kernels + all-reduce + D2H) per step"},
                "gpu_launches": m5["launches_per_step"] * args.steps * world,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                             "frac": achieved / (peak * world), "traffic": None, "kernel": "k_wsolve_batch",
                             "peak_source": src, "algorithmic_bytes": int(balg),
                             "note": "aggregate over ranks; see the N=1 line and DESIGN.md for what the fraction means"},
                "clocks": sampler.summary(), "allreduce_ms": ar_ms, "counter_table_sum": m5["counter_sum"],
                "unscheduled": unsched, "node_claims": claims, "wall_s_timed_region": m5["wall"], "ms_per_step_all": m5["ms_all"],
            }
    # ---- second headline metric: consolidation candidates/sec (C4), subsets sharded round-robin across ranks
    consol = None
    if not args.no_consolidation:
        consol = run_consolidation(args, h, rank, world, dist if world > 1 else None, torch)
    if rank == 0:
        if consol is not None:
            line["consolidation"] = consol
        print(json.dumps(line))
    h.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
