#!/usr/bin/env python
"""bench.py — headline benchmark: rows/sec of TPC-H lineitem SeqScan + HashAggregate on B200 segments.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    (also writes the last timed step's result rows)

Workload (BASELINE.json configs[1]): Q1's scan + filter + GROUP BY (l_returnflag, l_linestatus) with its
8 aggregates (no ORDER BY) over a 10^8-row synthetic lineitem heap relation (16 columns, 32 KB pages,
17 GB) per GPU segment.  One step = one execution of the plan through the executor-node surface
(GgExecReScan + GgExecProcNode to end of stream, include/gg_executor.h — the boundary the reference's
ExecProcNode switch would call, execProcnode.c:925):
  value  pages already resident in HBM (the segment's buffer pool), result rows returned as slots
  e2e    the same plan with the pages in pinned HOST memory: H2D copies inside the timed region
N > 1 is weak scaling: every rank scans its own 10^8-row segment (DISTRIBUTED RANDOMLY) and the plan is the
reference's two-stage one (tpch500GB.out:1771-1782): Gather Motion <- Agg(FINAL) <- Redistribute Motion on the
group keys <- Agg(PARTIAL) <- SeqScan, the Motions moving device-resident group records over the C interconnect
(gg_ic_*, NCCL; rank = segment).  torch.distributed (gloo) only hands the NCCL id around and reduces timings
on the CPU: it never touches the data path.

Parity gate: before a value is printed, the result rows are compared with the CPU oracle over the same pages
(`parity` block; counts bit-exact, float8 aggregates within 1e-6 relative); a mismatch aborts the run.

`secondary`: the other BASELINE configurations, measured after the headline (outside its timed region), each with
its own roofline and parity statement — 10^9-row lineitem-narrow Q1, HashJoin lineitem ⋈ orders, the Redistribute-
HashJoin in strong-scaling form (fixed total rows at every N), a 10^8-key sort, and the headline plan on the
run-time-specialised and interpreter kernels.

The reference arm times the CPU executor restatement (oracle/, one thread per segment over all host
cores) on a bounded sample of the same workload.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from greengage_b200 import capi, tpch  # noqa: E402

METRIC = "rows_per_sec_lineitem_scan_hashagg"
UNIT = "rows/s"
BLCKSZ = capi.GG_BLCKSZ


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_quota():
    """CPUs the container may actually use (cgroup quota), or None: the affinity mask can be far wider than that."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return float(q) / float(per)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return q / per
    except Exception:
        pass
    return None


def cores_note(cores):
    q = cpu_quota()
    return "%d threads (affinity mask)%s" % (cores, "" if q is None else ", cgroup CPU quota %.1f" % q)


def gen_threads():
    q = cpu_quota()
    n = host_cores() if q is None else max(int(q + 0.5), 1)
    return max(1, min(n, 64))


def _cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def gpu_numa_cpus(device):
    """(NUMA node of the GPU, the CPUs of that node this process may run on), or None where that cannot be told: the PCI
    address of CUDA device `device` (cuda-python's runtime binding, else nvidia-smi) -> sysfs."""
    bus = None
    try:
        try:
            from cuda.bindings import runtime as cudart
        except Exception:
            from cuda import cudart
        err, b = cudart.cudaDeviceGetPCIBusId(32, device)
        if int(err) == 0:
            bus = (b.decode() if isinstance(b, bytes) else str(b)).strip("\x00").strip()
    except Exception:
        bus = None
    if not bus:
        try:
            bus = subprocess.check_output(["nvidia-smi", "-i", str(device), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                          text=True, timeout=20).strip()
        except Exception:
            return None
    try:
        dom, rest = bus.lower().split(":", 1)
        node = int(open("/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:], rest)).read())
        if node < 0:
            return None
        cpus = _cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read()) & set(os.sched_getaffinity(0))
        return (node, cpus) if cpus else None
    except Exception:
        return None


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy kernel)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


_random_rates = None


def random_access_rates():
    """What this GPU sustains for the random accesses of the hash kernels, measured now by build/gather_peak (scripts/
    gather_peak.cu: random 32-byte-entry gathers, CAS inserts and atomic pairs over a 2 GB table, nothing else in the kernel):
    {"gather_g_per_s", "cas_insert_g_per_s", "atomic_pair_g_per_s"} in 10^9 accesses per second, or None without the tool."""
    global _random_rates
    if _random_rates is None:
        _random_rates = {}
        exe = os.path.join(ROOT, "build", "gather_peak")
        if os.path.exists(exe):
            try:
                env = dict(os.environ)
                if "LOCAL_RANK" in env and "CUDA_VISIBLE_DEVICES" not in env:
                    env["CUDA_VISIBLE_DEVICES"] = env["LOCAL_RANK"]
                out = subprocess.run([exe, "2048", "2e8"], capture_output=True, timeout=120, env=env, text=True)
                d = json.loads(out.stdout.strip().splitlines()[-1])
                _random_rates = {"gather_g_per_s": max(d["gather_g_per_s"].values()), "cas_insert_g_per_s": d["cas_insert_g_per_s"],
                                 "atomic_pair_g_per_s": d["atomic_pair_g_per_s"], "table_bytes": d["table_bytes"],
                                 "source": "build/gather_peak (scripts/gather_peak.cu), this run"}
            except Exception as exc:
                _random_rates = {"error": "%s: %s" % (type(exc).__name__, exc)}
    return _random_rates if "gather_g_per_s" in _random_rates else None


def join_random_bound(stream_bytes_build, inserts, stream_bytes_probe, probes, build_ms, probe_ms, peak):
    """The join's bound when its random accesses are counted at the rate this GPU sustains for them instead of at streaming
    bandwidth: build = inner pages at copy bandwidth + one CAS insert per inner row; probe = outer pages at copy bandwidth +
    one 32-byte table entry per outer row (the load factor's extra steps are the kernel's business).  The two terms of each are
    ADDED (both draw on the same HBM), so frac_of_bound can exceed what a kernel overlapping them perfectly would show."""
    rr = random_access_rates()
    if not rr:
        return None
    b_ms = stream_bytes_build / (peak * 1e9) * 1e3 + inserts / (rr["cas_insert_g_per_s"] * 1e9) * 1e3
    p_ms = stream_bytes_probe / (peak * 1e9) * 1e3 + probes / (rr["gather_g_per_s"] * 1e9) * 1e3
    out = {"rates": rr, "build_bound_ms": b_ms, "probe_bound_ms": p_ms}
    if build_ms:
        out["build_frac_of_bound"] = b_ms / build_ms
    if probe_ms:
        out["probe_frac_of_bound"] = p_ms / probe_ms
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, device):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def has_sample(self):
        try:
            return os.path.getsize(self.path) > 0
        except OSError:
            return False

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in open(self.path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


# --------------------------------------------------------------------------------------------------------------------
# reference arm: the CPU executor restatement on the host cores
# --------------------------------------------------------------------------------------------------------------------

def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = host_cores()
    table = capi.TAB_LINEITEM_NARROW if args.table == "narrow" else capi.TAB_LINEITEM_WIDE
    # bounded sample (a rate, so the sample need not grow with N): a few seconds of CPU work per step; <= 34 GB of pages
    rows = int(min(args.rows * min(max(world, 1), 2), 8_000_000 * cores, 200_000_000))
    t0 = time.time()
    total_secs = 0.0
    from oracle import pyoracle as po
    spec = tpch.synth_spec(table, rows)
    pages, nb, nr = tpch.synth_generate(spec, nthreads=gen_threads())
    scan, part, pool = tpch.q1_plan(table, capi.AGGSTAGE_PARTIAL)
    fin = tpch.q1_final_agg(part)
    for i in range(args.warmup + args.steps):
        out, secs, scanned = po.seqscan_agg_mt(scan, part, fin, pool, pages, cores)
        if i >= args.warmup:
            total_secs += secs
    value = nr * args.steps / total_secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * total_secs / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "Q1 scan+filter+hashagg (no ORDER BY), lineitem-%s, %d rows/GPU" % (args.table, args.rows),
                   "sample_rows": nr, "threads": cores,
                   "sample_note": "a rate measured on a bounded sample: at most 2x10^8 rows whatever N is (the CPU arm's rows/s does not depend on N)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d of the workload's rows, one oracle thread (= CPU segment) per host core, pages in RAM; %s" % (nr, cores_note(cores))},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "setup_s": round(time.time() - t0 - total_secs, 1),
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------------
# plumbing between the ranks (never on the data path)
# --------------------------------------------------------------------------------------------------------------------

class Plumbing:
    """torch.distributed over gloo, CPU tensors only: hands the NCCL unique id of the C interconnect around, reduces
    timings, gathers the oracle's rows for the parity check.  With one rank nothing is imported."""

    def __init__(self, world):
        self.world = world
        self.dist = None
        if world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")
            import torch
            import torch.distributed as dist
            self.torch, self.dist = torch, dist
            dist.init_process_group("gloo")

    def bcast_obj(self, obj, src=0):
        if self.dist is None:
            return obj
        box = [obj]
        self.dist.broadcast_object_list(box, src)
        return box[0]

    def gather_obj(self, obj):
        """every rank's object, on rank 0 (None elsewhere)"""
        if self.dist is None:
            return [obj]
        out = [None] * self.world if self.dist.get_rank() == 0 else None
        self.dist.gather_object(obj, out, 0)
        return out

    def reduce(self, x, op):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------------------------
# parity helpers
# --------------------------------------------------------------------------------------------------------------------

def b2f(v):
    return np.int64(v).view(np.float64).item()


def q1_rows_from_slots(rows):
    """Executor.rows() of the Q1 plan -> {(flag, status): ([7 float8 aggregates], count)}"""
    return {(v[0], v[1]): ([b2f(v[2 + i]) for i in range(7)], int(v[9])) for v, nl, ty, ln in rows}


def q1_rows_from_oracle(rows):
    return {(r.key[0], r.key[1]): ([r.agg[i].f[0] for i in range(7)], int(r.agg[7].i)) for r in rows}


def q1_combine(parts):
    """combine per-segment one-stage answers: sums add, counts add, avg = sum(avg_i * n_i) / sum(n_i)"""
    out = {}
    for p in parts:
        for k, (f, n) in p.items():
            if k not in out:
                out[k] = ([0.0] * 7, 0)
            g, m = out[k]
            for i in range(4):
                g[i] += f[i]
            for i in range(4, 7):
                g[i] += f[i] * n
            out[k] = (g, m + n)
    for k, (g, m) in out.items():
        for i in range(4, 7):
            g[i] = g[i] / m if m else float("nan")
    return out


Q1_COLUMNS = ("l_returnflag", "l_linestatus", "sum_qty", "sum_base_price", "sum_disc_price", "sum_charge", "avg_qty", "avg_price",
              "avg_disc", "count_order")


def dump_q1_rows(rows, outdir):
    """Executor.rows() of the Q1 plan -> outdir/<output column>.npy, float64, one entry per group in (l_returnflag, l_linestatus)
    order, since a hash aggregate hands its groups up in no fixed order.  The two keys are stored as their character codes, the
    float8 aggregates bit for bit, count(*) exactly (float64 holds integers up to 2^53).  So two builds, run with the same
    arguments over the same seeded relation, can be compared column by column."""
    groups = sorted((capi.unpack_str(v[0], ln[0]), capi.unpack_str(v[1], ln[1]), [b2f(v[2 + i]) for i in range(7)], int(v[9]))
                    for v, nl, ty, ln in rows)
    os.makedirs(outdir, exist_ok=True)
    cols = [[ord(g[0]) for g in groups], [ord(g[1]) for g in groups]] + [[g[2][i] for g in groups] for i in range(7)] + [[g[3] for g in groups]]
    for name, col in zip(Q1_COLUMNS, cols):
        np.save(os.path.join(outdir, name + ".npy"), np.array(col, dtype=np.float64))


def q1_compare(got, want, tol=1e-6):
    """-> parity dict; counts and keys bit-exact, float8 aggregates within tol relative"""
    ok = set(got) == set(want)
    counts_equal = ok and all(got[k][1] == want[k][1] for k in want)
    worst = 0.0
    if ok:
        for k in want:
            for a, b in zip(got[k][0], want[k][0]):
                worst = max(worst, abs(a - b) / abs(b) if b else abs(a))
    return {"checked": True, "rows": len(want), "keys_equal": ok, "counts_equal": bool(counts_equal), "max_rel_err": worst,
            "tolerance": tol, "ok": bool(ok and counts_equal and worst <= tol)}


# --------------------------------------------------------------------------------------------------------------------
# main arm
# --------------------------------------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--rows", type=float, default=1e8, help="rows per GPU segment")
    ap.add_argument("--table", default="wide", choices=["wide", "narrow"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="profiling runs only: the line then carries parity.checked = false")
    ap.add_argument("--secondary", default="all", help="all | none | comma list of narrow,join,rjoin,sort,paths,aocs,groupby,motion")
    ap.add_argument("--narrow-rows", type=float, default=1e9)
    ap.add_argument("--rjoin-rows", type=float, default=2e8, help="lineitem rows of the Redistribute-HashJoin, TOTAL over all GPUs")
    ap.add_argument("--rjoin-child", default=None, help=argparse.SUPPRESS)      # internal: see rjoin_in_children
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result rows of the last timed step as DIR/<output column>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.rows = int(args.rows)
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    from greengage_b200 import executor as ex
    from greengage_b200.engine import Engine, Interconnect, Relation, host_alloc, host_free

    plumb = Plumbing(world)
    device = local_rank
    eng = Engine(device)
    ic = None
    if world > 1:
        uid = plumb.bcast_obj(Interconnect.unique_id() if rank == 0 else None)
        ic = Interconnect(eng, world, rank, uid)
    table = capi.TAB_LINEITEM_NARROW if args.table == "narrow" else capi.TAB_LINEITEM_WIDE
    nthreads = max(1, gen_threads() // world) if world > 1 else gen_threads()

    def barrier():
        plumb.barrier()
        eng.sync()
        if ic is not None:
            ic.allgather_u64(0)               # device-side barrier on the engine's stream
            eng.sync()

    if args.rjoin_child:
        # one of the child processes of rjoin_in_children: this measurement and nothing else.  Should it hang, where it hangs is
        # in its log shortly before the parent gives up on it.
        import faulthandler
        faulthandler.dump_traceback_later(max(10, int(os.environ.get("GGB200_RJOIN_TIMEOUT", "180")) - 10), exit=False)
        ctx = dict(eng=eng, ic=ic, plumb=plumb, rank=rank, world=world, rel=None, nb=0, nr=0, args=args, barrier=barrier,
                   nthreads=nthreads, table=table, hview=None)
        try:
            r = sec_rjoin(ctx)
        except Exception as exc:
            r = {"error": "%s: %s" % (type(exc).__name__, exc)}
        if rank == 0:
            with open(args.rjoin_child + ".tmp", "w") as f:
                json.dump(r, f)
            os.replace(args.rjoin_child + ".tmp", args.rjoin_child)
        if ic is not None:
            ic.close()
        eng.close()
        plumb.close()
        return

    # ---- the segment's relation: generated on the host (pinned), loaded into HBM ----
    # The pinned buffer is what the end-to-end path copies from every step: it should live in the memory of the GPU's own NUMA
    # node (round 1's N = 8 run moved 34 GB/s per GPU instead of 55 with every rank's buffer wherever its main thread happened to
    # run).  Pages are placed where the thread that pins them runs, so this process runs on the GPU's node while it allocates and
    # fills the buffer, and gets its full mask back afterwards (the CPU baseline and the parity oracle use every core).
    numa = gpu_numa_cpus(device)
    full_mask = None
    if numa is not None:
        try:
            full_mask = os.sched_getaffinity(0)
            os.sched_setaffinity(0, numa[1])
        except Exception:
            numa, full_mask = None, None
    t_setup = time.time()
    spec = tpch.synth_spec(table, args.rows * world, nsegs=world, seg=rank)
    nb, nr = tpch.synth_measure(spec, nthreads)
    nbytes = nb * BLCKSZ
    pinned = True
    try:
        haddr, hview = host_alloc(nbytes)
    except Exception:
        pinned = False
        hview = np.empty(nbytes, dtype=np.uint8)
        haddr = hview.ctypes.data
    tpch.synth_generate(spec, out=haddr, nthreads=nthreads, measured=(nb, nr))
    rel = Relation(eng, nblocks=nb)
    rel.load(0, hview)
    eng.sync()
    setup_s = time.time() - t_setup
    if full_mask is not None:
        os.sched_setaffinity(0, full_mask)

    b = ex.PlanBuilder()
    plan, pool = tpch.q1_exec_plan(b, table, two_stage=world > 1)
    x = ex.Executor(eng, pool, [rel], plan, nsegs=world, segindex=rank, interconnect=ic)
    plan_text = "Agg(NORMAL)<-SeqScan" if world == 1 else "Gather<-Agg(FINAL)<-Redistribute<-Agg(PARTIAL)<-SeqScan"

    scan_ms_tot, scan_launches = 0.0, 0
    last_rows = [0]
    kept_rows = None

    def step_resident(keep=False):
        """keep: hand the rows up as Python lists (kept_rows) instead of only counting them; 4 rows, microseconds"""
        nonlocal scan_ms_tot, scan_launches, kept_rows
        x.rescan()
        if keep:
            kept_rows = x.rows()
            last_rows[0] = len(kept_rows)
        else:
            last_rows[0] = x.drain()
        ms, k, _, _ = x.kernel_ms()
        scan_ms_tot += ms
        scan_launches += k

    # ---- resident: W warm-up steps, then exactly K timed steps ----
    # The clock sampler (nvidia-smi) is started first and the GPU is kept under load, untimed, until its first line is
    # out: NVML initialisation can stall CUDA calls for hundreds of milliseconds, which must not land in the K steps.
    sampler = ClockSampler(device) if rank == 0 else None
    t_pre = time.time()
    while True:
        more = 1 if (rank == 0 and sampler.proc is not None and not sampler.has_sample() and time.time() - t_pre < 8.0) else 0
        more = int(plumb.bcast_obj(more))
        if not more:
            break
        step_resident()
    for _ in range(args.warmup):
        step_resident()
    scan_ms_tot, scan_launches = 0.0, 0
    barrier()
    l0 = eng.launch_count()
    eng.timer_start()
    for i in range(args.steps):
        step_resident(keep=args.dump_outputs is not None and i == args.steps - 1)
    ms = eng.timer_stop()
    barrier()
    launches = eng.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    ms = plumb.reduce(ms, "max")
    total_rows = plumb.reduce(float(nr), "sum")
    value = total_rows * args.steps / (ms / 1000.0)
    scan_ms = scan_ms_tot / max(scan_launches, 1)
    variant = x.kernel_ms()[2]
    result_rows = last_rows[0]
    if args.dump_outputs is not None and rank == 0:
        dump_q1_rows(kept_rows, args.dump_outputs)

    # ---- end to end: pages start in host memory every step (same plan, the relation given as host pages) ----
    e2e = None
    if not args.no_e2e:
        be = ex.PlanBuilder()
        plan_e, pool_e = tpch.q1_exec_plan(be, table, two_stage=world > 1)
        xe = ex.Executor(eng, pool_e, [(haddr, nb)], plan_e, nsegs=world, segindex=rank, interconnect=ic)
        xe.drain()
        barrier()
        eng.timer_start()
        nres = 0
        for _ in range(args.e2e_steps):
            xe.rescan()
            nres = xe.drain()
        ems = plumb.reduce(eng.timer_stop(), "max")
        barrier()
        xe.end()
        e2e = {"value": total_rows * args.e2e_steps / (ems / 1000.0), "unit": UNIT,
               "h2d_bytes_per_step": int(plumb.reduce(float(nbytes), "sum")),
               "d2h_bytes_per_step": int((max(nres, result_rows) * C.sizeof(capi.gg_aggrow) + 64) * max(world, 1)),
               "steps": args.e2e_steps, "ms_per_step": ems / args.e2e_steps,
               "host_memory": "pinned" if pinned else "pageable",
               "api": "GgExecInitNode/GgExecProcNode over a relation in host memory (GgEState.host_pages)"}

    # ---- parity gate + CPU baseline: the oracle over (a bounded prefix of) the very pages the GPU scanned ----
    parity = {"checked": False}
    cpu = None
    want_oracle = (not args.no_parity) or (world == 1 and not args.no_cpu_baseline)
    if want_oracle:
        from oracle import pyoracle as po
        cores = host_cores()
        threads = max(1, cores // world)
        sample_rows = int(min(nr, 4_000_000 * threads))
        sample_nb = nb if sample_rows >= nr else max(1, int(nb * (sample_rows / nr)))
        scan_o, part_o, pool_o = tpch.q1_plan(table, capi.AGGSTAGE_PARTIAL)
        fin_o = tpch.q1_final_agg(part_o)
        orows, secs, oscanned = po.seqscan_agg_mt(scan_o, part_o, fin_o, pool_o, hview[:sample_nb * BLCKSZ], threads)
        if world == 1 and not args.no_cpu_baseline:
            cpu = {"value": oscanned / secs, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": "%d of the workload's %d rows (the first %d of %d pages), one oracle thread (= one CPU segment) per host core, pages in RAM; %s"
                             % (oscanned, nr, sample_nb, nb, cores_note(cores))}
        if not args.no_parity:
            # the GPU answer over the same pages: the timed plan itself when the sample is the whole relation, else the same
            # plan over the prefix (an attached view of the resident pages)
            if sample_nb == nb:
                xp, sub = x, None
            else:
                sub = Relation(eng, nblocks=sample_nb, device_ptr=rel.device_ptr())
                bp = ex.PlanBuilder()
                plan_p, pool_p = tpch.q1_exec_plan(bp, table, two_stage=world > 1)
                xp = ex.Executor(eng, pool_p, [sub], plan_p, nsegs=world, segindex=rank, interconnect=ic)
            xp.rescan()
            grows = xp.rows()
            if sub is not None:
                xp.end()
                sub.free()
            parts = plumb.gather_obj((q1_rows_from_oracle(orows), oscanned))
            if rank == 0:
                want = q1_combine([p for p, _ in parts])
                parity = q1_compare(q1_rows_from_slots(grows), want)
                parity["rows_checked"] = int(sum(n for _, n in parts))
                parity["of_rows"] = int(total_rows)
                parity["how"] = "GPU plan result vs the CPU oracle over the same heap pages (every segment's first %d of %d pages)" % (sample_nb, nb)
                parity["count_sum"] = int(sum(c for _, c in want.values()))
            ok = plumb.bcast_obj(parity.get("ok", False) if rank == 0 else None)
            if not ok:
                if rank == 0:
                    print("PARITY FAILURE: " + json.dumps(parity), file=sys.stderr, flush=True)
                sys.exit(3)

    # ---- the other BASELINE configurations ----
    secondary = {}
    want_sec = [] if args.secondary == "none" else (["join", "paths", "aocs", "rjoin", "narrow", "sort", "groupby", "motion"] if args.secondary == "all" else args.secondary.split(","))
    ctx = dict(eng=eng, ic=ic, plumb=plumb, rank=rank, world=world, rel=rel, nb=nb, nr=nr, args=args, barrier=barrier,
               nthreads=nthreads, table=table, hview=hview)
    for name in want_sec:
        if world > 1 and name != "rjoin":
            continue
        if name == "narrow":
            # the 76 GB relation wants the headline's HBM (and nothing after it needs the wide relation)
            x.end(); x = None
            rel.free(); rel = None
            ctx["rel"] = None
        try:
            t0 = time.time()
            r = rjoin_in_children(args, rank, world) if (name == "rjoin" and world > 1) else SECONDARY[name](ctx)
            if r is not None and rank == 0:
                r["wall_s"] = round(time.time() - t0, 1)
                secondary[name] = r
        except Exception as exc:      # a secondary measurement never takes the headline down
            if rank == 0:
                secondary[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        barrier()

    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = nbytes / (scan_ms / 1000.0) / 1e9 if scan_ms > 0 else 0.0
        traffic, traffic_src = None, None
        for tp in ("r2_scanagg_traffic.json", "r1_scanagg_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", tp)
            if os.path.exists(tpath) and world == 1:
                try:
                    tj = json.load(open(tpath))
                    if tj.get("table") == args.table:
                        traffic = tj["dram_bytes_per_block"] * nb
                        traffic_src = "profiles/%s (ncu --set full of this kernel, bytes per page x pages)" % tp
                        break
                except Exception:
                    pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "Q1 scan+filter+hashagg (no ORDER BY), lineitem-%s, %d rows/GPU" % (args.table, args.rows),
                       "rows_per_gpu": nr, "blocks_per_gpu": nb, "bytes_per_gpu": nbytes,
                       "l2": "input %.1f GB per GPU >> 126 MB L2, streamed once per step" % (nbytes / 1e9),
                       "plan": plan_text, "api": "GgExecReScan + GgExecProcNode to end of stream (libggexec.so)",
                       "interconnect": "gg_ic_* over NCCL (C)" if world > 1 else "none",
                       "kernel_variant": variant, "result_rows": result_rows,
                       "host_numa": None if numa is None else {"node": numa[0], "cpus": len(numa[1]),
                                                               "note": "pinned host buffer allocated and filled on the GPU's NUMA node"}},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": "gg scan+agg (TMA page ring)", "kernel_ms": scan_ms,
                         "algorithmic_bytes": nbytes, "peak_source": peak_src},
            "parity": parity,
            "gpu_launches": int(launches), "clocks": clocks, "setup_s": round(setup_s, 1),
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if secondary:
            line["secondary"] = secondary
        print(json.dumps(line), flush=True)

    if x is not None:
        x.end()
    if rel is not None:
        rel.free()
    if pinned:
        host_free(haddr)
    if ic is not None:
        ic.close()
    eng.close()
    plumb.close()


# --------------------------------------------------------------------------------------------------------------------
# secondary measurements
# --------------------------------------------------------------------------------------------------------------------

def rjoin_in_children(args, rank, world, timeout_s=None):
    """At N > 1 the Redistribute-HashJoin is measured in child processes — one per rank on the rank's GPU, with their own gloo
    group and their own NCCL communicator — so that a fault there (an exchange that never completes) costs this entry and not the
    headline line: a child that does not come back within timeout_s is killed.  The numbers are the child's own CUDA-event
    timings, max over ranks, exactly as sec_rjoin takes them."""
    if timeout_s is None:
        timeout_s = int(os.environ.get("GGB200_RJOIN_TIMEOUT", "180"))
    port = int(os.environ.get("MASTER_PORT", "29500"))
    out = os.path.join(tempfile.gettempdir(), "ggb200_rjoin_%d.json" % port)
    log = os.path.join(tempfile.gettempdir(), "ggb200_rjoin_%d_rank%d.err" % (port, rank))
    if rank == 0 and os.path.exists(out):
        os.remove(out)
    env = dict(os.environ)
    env["MASTER_PORT"] = str(port + 173 if port + 173 < 65000 else port - 173)
    env.pop("TORCHELASTIC_USE_AGENT_STORE", None)        # the children's rank 0 hosts their store itself
    cmd = [sys.executable, os.path.abspath(__file__), "--gpus", str(world), "--rjoin-child", out, "--rjoin-rows", repr(float(args.rjoin_rows))]
    with open(log, "w") as lf:
        proc = subprocess.Popen(cmd, env=env, stdout=subprocess.DEVNULL, stderr=lf)
        try:
            rc = proc.wait(timeout=timeout_s)
            note = None if rc == 0 else "child exited with %d" % rc
        except subprocess.TimeoutExpired:
            proc.kill()
            proc.wait()
            note = "no answer within %d s: the child processes were killed" % timeout_s
    if rank != 0:
        return None
    if os.path.exists(out):
        with open(out) as f:
            r = json.load(f)
        r["isolation"] = "child processes (one per rank), own NCCL communicator"
        return r
    tails = []
    for r in range(world):            # one box: every rank's log is in the same temporary directory
        try:
            t = open(os.path.join(tempfile.gettempdir(), "ggb200_rjoin_%d_rank%d.err" % (port, r))).read().strip()
            if t:
                tails.append("rank %d: %s" % (r, t[-700:]))
        except Exception:
            pass
    return {"error": (note or "the child wrote no result") + ((" | " + " | ".join(tails)) if tails else "")}


def _timed_steps(ctx, x, steps=5, warmup=3):
    """(ms per step: max over ranks of the CUDA-event time of `steps` executions, rows the last one returned, launches per step)"""
    eng, plumb = ctx["eng"], ctx["plumb"]
    n = 0
    for _ in range(warmup):
        x.rescan()
        n = x.drain()
    ctx["barrier"]()
    l0 = eng.launch_count()
    eng.timer_start()
    for _ in range(steps):
        x.rescan()
        n = x.drain()
    ms = eng.timer_stop()
    launches = (eng.launch_count() - l0) / steps
    ctx["barrier"]()
    return plumb.reduce(ms, "max") / steps, n, launches


def _load_shards(ctx, table, total, norders=None, chunk_rows=25_000_000):
    """This rank's share of a `total`-row table as one resident relation, generated and loaded shard by shard through one
    reusable host buffer (the shards of a DISTRIBUTED RANDOMLY table are independent: spec.nsegs / spec.seg)."""
    from greengage_b200.engine import Relation
    eng, world, rank, nthreads = ctx["eng"], ctx["world"], ctx["rank"], ctx["nthreads"]
    per_rank = (total + world - 1) // world
    K = max(1, int((per_rank + chunk_rows - 1) // chunk_rows))
    specs = [tpch.synth_spec(table, total, nsegs=world * K, seg=rank * K + j, norders=norders) for j in range(K)]
    sizes = [tpch.synth_measure(s, nthreads) for s in specs]
    rel = Relation(eng, nblocks=sum(nb for nb, _ in sizes))
    buf = np.empty(max(nb for nb, _ in sizes) * BLCKSZ, dtype=np.uint8)
    off = 0
    for s, (nb, nr) in zip(specs, sizes):
        tpch.synth_generate(s, out=buf.ctypes.data, nthreads=nthreads, measured=(nb, nr))
        rel.load(off, buf[:nb * BLCKSZ])
        eng.sync()
        off += nb
    return rel, off, sum(nr for _, nr in sizes)


def _join_small_parity(ctx, table, redistribute):
    """The same plan shape on tables the oracle joins in a second: 2x10^6 lineitem rows x 5x10^5 orders over all ranks,
    GPU plan result vs or_hashjoin_agg on rank 0 (count and sum(o_custkey) bit-exact, sum(l_extendedprice) within 1e-6)."""
    from greengage_b200 import executor as ex
    from greengage_b200.engine import Relation
    from oracle import pyoracle as po
    eng, world, rank, ic = ctx["eng"], ctx["world"], ctx["rank"], ctx["ic"]
    nl, no = 2_000_000, 500_000
    li, _, _ = tpch.synth_generate(tpch.synth_spec(table, nl, seed=7, norders=no, nsegs=world, seg=rank), nthreads=ctx["nthreads"])
    od, _, _ = tpch.synth_generate(tpch.synth_spec(capi.TAB_ORDERS, no, seed=7, nsegs=world, seg=rank), nthreads=ctx["nthreads"])
    b = ex.PlanBuilder()
    plan, pool, _, _ = tpch.rjoin_exec_plan(b, "survey", table=table, redistribute=redistribute)
    rels = [Relation(eng, host_pages=li), Relation(eng, host_pages=od)]
    x = ex.Executor(eng, pool, rels, plan, nsegs=world, segindex=rank, interconnect=ic)
    rows = x.rows()
    x.end()
    for r in rels:
        r.free()
    out = None
    if rank == 0:
        fl, _, _ = tpch.synth_generate(tpch.synth_spec(table, nl, seed=7, norders=no), nthreads=ctx["nthreads"])
        fo, _, _ = tpch.synth_generate(tpch.synth_spec(capi.TAB_ORDERS, no, seed=7), nthreads=ctx["nthreads"])
        outer, inner, hj, agg, opool = tpch.join_plan(table, "survey", capi.JOIN_INNER)
        want, nj = po.hashjoin_agg(outer, inner, hj, agg, opool, fl, fo)
        v, w = rows[0][0], want[0]
        rel_err = abs(b2f(v[2]) - w.agg[2].f[0]) / abs(w.agg[2].f[0])
        out = {"checked": True, "how": "same plan over 2x10^6 x 5x10^5 rows vs the CPU oracle's hash join",
               "count_equal": bool(v[0] == w.agg[0].i == nj), "int_sum_equal": bool(v[1] == w.agg[1].i), "max_rel_err": rel_err,
               "ok": bool(v[0] == w.agg[0].i == nj and v[1] == w.agg[1].i and rel_err <= 1e-6)}
    return out


def sec_join(ctx):
    """BASELINE configs[2]: HashJoin lineitem ⋈ orders on l_orderkey (int64), 10^8 LI-wide x 2.5x10^7 orders, one GPU.
    SELECT count(*), sum(o_custkey), sum(l_extendedprice) (SURVEY §8d) through Agg <- HashJoin(SeqScan, Hash(SeqScan))."""
    from greengage_b200 import executor as ex
    eng, rel, nb, nr = ctx["eng"], ctx["rel"], ctx["nb"], ctx["nr"]
    if ctx["table"] != capi.TAB_LINEITEM_WIDE:
        return None
    norders = max(ctx["args"].rows // 4, 1)              # the key space the headline relation's l_orderkey draws from
    t0 = time.time()
    od, onb, onr = _load_shards(ctx, capi.TAB_ORDERS, norders)
    setup = time.time() - t0
    outer, inner, hj, agg, pool = tpch.join_plan(capi.TAB_LINEITEM_WIDE, "survey", capi.JOIN_INNER)
    b = ex.PlanBuilder()
    plan = b.agg(b.hashjoin(b.seqscan(0, outer.desc, outer.qual), b.hash(b.seqscan(1, inner.desc, inner.qual)), hj), agg)
    x = ex.Executor(eng, pool, [rel, od], plan)
    ms, n, launches = _timed_steps(ctx, x)
    probe_ms, _, variant, build_ms = x.kernel_ms()
    x.rescan()
    rows = x.rows()
    x.end()
    od.free()
    v = rows[0][0]
    peak, _ = measured_peak()
    algo = nb * BLCKSZ + onb * BLCKSZ + 16 * onr + 32 * nr
    par = _join_small_parity(ctx, capi.TAB_LINEITEM_WIDE, redistribute=False)
    par["full_size_property"] = {"rows_joined": int(v[0]), "outer_rows": int(nr), "fk_join_count_equals_outer_rows": bool(v[0] == nr)}
    par["ok"] = bool(par["ok"] and v[0] == nr)
    return {"workload": "HashJoin lineitem-wide ⋈ orders on l_orderkey (int64): %d x %d rows; count(*), sum(o_custkey), sum(l_extendedprice)" % (nr, onr),
            "plan": "Agg<-HashJoin(SeqScan, Hash(SeqScan))", "api": "GgExecProcNode",
            "ms": ms, "build_ms": build_ms, "probe_ms": probe_ms, "rows_per_s": (nr + onr) / (ms / 1e3), "probe_rows_per_s": nr / (probe_ms / 1e3),
            "kernel_variant": variant, "gpu_launches_per_step": launches,
            "roofline": {"bound": "hbm", "algorithmic_bytes": algo, "achieved": algo / ((build_ms + probe_ms) / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / ((build_ms + probe_ms) / 1e3) / 1e9 / peak,
                         "probe_frac": (nb * BLCKSZ + 32 * nr) / (probe_ms / 1e3) / 1e9 / peak,
                         "build_frac": (onb * BLCKSZ + 16 * onr) / (build_ms / 1e3) / 1e9 / peak,
                         "note": "SURVEY §8d: both relations' pages once + 16 B/inner row written + one 32 B table sector per probe, over build + probe kernel time",
                         "random_access_bound": join_random_bound(onb * BLCKSZ, onr, nb * BLCKSZ, nr, build_ms, probe_ms, peak)},
            "parity": par, "setup_s": round(setup, 1)}


def sec_rjoin(ctx):
    """BASELINE configs[3]: Redistribute Motion on the join key (both sides) + HashJoin + two-stage Agg, STRONG scaling: the
    total (--rjoin-rows lineitem-wide rows, a quarter as many orders) is the same at every N, each rank holds 1/N of it
    (DISTRIBUTED RANDOMLY), so value(N) / value(1) is the speed-up of the north star's >= 6x bar."""
    from greengage_b200 import executor as ex
    eng, world, rank, ic, plumb = ctx["eng"], ctx["world"], ctx["rank"], ctx["ic"], ctx["plumb"]
    T = int(ctx["args"].rjoin_rows)
    TO = max(T // 4, 1)
    t0 = time.time()
    li, lnb, lnr = _load_shards(ctx, capi.TAB_LINEITEM_WIDE, T, norders=TO)
    od, onb, onr = _load_shards(ctx, capi.TAB_ORDERS, TO)
    setup = time.time() - t0
    b = ex.PlanBuilder()
    plan, pool, lt, ot = tpch.rjoin_exec_plan(b, "survey", table=capi.TAB_LINEITEM_WIDE, redistribute=True)
    x = ex.Executor(eng, pool, [li, od], plan, nsegs=world, segindex=rank, interconnect=ic)
    ms, n, launches = _timed_steps(ctx, x)
    probe_ms, _, variant, build_ms = x.kernel_ms()
    x.rescan()
    rows = x.rows()
    x.end()
    li.free()
    od.free()
    tot_li = plumb.reduce(float(lnr), "sum")
    tot_od = plumb.reduce(float(onr), "sum")
    tot_bytes = plumb.reduce(float((lnb + onb) * BLCKSZ), "sum")
    par = _join_small_parity(ctx, capi.TAB_LINEITEM_WIDE, redistribute=True)
    if rank != 0:
        return None
    v = rows[0][0]
    peak, _ = measured_peak()
    Wl, Wo = 1 + len(lt), 1 + len(ot)
    algo = tot_bytes + 2 * 8 * (Wl * tot_li + Wo * tot_od) + 16 * tot_od + 32 * tot_li
    par["full_size_property"] = {"rows_joined": int(v[0]), "outer_rows": int(tot_li), "fk_join_count_equals_outer_rows": bool(v[0] == int(tot_li)),
                                 "sum_o_custkey": int(v[1])}
    par["ok"] = bool(par["ok"] and v[0] == int(tot_li))
    return {"workload": "Redistribute-HashJoin lineitem-wide ⋈ orders: %d x %d rows IN TOTAL over %d GPU(s) (strong scaling); count(*), sum(o_custkey), sum(l_extendedprice)"
                        % (int(tot_li), int(tot_od), world),
            "plan": "Agg(FINAL)<-Gather<-Agg(PARTIAL)<-HashJoin(Redistribute<-SeqScan, Hash(Redistribute<-SeqScan))", "api": "GgExecProcNode",
            "interconnect": "gg_ic_* over NCCL (C)" if world > 1 else "loopback (one segment)",
            "scaling": "strong", "n_gpus": world, "ms": ms, "rows_per_s": (tot_li + tot_od) / (ms / 1e3),
            "build_ms": build_ms, "probe_ms": probe_ms, "kernel_variant": variant, "gpu_launches_per_step": launches,
            "roofline": {"bound": "hbm", "algorithmic_bytes_all_gpus": algo, "achieved_per_gpu": algo / world / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / world / (ms / 1e3) / 1e9 / peak,
                         "note": "whole step (partition, exchange, build, probe): base pages once + the travelling datum rows written and read once "
                                 "(%d / %d B per lineitem / orders row) + 16 B/inner row + 32 B per probe; NVLink carries (N-1)/N of the rows" % (8 * Wl, 8 * Wo)},
            "parity": par, "setup_s": round(setup, 1)}


def sec_narrow(ctx):
    """The north star's full-size configuration: Q1 scan+agg over a 10^9-row lineitem-narrow relation (76 GB) on ONE GPU."""
    from greengage_b200 import executor as ex
    from greengage_b200.engine import Relation
    from oracle import pyoracle as po
    eng = ctx["eng"]
    R = int(ctx["args"].narrow_rows)
    copies = 10
    t0 = time.time()
    # one 1/10 shard of the 10^9-row table is generated on the host (the host generator makes ~6 M rows/s on this container's
    # cores); the relation is that shard's pages ten times over, copied on the device
    spec = tpch.synth_spec(capi.TAB_LINEITEM_NARROW, R, nsegs=copies, seg=0)
    snb, snr = tpch.synth_measure(spec, ctx["nthreads"])
    pages, _, _ = tpch.synth_generate(spec, nthreads=ctx["nthreads"], measured=(snb, snr))
    rel = Relation(eng, nblocks=snb * copies)
    rel.load(0, pages)
    eng.sync()
    shard = Relation(eng, nblocks=snb, device_ptr=rel.device_ptr())
    for c in range(1, copies):
        rel.copy_from(shard, dst_first=c * snb)
    eng.sync()
    setup = time.time() - t0
    nb, nr = snb * copies, snr * copies
    b = ex.PlanBuilder()
    plan, pool = tpch.q1_exec_plan(b, capi.TAB_LINEITEM_NARROW)
    x = ex.Executor(eng, pool, [rel], plan)
    ms, n, launches = _timed_steps(ctx, x, steps=5, warmup=3)
    kms, k, variant, _ = x.kernel_ms()
    x.rescan()
    full = q1_rows_from_slots(x.rows())
    x.end()
    # parity: the oracle over a bounded prefix of the shard vs the same plan over the same pages; then the full-size
    # property: 10 copies of the shard => every count is exactly 10x the shard's, every sum 10x within rounding
    cores = host_cores()
    sample_nb = min(snb, max(1, int(snb * min(1.0, 4_000_000 * cores / snr))))
    scan_o, part_o, pool_o = tpch.q1_plan(capi.TAB_LINEITEM_NARROW, capi.AGGSTAGE_PARTIAL)
    orows, secs, oscanned = po.seqscan_agg_mt(scan_o, part_o, tpch.q1_final_agg(part_o), pool_o, pages[:sample_nb * BLCKSZ], cores)
    sub = Relation(eng, nblocks=sample_nb, device_ptr=rel.device_ptr())
    bp = ex.PlanBuilder()
    plan_p, pool_p = tpch.q1_exec_plan(bp, capi.TAB_LINEITEM_NARROW)
    xp = ex.Executor(eng, pool_p, [sub], plan_p)
    par = q1_compare(q1_rows_from_slots(xp.rows()), q1_rows_from_oracle(orows))
    xp.end()
    sub.free()
    bs = ex.PlanBuilder()
    plan_s, pool_s = tpch.q1_exec_plan(bs, capi.TAB_LINEITEM_NARROW)
    xs = ex.Executor(eng, pool_s, [shard], plan_s)
    one = q1_rows_from_slots(xs.rows())
    xs.end()
    lin_counts = set(full) == set(one) and all(full[k][1] == copies * one[k][1] for k in one)
    lin_err = max(abs(full[k][0][i] - copies * one[k][0][i]) / abs(copies * one[k][0][i]) for k in one for i in range(4)) if lin_counts else None
    par["rows_checked"] = int(oscanned)
    par["how"] = "oracle over the first %d pages of the shard vs the same plan over the same pages" % sample_nb
    par["full_size_property"] = {"counts_equal_10x_shard": bool(lin_counts), "sums_rel_err_vs_10x_shard": lin_err,
                                 "count_sum": int(sum(c for _, c in full.values())), "rows": int(nr)}
    par["ok"] = bool(par["ok"] and lin_counts and lin_err is not None and lin_err <= 1e-9)
    shard.free()
    rel.free()
    peak, _ = measured_peak()
    kernel_ms = kms / max(k, 1)
    return {"workload": "Q1 scan+filter+hashagg over %d rows of lineitem-narrow, %d pages = %.1f GB resident on one GPU" % (nr, nb, nb * BLCKSZ / 1e9),
            "data": "synthetic; %d device-side copies of one %d-row shard of the 10^9-row table (host generation of all ten shards takes minutes)" % (copies, snr),
            "plan": "Agg(NORMAL)<-SeqScan", "api": "GgExecProcNode", "ms": ms, "rows_per_s": nr / (ms / 1e3), "kernel_variant": variant,
            "gpu_launches_per_step": launches,
            "roofline": {"bound": "hbm", "algorithmic_bytes": nb * BLCKSZ, "kernel_ms": kernel_ms, "achieved": nb * BLCKSZ / (kernel_ms / 1e3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": nb * BLCKSZ / (kernel_ms / 1e3) / 1e9 / peak, "frac_of_nominal_8TBs": nb * BLCKSZ / (kernel_ms / 1e3) / 8e12,
                         "target": "north star: >= 0.40 of the per-GPU HBM roofline"},
            "parity": par, "setup_s": round(setup, 1)}


def sec_aocs(ctx):
    """SURVEY §8f rank 1: the same 10^8 lineitem rows stored append-only column-oriented (compresstype none, checksums on), Q1's
    seven projected columns only: fused scan over the column files (gg_scanagg_run_aocs).  Roofline on the PROJECTED bytes."""
    from greengage_b200 import aocs
    from greengage_b200.engine import ScanAgg
    eng, rel, table = ctx["eng"], ctx["rel"], ctx["table"]
    if table != capi.TAB_LINEITEM_WIDE or rel is None:
        return None
    cols = [4, 5, 6, 7, 8, 9, 10]
    names = dict(quantity=1, extendedprice=2, discount=3, tax=4, returnflag=5, linestatus=6, shipdate=7)
    spec = tpch.synth_spec(table, ctx["args"].rows)
    t0 = time.time()
    files, nrows = aocs.synth_columns(spec, cols, ctx["nr"], nthreads=ctx["nthreads"])
    gen_s = time.time() - t0
    desc = capi.synth_tupdesc(table)
    t0 = time.time()
    dc = aocs.DeviceColumns(eng, desc, cols, files, pinned=True)
    eng.sync()
    load_s = time.time() - t0
    del files
    scan, agg, pool = tpch.q1_plan(stage=capi.AGGSTAGE_NORMAL, desc=dc.rows_tupdesc([1] * len(cols)), cols=names)
    sa = ScanAgg(eng, scan, agg, pool)
    kms = []
    for it in range(8):
        sa.reset()
        sa.run_aocs(dc)
        got, sc, ps = sa.fetch()
        if it >= 3:
            kms.append(sa.scan_kernel_ms()[0])
    kernel_ms = float(np.mean(kms))
    # end to end: the column files (with the block directory and tile plan the loader made) start in pinned host memory
    eng.sync()
    eng.timer_start()
    for _ in range(3):
        sa.reset()
        dc.upload()
        sa.run_aocs(dc)
        got_e, sc_e, ps_e = sa.fetch()
    ems = eng.timer_stop() / 3
    variant = sa.variant()
    # parity: the heap pages of the same rows through the same engine (that answer is the one the headline's parity gate held to
    # the oracle): counts exact, sums 1e-9
    hs, ha, hp = tpch.q1_plan(table)
    sh = ScanAgg(eng, hs, ha, hp)
    sh.run(rel)
    want, wsc, wps = sh.fetch()
    sh.free()
    sa.free()
    g = q1_rows_from_oracle(got)
    par = q1_compare(g, q1_rows_from_oracle(want), tol=1e-9)
    par["how"] = "fused scan over the column files vs the heap pages of the same %d rows on the same engine (the heap answer is the one held to the oracle above)" % nrows
    par["rows_scanned_equal"] = bool((sc, ps) == (wsc, wps) == (sc_e, ps_e))
    par["ok"] = bool(par["ok"] and par["rows_scanned_equal"])
    bytes_in = dc.bytes_in
    arena = dc.arena_bytes
    dc.free()
    peak, _ = measured_peak()
    return {"workload": "Q1 scan+filter+hashagg over the same %d rows stored append-only column-oriented, 7 projected columns = %.1f B/row (heap: 172 B/row)" % (nrows, bytes_in / nrows),
            "api": "gg_scanagg_run_aocs (C-ABI)", "ms": kernel_ms, "rows_per_s": nrows / (kernel_ms / 1e3), "kernel_variant": variant,
            "roofline": {"bound": "hbm", "algorithmic_bytes": bytes_in, "achieved": bytes_in / (kernel_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": bytes_in / (kernel_ms / 1e3) / 1e9 / peak, "note": "bytes of the projected column files, read once"},
            "e2e": {"value": nrows / (ems / 1e3), "unit": UNIT, "ms_per_step": ems, "h2d_bytes_per_step": int(arena),
                    "note": "column files + block directory + tile plan copied from pinned host memory every step, then the fused scan; the loader's "
                            "host work (CRC-32C of every block, directory, tile plan) is done once at load: host_load_s"},
            "host_generate_s": round(gen_s, 1), "host_load_s": round(load_s, 2), "parity": par}


def sec_sort(ctx):
    """Sort of 10^8 int64 keys on the device (gg_sort_device: the radix sort behind the Sort node)."""
    from greengage_b200.engine import Relation
    eng = ctx["eng"]
    L = capi.dev_lib()
    n = 100_000_000
    n = (n * 8 // BLCKSZ) * BLCKSZ // 8                       # whole pages of keys
    rng = np.random.default_rng(1)
    rows = rng.integers(0, 6 * 10**9, n, dtype=np.int64)     # l_orderkey-like: 33 significant bits
    buf = Relation(eng, nblocks=n * 8 // BLCKSZ + 1)
    perm = Relation(eng, nblocks=n * 4 // BLCKSZ + 1)
    buf.load(0, rows.view(np.uint8))
    eng.sync()
    keys = (capi.gg_sortkey * 1)(capi.make_sortkey(0, capi.INT8OID))
    passes = C.c_int(0)
    ms = []
    for it in range(8):
        capi.check(L.gg_sort_device(eng.h, keys, 1, 1, C.c_void_p(buf.device_ptr()), None, n, C.c_void_p(perm.device_ptr()), C.byref(passes)))
        if it >= 3:
            ms.append(eng.last_kernel_ms())
    t = float(np.mean(ms))
    out = perm.read().view(np.uint32)[:n]
    srt = rows[out.astype(np.int64)]
    sorted_ok = bool(np.all(np.diff(srt) >= 0))
    perm_ok = bool(np.array_equal(np.sort(out), np.arange(n, dtype=np.uint32)))
    buf.free()
    perm.free()
    peak, _ = measured_peak()
    algo = n * (8 + 8 + passes.value * 32)
    return {"workload": "sort %d int64 keys (33 significant bits) on the device, row numbers out" % n, "api": "gg_sort_device (C-ABI)",
            "ms": t, "passes": passes.value, "rows_per_s": n / (t / 1e3),
            "roofline": {"bound": "hbm", "algorithmic_bytes": algo, "achieved": algo / (t / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / (t / 1e3) / 1e9 / peak, "note": "16 B/row key build + 32 B/row per executed radix pass"},
            "parity": {"checked": True, "how": "full size: output is a permutation and the keys come back in non-decreasing order (numpy on the host)",
                       "sorted": sorted_ok, "is_permutation": perm_ok, "ok": sorted_ok and perm_ok}}


def sec_paths(ctx):
    """The headline plan on the other two kernel paths, once: the bench line's kernel is registered at build time
    (csrc/plans); any other plan is specialised at run time through NVRTC, or runs on the interpreter kernel."""
    from greengage_b200 import executor as ex
    eng, rel, nb = ctx["eng"], ctx["rel"], ctx["nb"]
    out = {}
    peak, _ = measured_peak()
    for name, env in (("nvrtc", {"GGB200_PLAN_CACHE": "0"}), ("interpreter", {"GGB200_JIT": "0"})):
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            b = ex.PlanBuilder()
            plan, pool = tpch.q1_exec_plan(b, ctx["table"])
            x = ex.Executor(eng, pool, [rel], plan)
            ms, n, _ = _timed_steps(ctx, x, steps=3, warmup=2)
            kms, k, variant, _ = x.kernel_ms()
            x.end()
            out[name] = {"ms": ms, "kernel_ms": kms / max(k, 1), "kernel_variant": variant, "frac": nb * BLCKSZ / (kms / max(k, 1) / 1e3) / 1e9 / peak}
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    out["note"] = "kernel_variant: +16 registered at build time, +32 specialised at run time (NVRTC), neither = interpreter"
    return out


def _side_relation(ctx, rows):
    """A lineitem-wide relation of `rows` rows for the last two secondaries (the headline's relation is gone by then): host
    pages (kept for the parity samples) and the resident relation"""
    from greengage_b200.engine import Relation
    spec = tpch.synth_spec(capi.TAB_LINEITEM_WIDE, rows, norders=max(rows // 4, 1), seed=11)
    pages, nb, nr = tpch.synth_generate(spec, nthreads=ctx["nthreads"])
    rel = Relation(ctx["eng"], host_pages=pages)
    return pages, rel, nb, nr


def sec_groupby(ctx):
    """SURVEY §8a row 9, the general HashAggregate (lookup_agg_hash_entry, execHHashagg.c:456): GROUP BY l_orderkey — a quarter
    as many groups as rows, one table in HBM — with count(*) and sum(l_extendedprice).  Parity: the same plan over a prefix of
    the pages against the oracle, group by group."""
    from greengage_b200.engine import Relation, ScanAgg
    from oracle import pyoracle as po
    eng = ctx["eng"]
    rows = max(int(ctx["args"].rows) // 4, 100_000)
    pages, rel, nb, nr = _side_relation(ctx, rows)
    c = tpch.LI_WIDE_COLS
    p = capi.ExprPool()
    agg = capi.make_agg(capi.AGGSTAGE_NORMAL, [p.var(c["orderkey"], capi.INT8OID)],
                        [(capi.AGG_COUNT_STAR, -1), (capi.AGG_SUM_FLOAT8, p.var(c["extendedprice"], capi.FLOAT8OID))], num_groups=max(rows // 4, 1))
    scan = capi.make_scan(capi.synth_tupdesc(capi.TAB_LINEITEM_WIDE), -1)
    sa = ScanAgg(eng, scan, agg, p.pool)
    ms = []
    for it in range(8):
        sa.reset()
        sa.run(rel)
        eng.sync()
        if it >= 3:
            ms.append(sa.scan_kernel_ms()[0])
    t = float(np.mean(ms))
    variant = sa.variant()
    # parity on a prefix small enough for the oracle's row-at-a-time table and a full fetch of the groups
    k = min(nb, 300)
    sub = Relation(eng, nblocks=k, device_ptr=rel.device_ptr())
    sa.reset()
    sa.run(sub)
    got, sc, ps = sa.fetch(cap=1 << 17)
    want, wsc, wps = po.seqscan_agg(scan, agg, p.pool, pages[:k * BLCKSZ], cap=1 << 17)
    g = {r.key[0]: (r.agg[0].i, r.agg[1].f[0]) for r in got}
    w = {r.key[0]: (r.agg[0].i, r.agg[1].f[0]) for r in want}
    rel_err = max([abs(g[kk][1] - w[kk][1]) / max(abs(w[kk][1]), 1e-300) for kk in w if kk in g] or [0.0])
    par = {"checked": True, "how": "the same plan over the first %d pages vs the CPU oracle, group by group" % k, "groups": len(w),
           "groups_equal": bool(set(g) == set(w)), "counts_equal": bool(all(kk in g and g[kk][0] == w[kk][0] for kk in w)),
           "rows_scanned_equal": bool((sc, ps) == (wsc, wps)), "max_rel_err": rel_err}
    par["ok"] = bool(par["groups_equal"] and par["counts_equal"] and par["rows_scanned_equal"] and rel_err <= 1e-9)
    sa.free()
    sub.free()
    rel.free()
    peak, _ = measured_peak()
    rr = random_access_rates()
    bound = None
    if rr:
        b_ms = nb * BLCKSZ / (peak * 1e9) * 1e3 + nr / (rr["gather_g_per_s"] * 1e9) * 1e3 + nr / (rr["atomic_pair_g_per_s"] * 1e9) * 1e3
        bound = {"rates": rr, "bound_ms": b_ms, "frac_of_bound": b_ms / t,
                 "note": "pages at copy bandwidth + one random 32-byte table entry read per row + one atomic pair (count, sum) per row, terms added"}
    return {"workload": "general HashAggregate: GROUP BY l_orderkey over %d lineitem-wide rows (~%d groups), count(*) + sum(l_extendedprice)" % (nr, rows // 4),
            "api": "gg_scanagg_run (C-ABI), table in HBM", "ms": t, "rows_per_s": nr / (t / 1e3), "kernel_variant": variant,
            "roofline": {"bound": "hbm", "algorithmic_bytes": nb * BLCKSZ, "achieved": nb * BLCKSZ / (t / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": nb * BLCKSZ / (t / 1e3) / 1e9 / peak, "note": "pages read once; the table's random traffic is in random_access_bound",
                         "random_access_bound": bound},
            "parity": par}


def sec_motion(ctx):
    """SURVEY §8a rows 15-16, the sending half of a Redistribute Motion (execMotionSender, nodeMotion.c:270; cdbhash +
    jump consistent hash): lineitem-wide on l_orderkey to 8 destinations, two columns travel.  Parity: rows per destination over
    a prefix of the pages (exact claims) against the oracle's routing."""
    from greengage_b200.engine import Relation, motion_partition
    from oracle import pyoracle as po
    eng = ctx["eng"]
    rows = max(int(ctx["args"].rows) // 4, 100_000)
    pages, rel, nb, nr = _side_relation(ctx, rows)
    nsegs = 8
    c = tpch.LI_WIDE_COLS
    p = capi.ExprPool()
    key = p.var(c["orderkey"], capi.INT8OID)
    payload = [key, p.var(c["extendedprice"], capi.FLOAT8OID)]
    W = 1 + len(payload)
    scan = capi.make_scan(capi.synth_tupdesc(capi.TAB_LINEITEM_WIDE), -1)
    cap = (int(nr / nsegs * 1.25) + 8192) * nsegs
    out = Relation(eng, nblocks=(cap * W * 8 + 64 + BLCKSZ - 1) // BLCKSZ)
    ms = []
    for it in range(8):
        counts, offs = motion_partition(eng, scan, p.pool, [key], payload, nsegs, rel, out.device_ptr(), cap)
        if it >= 3:
            ms.append(eng.last_kernel_ms())
    t = float(np.mean(ms))
    k = min(nb, 2000)
    old = os.environ.get("GGB200_MOTION_WINDOW")
    os.environ["GGB200_MOTION_WINDOW"] = "0"          # exact claims: the counts are the rows, no dead slots
    try:
        pc, _ = motion_partition(eng, scan, p.pool, [key], payload, nsegs, rel, out.device_ptr(), cap, first_block=0, nblocks=k)
    finally:
        if old is None:
            os.environ.pop("GGB200_MOTION_WINDOW", None)
        else:
            os.environ["GGB200_MOTION_WINDOW"] = old
    dest = po.motion_route(scan, p.pool, [key], nsegs, pages[:k * BLCKSZ])
    want = np.bincount(dest, minlength=nsegs).tolist()
    par = {"checked": True, "how": "rows per destination over the first %d pages (exact claims) vs the oracle's cdbhash routing" % k,
           "counts": [int(x) for x in pc], "counts_equal": bool([int(x) for x in pc] == want), "ok": bool([int(x) for x in pc] == want)}
    out.free()
    rel.free()
    peak, _ = measured_peak()
    algo = nb * BLCKSZ + nr * W * 8
    return {"workload": "Motion send: lineitem-wide (%d rows) redistributed on l_orderkey to %d destinations, %d columns travel" % (nr, nsegs, len(payload)),
            "api": "gg_motion_partition (C-ABI)", "ms": t, "rows_per_s": nr / (t / 1e3), "slots_claimed": int(sum(counts)),
            "roofline": {"bound": "hbm", "algorithmic_bytes": algo, "achieved": algo / (t / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / (t / 1e3) / 1e9 / peak, "note": "pages read once + %d B/row written" % (W * 8)},
            "parity": par}


SECONDARY = {"join": sec_join, "rjoin": sec_rjoin, "narrow": sec_narrow, "sort": sec_sort, "paths": sec_paths, "aocs": sec_aocs,
             "groupby": sec_groupby, "motion": sec_motion}


if __name__ == "__main__":
    main()
