#!/usr/bin/env python
"""bench.py -- TPC-H Q1 (filter + 2-key group-by, 4 sums, 3 avgs, count) over synthetic SF100 lineitem.

One "step" = one full pass of the hot path over the rank's lineitem partition:
  HashAggregate(Partial) over [Scan -> Filter -> Project] as ONE fused sm_100a kernel launch per
  device chunk (+ fold/finalize), then the partial states of all ranks are gathered on rank 0 and
  merged by HashAggregate(Final) (merge_batch semantics) -- the same two plans Spark + Comet run on
  either side of the shuffle (SURVEY.md section 3D).

`value`  : rows/s with the Arrow columns already resident in HBM (bound through cb200_table_*).
`e2e`    : the same plans through cb200_create_plan / cb200_execute with HOST Arrow buffers handed over
           as an ArrowArrayStream (pinned host memory; H2D inside the timed region; result D2H).
`roofline`: algorithmic bytes of the fused Q1 kernel / its CUDA-event duration (events recorded by the
           library on the stream it launches on) against MEASURED_PEAKS.json hbm_gbs.
`cpu_baseline` / `--impl reference`: the CPU oracle port (oracle/comet_oracle.c, OpenMP, all host
           cores) -- the reference's Rust/DataFusion path cannot be built in this image (no Rust).

Launch: python bench.py [--gpus N --steps K --warmup W]   (torchrun for N>1, one rank per GPU)
`--dump-outputs DIR`: after the timed steps, the Q1 result of the last timed step as DIR/<output>.npy (float64), for comparing
           two builds on the same seeded inputs.
"""
import argparse
import atexit
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True   # the source tree may be read-only: nothing is written into it

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "datafusion-comet_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

SF100_ROWS = 600_037_902
METRIC = "rows/sec on TPC-H Q1 filter+agg"
# bytes the fused kernel must read per row (Arrow layout, dictionary-coded flags):
#   l_shipdate date32 4 + returnflag/linestatus codes 1+1 + 4 x Decimal128 16  (DESIGN.md "algorithmic bytes")
BYTES_PER_ROW = {"dec": 4 + 1 + 1 + 4 * 16, "f64": 4 + 1 + 1 + 4 * 8}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic(rows, variant):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE bulk launch of the fused kernel, from the committed `ncu --set full`
    capture of this same workload (profiles/r1_traffic.json, written by tools/summarize_ncu.py); None when the capture was taken
    at another size / variant."""
    try:
        with open(os.path.join(ROOT, "profiles", "r1_traffic.json")) as f:
            t = json.load(f)["cb_pipeline_agg"]
        return int(t["dram_bytes"]) if int(t["rows"]) == int(rows) and t["variant"] == variant else None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  The sampler is started BEFORE the warm-up
    (nvidia-smi's own start-up takes a second and its NVML initialisation can stall CUDA calls of other processes); only
    samples whose timestamp falls inside [mark_begin, mark_end] are reported."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.t0 = self.t1 = None

    def start(self):
        self.path = tempfile.mktemp(prefix="cb200_clocks_", suffix=".csv")
        q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.05)  # let the sample that covers the end of the region land
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(f[1]), float(f[2]), f[4:8]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        inside = [r for r in rows if self.t0 is not None and self.t0 - 0.02 <= r[0] <= (self.t1 or r[0]) + 0.02]
        if not inside and rows and self.t0 is not None:  # region shorter than the sampling period: the sample nearest to it
            inside = [min(rows, key=lambda r: abs(r[0] - self.t0))]
        if inside:
            reasons = set()
            for r in inside:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            out = {"sm_mhz": statistics.median(r[1] for r in inside), "sm_max_mhz": max(r[2] for r in inside), "reasons": sorted(reasons), "samples": len(inside)}
        return out


# ---- data ---------------------------------------------------------------------------------------
def gen_device(torch, n, seed, device):
    """TPC-H-shaped lineitem columns on the device (SURVEY.md 8d distribution; torch Philox, seeded)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)

    def ri(lo, hi, dtype=torch.int64):
        return torch.randint(lo, hi, (n,), generator=g, device=device, dtype=dtype)

    qty_units = ri(1, 51)
    price = qty_units * ri(90000, 210001)          # cents
    qty = qty_units * 100
    disc = ri(0, 11)
    tax = ri(0, 9)
    ship = ri(8036, 10562, torch.int32)
    receipt = ship + ri(1, 31, torch.int32)
    ar = (ri(0, 2, torch.int8) * 2)
    rf = torch.where(receipt <= 9298, ar, torch.ones_like(ar)).contiguous()
    ls = (ship > 9298).to(torch.int8).contiguous()
    del receipt, ar, qty_units
    return dict(l_quantity=qty, l_extendedprice=price, l_discount=disc, l_tax=tax, l_shipdate=ship, l_returnflag=rf, l_linestatus=ls)


def to_dec128(torch, cents):
    """int64 unscaled -> Arrow Decimal128 layout (n,2) int64 (lo, sign-extended hi)"""
    out = torch.empty((cents.shape[0], 2), dtype=torch.int64, device=cents.device)
    out[:, 0] = cents
    out[:, 1] = cents >> 63
    return out


def build_columns(torch, cols, variant):
    money = {}
    for k in ("l_quantity", "l_extendedprice", "l_discount", "l_tax"):
        money[k] = to_dec128(torch, cols[k]) if variant == "dec" else (cols[k].to(torch.float64) / 100.0)
    return money


def bind_table(native, P, tpch, variant, n, money, cols):
    m = tpch.D12 if variant == "dec" else P.DOUBLE
    w = 16 if variant == "dec" else 8
    t = native.DeviceTable(n)
    for k in ("l_quantity", "l_extendedprice", "l_discount", "l_tax"):
        t.add(m, money[k].data_ptr(), w, keep=money[k])
    t.add(P.STRING, cols["l_returnflag"].data_ptr(), 1, dictionary=tpch.RETURNFLAGS, keep=cols["l_returnflag"])
    t.add(P.STRING, cols["l_linestatus"].data_ptr(), 1, dictionary=tpch.LINESTATUS, keep=cols["l_linestatus"])
    t.add(P.DATE, cols["l_shipdate"].data_ptr(), 4, keep=cols["l_shipdate"])
    return t


def host_arrow_batches(torch, pa, tpch, variant, money, cols, batch_rows, pin=True):
    """Copy the device columns into host memory (PINNED when they are uploaded from there: the Arrow e2e leg; pageable when they
    only feed the Parquet writer or the CPU baseline -- 8 ranks x 42 GB of pinned memory is not something to ask of a box) and
    wrap them as zero-copy Arrow batches."""
    host = {}
    for k, t in list(money.items()) + [(k, cols[k]) for k in ("l_returnflag", "l_linestatus", "l_shipdate")]:
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=pin)
        h.copy_(t)
        host[k] = h
    torch.cuda.synchronize()
    n = cols["l_shipdate"].shape[0]

    def buf(t):
        return pa.foreign_buffer(t.data_ptr(), t.numel() * t.element_size(), base=t)

    arrays = []
    for k in ("l_quantity", "l_extendedprice", "l_discount", "l_tax"):
        typ = pa.decimal128(12, 2) if variant == "dec" else pa.float64()
        arrays.append(pa.Array.from_buffers(typ, n, [None, buf(host[k])]))
    for k, vals in (("l_returnflag", tpch.RETURNFLAGS), ("l_linestatus", tpch.LINESTATUS)):
        idx = pa.Array.from_buffers(pa.int8(), n, [None, buf(host[k])])
        arrays.append(pa.DictionaryArray.from_arrays(idx, pa.array(vals)))
    arrays.append(pa.Array.from_buffers(pa.date32(), n, [None, buf(host["l_shipdate"])]))
    names = ["l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate"]
    tbl = pa.table(arrays, names=names)
    return tbl.to_batches(max_chunksize=batch_rows), host


# ---- one step -----------------------------------------------------------------------------------
DEVICE = 0  # CUDA ordinal of this rank (set in main)


def run_partial(native, plan_bytes, inp, chunk_rows):
    with native.Plan(plan_bytes, [inp] if inp is not None else [], config={"spark.comet.b200.chunkRows": str(chunk_rows)}, device=DEVICE) as p:
        state = p.collect()
        st = p.stats()
    return state, st


def run_final(native, pa, plan_bytes, states):
    tbl = pa.concat_tables(states)
    with native.Plan(plan_bytes, [tbl], device=DEVICE) as p:
        res = p.collect()
        st = p.stats()
    return res, st


def usable_cores():
    """Cores this process may actually run on: the affinity mask, capped by the cgroup CPU quota (os.cpu_count() reports the
    machine, not the container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def best_thread_count(fn, cores):
    """The oracle is timed with the thread count that makes it FASTEST (all cores is not always it: SMT siblings, NUMA, an
    oversubscribed container): one untimed + one timed pass per candidate."""
    best, best_t = cores, None
    for c in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
        fn(c)
        t = time.perf_counter()
        fn(c)
        dt = time.perf_counter() - t
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    return best


def gpu_numa_cpus(gpu_index):
    """CPUs of the NUMA node the GPU hangs off (intersected with what this process may use), or None."""
    try:
        bus = subprocess.check_output(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], text=True).strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None, None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        return node, (cpus or None)
    except Exception:
        return None, None


class NumaLocal:
    """Run the host side of a rank on the CPUs next to its GPU while pinned buffers are allocated and filled (first touch places
    the pages on that node): H2D copies then do not cross the socket interconnect.  What a NUMA-aware executor launch does."""

    def __init__(self, gpu_index, enabled=True):
        self.node, self.cpus = gpu_numa_cpus(gpu_index) if enabled else (None, None)
        self.saved = None

    def __enter__(self):
        if self.cpus:
            self.saved = os.sched_getaffinity(0)
            os.sched_setaffinity(0, self.cpus)
        return self

    def __exit__(self, *a):
        if self.saved:
            os.sched_setaffinity(0, self.saved)


def setup(args):
    import torch
    import torch.distributed as dist
    from comet_b200 import native
    global DEVICE
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    DEVICE = local_rank
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    comm = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

        def bcast(b):  # the control channel for the library's NCCL id: torch.distributed is plumbing here
            t = torch.tensor(list(b) if b is not None else [0] * 128, dtype=torch.uint8, device=device)
            dist.broadcast(t, 0)
            return bytes(t.cpu().tolist())
        comm = native.Comm(rank, world, local_rank, bcast)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=device, dtype=torch.int64)
        dist.all_reduce(t)
        return int(t.item())
    return dict(torch=torch, dist=dist, native=native, rank=rank, local_rank=local_rank, world=world, device=device, comm=comm, barrier=barrier,
                max_over_ranks=max_over_ranks, sum_over_ranks=sum_over_ranks)


def private_jit_cache():
    """Kernels compiled at run time (range-specialised variants of the pipelines) are cached in a temporary directory rather
    than next to the library, so the source tree stays untouched; the cubins build() compiled are linked in and not compiled
    again."""
    if os.environ.get("CB200_CACHE_DIR"):
        return
    shipped = os.path.join(ROOT, "datafusion-comet_b200", ".jitcache")
    d = tempfile.mkdtemp(prefix="cb200_jitcache_")
    atexit.register(shutil.rmtree, d, True)
    if os.path.isdir(shipped):
        for f in os.listdir(shipped):
            os.symlink(os.path.join(shipped, f), os.path.join(d, f))
    os.environ["CB200_CACHE_DIR"] = d


def timed_region(env, sampler, step_fn, warmup, steps):
    """W untimed steps, then exactly K steps between barrier + synchronize on both sides; max over ranks."""
    import gc
    for _ in range(warmup):
        step_fn()
    gc.collect()
    gc.disable()  # a collector pause in the middle of a 6 ms step is measurement noise, not engine time
    env["barrier"]()
    if sampler:
        sampler.mark_begin()
    t0 = time.perf_counter()
    outs, marks = [], [t0]
    for _ in range(steps):
        outs.append(step_fn())
        marks.append(time.perf_counter())     # host time when the step's call returned (its result is on the host / synchronised by then)
    env["barrier"]()
    elapsed = time.perf_counter() - t0
    per = sorted(1e3 * (b - a) for a, b in zip(marks, marks[1:]))
    env["step_ms"] = {"min": per[0], "median": per[len(per) // 2], "max": per[-1]}
    if sampler:
        sampler.mark_end()
    gc.enable()
    return env["max_over_ranks"](elapsed), outs


# =====================================================================================================================
# reference arm: the reference's CPU path (oracle port; the Rust original cannot be built here) on the host cores
# =====================================================================================================================
def reference_arm(args, rank, world):
    if rank != 0:
        return
    import numpy as np
    from comet_b200 import tpch
    from oracle import oracle
    oracle.build()
    n = args.ref_rows
    cols = tpch.gen_lineitem(n, seed=42)
    d = oracle.dec_from_i64
    cores_all = usable_cores()
    if args.workload == "q1":
        a = (d(cols["l_quantity"]), d(cols["l_extendedprice"]), d(cols["l_discount"]), d(cols["l_tax"]), cols["l_shipdate"],
             cols["l_returnflag"], cols["l_linestatus"], 3, 2, tpch.Q1_CUTOFF)
        fn, what, metric = (lambda c: oracle.q1_dec(*a, c)), "co_q1_dec", METRIC
    elif args.workload == "q6":
        a = (d(cols["l_quantity"]), d(cols["l_extendedprice"]), d(cols["l_discount"]), cols["l_shipdate"], tpch.DATE_1994_01_01, tpch.DATE_1995_01_01, 5, 7, 2400)
        fn, what, metric = (lambda c: oracle.q6_dec(*a, c)), "co_q6_dec", "rows/sec on TPC-H Q6 filter+sum"
    elif args.workload == "config1":
        a = (d(cols["l_quantity"]), d(cols["l_extendedprice"]), cols["l_shipdate"], tpch.DATE_1998_09_02)
        fn, what, metric = (lambda c: oracle.filter_project_dec(*a, c)), "co_filter_project_dec", "rows/sec on filter+project (Config 1)"
    else:
        keys, vals = cols["l_orderkey"], d(cols["l_extendedprice"])
        a = (keys, vals)
        fn, what, metric = (lambda c: oracle.groupby_sum_dec(keys, vals, c)), "co_groupby_sum_dec", GROUPBY_METRIC
    a = tuple(oracle.numa_spread(x, cores_all) if isinstance(x, np.ndarray) else x for x in a)
    cores = best_thread_count(fn, cores_all)
    for _ in range(args.warmup):
        fn(cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn(cores)
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    line = {"impl": "reference", "metric": metric, "value": v, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i128",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}: DECIMAL(12,2), bounded sample of {n} rows of the SF100 lineitem shape per step, in-memory Arrow columns "
                                   "(no Parquet decode: the CPU arm starts from decoded columns, which favours it against the GPU arm's e2e leg that decodes pages)",
                       "rows": n, "why_not_the_full_workload": "the bench contract bounds the reference arm to a sample that finishes in minutes; the metric is a rate, "
                                                              "and the port's rate is flat in the row count (one streaming pass per thread)"},
            "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port",
                             "sample": f"{n} rows/step, oracle/comet_oracle.c {what}, OpenMP {cores} threads (reference Rust path not buildable here)"},
            "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# =====================================================================================================================
# Q1 (default): BASELINE.json configs[1]
# =====================================================================================================================
def q1_expected_from_torch(torch, cols, cutoff):
    """All eight Q1 outputs of this rank's partition, exact, from torch int64 arithmetic on the device (independent of the library
    AND of the oracle): sums as python ints, averages by the reference's HALF_UP rule, per group index 0..5."""
    keep = cols["l_shipdate"] <= cutoff
    gid = (cols["l_returnflag"].to(torch.int64) * 2 + cols["l_linestatus"].to(torch.int64))[keep]
    q, p, dsc, tax = (cols[k][keep] for k in ("l_quantity", "l_extendedprice", "l_discount", "l_tax"))

    def gsum(v):
        return torch.zeros(6, dtype=torch.int64, device=v.device).scatter_add_(0, gid, v).cpu().tolist()
    cnt = torch.bincount(gid, minlength=6).cpu().tolist()
    sq, sp, sd = gsum(q), gsum(p), gsum(dsc)
    dp = p * (100 - dsc)                      # d(26,4) unscaled: < 2.1e9 per row
    sdp = gsum(dp)
    ch = dp * (100 + tax)                     # d(38,6) unscaled: < 2.3e11 per row; 1.5e8 rows per group overflow int64 -> split
    sch = [hi * (1 << 20) + lo for hi, lo in zip(gsum(ch >> 20), gsum(ch & ((1 << 20) - 1)))]

    def avg(s, c):                            # avg_decimal.rs:670-689: sum * 10^4 / count, HALF_UP
        qq, r = divmod(abs(s) * 10**4, c)
        v = qq + (1 if 2 * r >= c else 0)
        return v if s >= 0 else -v
    out = {}
    for g in range(6):
        if cnt[g]:
            out[g] = dict(sum_qty=sq[g], sum_base_price=sp[g], sum_disc_price=sdp[g], sum_charge=sch[g], avg_qty=avg(sq[g], cnt[g]),
                          avg_price=avg(sp[g], cnt[g]), avg_disc=avg(sd[g], cnt[g]), count=cnt[g])
    return out


Q1_OUT = ["sum_qty", "sum_base_price", "sum_disc_price", "sum_charge", "avg_qty", "avg_price", "avg_disc"]
Q1_SCALE = [2, 2, 4, 6, 6, 6, 6]


def q1_dump(res, out_dir):
    """The Final plan's result rows, ordered by (l_returnflag, l_linestatus), one float64 array per output column: the flags
    as their character codes, decimals and doubles by value, count_order as a number."""
    import numpy as np
    rows = sorted(res.to_pylist(), key=lambda r: (r["col_0"], r["col_1"]))
    os.makedirs(out_dir, exist_ok=True)
    names = ["l_returnflag", "l_linestatus"] + Q1_OUT + ["count_order"]
    for j, name in enumerate(names):
        v = [ord(r[f"col_{j}"]) if j < 2 else float(r[f"col_{j}"]) for r in rows]
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))


def q1_compare(tpch, res, expected):
    """res: the Final plan's Arrow table; expected: {group index: dict}.  True iff all eight outputs of every group agree."""
    got = {(r["col_0"], r["col_1"]): r for r in res.to_pylist()}
    if len(got) != len(expected):
        return False
    ok = True
    for g, e in expected.items():
        r = got.get((tpch.RETURNFLAGS[g // 2], tpch.LINESTATUS[g % 2]))
        if r is None:
            return False
        for j, (name, sc) in enumerate(zip(Q1_OUT, Q1_SCALE)):
            want = e[name] if name in e else e["sum_base"]          # the oracle names the second sum `sum_base`
            ok &= int(r[f"col_{2 + j}"].scaleb(sc)) == want
        ok &= r["col_9"] == e["count"]
    return bool(ok)


def workload_q1(args, env):
    import numpy as np
    import pyarrow as pa
    torch, native, rank, world, device, comm = env["torch"], env["native"], env["rank"], env["world"], env["device"], env["comm"]
    from comet_b200 import proto as P, tpch
    from comet_b200.dist import table_from_bytes, table_to_bytes
    variant, n = args.variant, args.rows
    cols = gen_device(torch, n, 42 + rank, device)
    money = build_columns(torch, cols, variant)
    partial_plan, final_plan = tpch.q1_partial_plan(variant), tpch.q1_final_plan(variant)
    chunk_rows = min(args.chunk_rows, 2_000_000_000)
    table = bind_table(native, P, tpch, variant, n, money, cols)   # the resident columns are bound once; every step runs fresh plans over them

    def gather_states(state):
        """Partial states of all ranks on rank 0: ONE fixed-size NCCL all-gather of the serialized state batch (a few rows) through
        the library's communicator."""
        if world == 1:
            return [state]
        blobs = comm.allgather_small(table_to_bytes(state) if state is not None else b"")
        return [table_from_bytes(b) for b in blobs if b] if rank == 0 else None

    def finish(state):
        states = gather_states(state)
        return run_final(native, pa, final_plan, states) if rank == 0 else (None, None)

    def step_resident():
        state, st = run_partial(native, partial_plan, table, chunk_rows)
        res, st2 = finish(state)
        return res, st, st2

    sampler = ClockSampler(env["local_rank"])
    if rank == 0:
        sampler.start()
    elapsed, outs = timed_region(env, sampler if rank == 0 else None, step_resident, args.warmup, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    pipe_ms = sum(o[1]["pipeline_ms"] for o in outs)
    pipe_launches = sum(o[1]["pipeline_launches"] for o in outs)
    launches = sum(o[1]["kernel_launches"] + (o[2]["kernel_launches"] if o[2] else 0) for o in outs)
    res = outs[-1][0]
    if rank == 0 and args.dump_outputs:
        q1_dump(res, args.dump_outputs)

    # ---- checks (outside the timed region) ---------------------------------------------------------------------------------------
    # (1) every output of every group at FULL size against exact torch int64 arithmetic (rank 0's partition; N = 1 only: the final
    #     result of an N-rank run merges all partitions)
    # (2) a 64 Mi-row prefix against the oracle, all eight outputs
    checks = {}
    if rank == 0 and variant == "dec" and not args.no_check:
        if world == 1:
            checks["full_size_all_outputs_vs_torch_int64"] = q1_compare(tpch, res, q1_expected_from_torch(torch, cols, tpch.Q1_CUTOFF))
        from oracle import oracle
        oracle.build()
        m = min(n, 1 << 26)
        sub_cols = {k: v[:m] for k, v in cols.items()}
        sub_money = {k: v[:m] for k, v in money.items()}
        t_sub = bind_table(native, P, tpch, variant, m, sub_money, sub_cols)
        st_sub, _ = run_partial(native, partial_plan, t_sub, chunk_rows)
        res_sub, _ = run_final(native, pa, final_plan, [st_sub])
        d = oracle.dec_from_i64
        h = {k: v.cpu().numpy() for k, v in sub_cols.items()}
        exp = oracle.q1_dec(d(h["l_quantity"]), d(h["l_extendedprice"]), d(h["l_discount"]), d(h["l_tax"]), h["l_shipdate"], h["l_returnflag"].view(np.uint8),
                            h["l_linestatus"].view(np.uint8), 3, 2, tpch.Q1_CUTOFF, usable_cores())
        checks["oracle_all_outputs_rows"] = m
        checks["oracle_all_outputs_ok"] = q1_compare(tpch, res_sub, {g: e for g, e in enumerate(exp) if e is not None})
        del h, t_sub

    # ---- end-to-end leg: HOST buffers -> C ABI -> result (per rank; rank 0 merges) ------------------------------------------------
    e2e, e2e_extra, host = None, {}, None
    numa = NumaLocal(env["local_rank"], enabled=not args.no_numa)
    if not args.no_e2e:
        with numa:
            batches, host = host_arrow_batches(torch, pa, tpch, variant, money, cols, args.e2e_batch_rows, pin=args.e2e_input in ("arrow", "both"))

        def timed_e2e(step_fn, steps):
            step_fn()  # warm-up (JIT variants, first use of the cached scan blocks)
            step_fn()
            env["barrier"]()
            t1 = time.perf_counter()
            h2d = d2h = 0
            for _ in range(steps):
                st, st2 = step_fn()
                h2d += st["h2d_bytes"] + (st2["h2d_bytes"] if st2 else 0)
                d2h += st["d2h_bytes"] + (st2["d2h_bytes"] if st2 else 0)
            env["barrier"]()
            el = env["max_over_ranks"](time.perf_counter() - t1)
            return {"value": world * n * steps / el, "unit": "rows/s", "h2d_bytes_per_step": h2d // steps, "d2h_bytes_per_step": d2h // steps,
                    "steps": steps, "ms_per_step": 1e3 * el / steps}

        if args.e2e_input in ("arrow", "both"):
            def step_arrow():
                state, st = run_partial(native, partial_plan, batches, 1 << 26)
                return st, finish(state)[1]
            r = timed_e2e(step_arrow, args.e2e_steps)
            r["input"] = f"pinned host Arrow batches of {args.e2e_batch_rows} rows via ArrowArrayStream, 64 Mi-row device chunks"
            e2e_extra["e2e_arrow"] = r
            e2e = r
        if args.e2e_input in ("parquet", "both"):
            import concurrent.futures as cf
            import pyarrow.parquet as pq
            tbl = pa.Table.from_batches(batches)
            nf = max(1, min(args.parquet_files, n // (1 << 20) or 1))
            per = (n + nf - 1) // nf

            def write_slice(i):
                sink = pa.BufferOutputStream()
                pq.write_table(tbl.slice(i * per, per), sink, row_group_size=1 << 20, compression=args.parquet_compression,
                               use_dictionary=args.parquet_dictionary == "all" or ["l_returnflag", "l_linestatus"], data_page_version="1.0", store_decimal_as_integer=True)
                return sink.getvalue()
            t_w = time.perf_counter()
            with cf.ThreadPoolExecutor(max_workers=nf) as ex:
                bufs = list(ex.map(write_slice, range(nf)))
            files, pinned = [], []
            with numa:
                for i, b in enumerate(bufs):
                    h = torch.empty(b.size, dtype=torch.uint8, pin_memory=True)
                    h.numpy()[:] = np.frombuffer(b, dtype=np.uint8)
                    pinned.append(h)
                    files.append(native.register_memory_file(f"lineitem-r{rank}-{i}", h))
            del bufs, tbl
            pq_bytes = sum(h.numel() for h in pinned)
            pq_plan = tpch.q1_partial_plan(variant, scan=tpch.q1_native_scan(variant, files))

            def step_parquet():
                state, st = run_partial(native, pq_plan, None, args.e2e_chunk_rows)
                return st, finish(state)[1]
            r = timed_e2e(step_parquet, args.e2e_steps)
            r["input"] = (f"{nf} Parquet file images in pinned host memory ({pq_bytes / 1e9:.2f} GB: compression {args.parquet_compression}, 1 Mi-row row groups, INT64 decimals, "
                          f"dictionary={args.parquet_dictionary}; written in {time.perf_counter() - t_w:.1f} s, not timed) through NativeScan in {args.e2e_chunk_rows}-row device batches "
                          f"(double-buffered upload, blocks allocated once); pages decoded on the device"
                          + (f"; host buffers on NUMA node {numa.node} next to the GPU" if numa.cpus else ""))
            r["pcie_GBps"] = r["h2d_bytes_per_step"] / (r["ms_per_step"] * 1e-3) / 1e9
            e2e_extra["e2e_parquet"] = r
            e2e = r

    # ---- CPU baseline (rank 0, N=1): oracle port on the host cores, bounded sample -------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and variant == "dec":
        from oracle import oracle
        oracle.build()
        m = min(n, 200_000_000)
        if host is None:
            _, host = host_arrow_batches(torch, pa, tpch, variant, {k: v[:m] for k, v in money.items()}, {k: v[:m] for k, v in cols.items()}, m, pin=False)
        hv = lambda k: host[k].numpy()[:m]
        a = (hv("l_quantity").view(np.uint64), hv("l_extendedprice").view(np.uint64), hv("l_discount").view(np.uint64), hv("l_tax").view(np.uint64),
             hv("l_shipdate"), hv("l_returnflag").view(np.uint8), hv("l_linestatus").view(np.uint8), 3, 2, tpch.Q1_CUTOFF)
        a = tuple(oracle.numa_spread(x, usable_cores()) if isinstance(x, np.ndarray) else x for x in a)
        cores = best_thread_count(lambda c: oracle.q1_dec(*a, c), usable_cores())
        reps, tc = 0, time.perf_counter()
        while reps < 3 or time.perf_counter() - tc < 5.0:
            oracle.q1_dec(*a, cores)
            reps += 1
            if time.perf_counter() - tc > 30.0:
                break
        dtc = time.perf_counter() - tc
        cpu = {"value": m * reps / dtc, "unit": "rows/s", "cores": cores, "kind": "port",
               "sample": f"{m} rows x {reps} passes, oracle/comet_oracle.c co_q1_dec (OpenMP, partial per thread + final merge)"}

    if rank == 0:
        peak, peak_src = measured_peak()
        ms_per_launch = pipe_ms / max(pipe_launches, 1)
        achieved = BYTES_PER_ROW[variant] * (n * args.steps / max(pipe_launches, 1)) / (ms_per_launch * 1e-3) / 1e9 if pipe_launches else 0.0
        line = {
            "metric": METRIC, "value": world * n * args.steps / elapsed, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i128" if variant == "dec" else "f64", "data": "synthetic",
            "config": {"workload": f"TPC-H Q1 (filter l_shipdate <= 1998-09-24 + group-by 2 keys, 4 sum + 3 avg + count) over SF100-shaped lineitem, "
                                   f"{'DECIMAL(12,2)' if variant == 'dec' else 'DOUBLE'} money columns, Arrow columns resident in HBM",
                       "rows_per_gpu": n, "variant": variant,
                       "parallelism": f"round-robin partitions x{world}; partial states gathered on rank 0 by one NCCL all-gather of a fixed-size buffer (library communicator), merged by the Final plan",
                       "l2": f"inputs ({BYTES_PER_ROW[variant] * n / 1e9:.1f} GB per GPU) exceed L2; no flush needed",
                       "checks": checks},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": profiled_traffic(n, variant),
                         "kernel": "cb_pipeline_agg (fused scan+filter+project+partial aggregate)", "ms_per_launch": ms_per_launch,
                         "spec_peak": 8000.0, "frac_of_spec_peak": achieved / 8000.0,
                         "algorithmic_bytes_per_row": BYTES_PER_ROW[variant], "peak_source": peak_src},
            "gpu_launches": launches, "clocks": clocks, "step_ms": env["step_ms"],
        }
        if e2e:
            line["e2e"] = e2e
            if len(e2e_extra) > 1:
                line.update(e2e_extra)
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))


# =====================================================================================================================
# group-by (BASELINE.json configs[3]): GROUP BY l_orderkey SUM(l_extendedprice), hash-repartition across the GPUs
# =====================================================================================================================
GROUPBY_METRIC = "rows/sec on GROUP BY l_orderkey SUM(l_extendedprice) (hash-repartitioned across GPUs)"


def workload_groupby(args, env):
    """Per rank: HashAggregate(Partial) [fused scan + hash-aggregate kernel] -> ShuffleWriter(HashPartitioning(l_orderkey, N))
    [murmur3 / pmod / stable counting sort on the device] -> cb200_exchange [NCCL over NVLink] -> HashAggregate(Final)."""
    import ctypes as C
    torch, native, rank, world, device, comm = env["torch"], env["native"], env["rank"], env["world"], env["device"], env["comm"]
    from comet_b200 import proto as P
    from comet_b200.dist import _DevPtr
    if comm is None:
        comm = native.Comm(0, 1, env["local_rank"])
    n = args.rows if args.rows != SF100_ROWS else 750_000_000   # SF1000 lineitem over 8 GPUs = 750 M rows per GPU
    dec = args.variant == "dec"
    g = torch.Generator(device=device)
    g.manual_seed(100 + rank)
    # clustered keys, ~4 lines per order (1..7); orders are dealt round-robin so that partitions hold disjoint keys (a row-group
    # partitioned, order-clustered lineitem)
    lines = torch.randint(1, 8, (n // 3 + 8,), generator=g, device=device)
    order = torch.repeat_interleave(torch.arange(lines.shape[0], device=device, dtype=torch.int64), lines)[:n].contiguous()
    keys = (order * world + rank).contiguous()
    n_groups_local = int(order[-1].item()) + 1
    del lines, order
    cents = (torch.randint(1, 51, (n,), generator=g, device=device) * torch.randint(90000, 210001, (n,), generator=g, device=device)).contiguous()
    if dec:
        val = to_dec128(torch, cents)
        m, sdt, w = P.DECIMAL(12, 2), P.DECIMAL(22, 2), 16
    else:
        val = (cents.to(torch.float64) / 100.0).contiguous()
        m, sdt, w = P.DOUBLE, P.DOUBLE, 8
    agg = P.hash_agg(P.scan([P.INT64, m]), [P.bound(0, P.INT64)], [P.agg_sum(P.bound(1, m), sdt)], P.PARTIAL)
    map_plan = P.shuffle_writer(agg, P.hash_partitioning([P.bound(0, P.INT64)], world))
    state_types = [P.INT64, sdt, P.BOOL] if dec else [P.INT64, sdt]
    final_plan = P.hash_agg(P.scan(state_types, source="shuffle"), [P.bound(0, P.INT64)], [P.agg_sum(P.unbound("c", m), sdt)], P.FINAL)
    cfg = {"spark.comet.b200.chunkRows": str(args.groupby_chunk_rows)}
    if os.environ.get("CB200_HASH_THREADS"):
        cfg["spark.comet.b200.hashThreads"] = os.environ["CB200_HASH_THREADS"]
    table = native.DeviceTable(n)
    table.add(P.INT64, keys.data_ptr(), 8, keep=keys)
    table.add(m, val.data_ptr(), w, keep=val)

    def view(ptr, nbytes):
        return torch.as_tensor(_DevPtr(ptr, nbytes), device=device) if nbytes else torch.empty(0, dtype=torch.uint8, device=device)

    py_trace = bool(os.environ.get("CB200_TRACE"))

    def step(keep_result=False):
        tm = [time.perf_counter()]
        p = native.Plan(map_plan, [table], config=cfg, device=DEVICE)
        tm.append(time.perf_counter())
        rows_state, _ = p.execute_device()
        tm.append(time.perf_counter())
        st = p.stats()
        recv, xs = comm.exchange(p)
        tm.append(time.perf_counter())
        p.release()
        tm.append(time.perf_counter())
        p2 = native.Plan(final_plan, [recv], config=cfg, device=DEVICE)
        out = p2.execute_device()
        tm.append(time.perf_counter())
        n_out = out[0] if out else 0
        st2 = p2.stats()
        result = None
        if keep_result and out:
            kk = view(out[1][0].values, n_out * 8).view(torch.int64).clone()
            vv = view(out[1][1].values, n_out * (16 if dec else 8))
            vv = (vv.view(torch.int64).view(-1, 2)[:, 0] if dec else vv.view(torch.float64)).clone()
            result = (kk, vv)
        torch.cuda.synchronize()
        tm.append(time.perf_counter())
        p2.release()
        tm.append(time.perf_counter())
        recv.release()
        tm.append(time.perf_counter())
        if py_trace:
            names = ["create", "map.execute", "exchange", "map.release", "final.create+execute", "sync", "final.release", "recv.release"]
            print("[py trace] " + "  ".join(f"{k} {1e3 * (b - a):.2f}" for k, a, b in zip(names, tm, tm[1:])), file=sys.stderr)
        return dict(rows_state=rows_state, n_out=n_out, st=st, st2=st2, xs=xs, result=result)

    sampler = ClockSampler(env["local_rank"])
    use_sampler = rank == 0 and not os.environ.get("CB200_BENCH_NO_SAMPLER")
    if use_sampler:
        sampler.start()
    elapsed, outs = timed_region(env, sampler if use_sampler else None, step, args.warmup, args.steps)
    clocks = sampler.stop() if use_sampler else None
    last = outs[-1]

    # ---- checks: exact totals per key (N = 1), ownership + global checksums (any N) -------------------------------------------------
    checks = {}
    if not args.no_check:
        chk = step(keep_result=True)
        kk, vv = chk["result"]
        groups_total = env["sum_over_ranks"](int(kk.shape[0]))
        checks["groups_total"] = groups_total
        checks["groups_expected"] = env["sum_over_ranks"](n_groups_local)
        if dec:
            checks["sum_of_sums_matches_input"] = env["sum_over_ranks"](int(vv.sum().item())) == env["sum_over_ranks"](int(cents.sum().item()))
        if world == 1 and dec:
            exp = torch.zeros(n_groups_local + 1, dtype=torch.int64, device=device).scatter_add_(0, keys, cents)
            checks["every_group_exact_vs_torch"] = bool((exp[kk] == vv).all().item())
            del exp
        # every key this rank ended up with belongs to it: pmod(murmur3_i64(key, 42), world) == rank (oracle, 1 Mi-key sample)
        from oracle import oracle
        oracle.build()
        sample = kk[: 1 << 20].cpu().numpy()
        hashes = oracle.murmur3_column("i64", sample)
        owners = (hashes.astype("int64").astype("int32").astype("int64") % world + world) % world
        checks["owner_is_this_rank"] = bool(env["sum_over_ranks"](int((owners != rank).sum())) == 0)
        del kk, vv, chk

    # ---- e2e: host Arrow columns -> ArrowArrayStream -> same plans (bounded to e2e_rows: 24 B/row over PCIe) ------------------------
    e2e = None
    if not args.no_e2e:
        import pyarrow as pa
        me = min(n, args.groupby_e2e_rows)
        numa = NumaLocal(env["local_rank"], enabled=not args.no_numa)
        with numa:
            hk = torch.empty(me, dtype=torch.int64, pin_memory=True)
            hk.copy_(keys[:me])
            hvv = torch.empty((me, 2) if dec else (me,), dtype=val.dtype, pin_memory=True)
            hvv.copy_(val[:me])
        torch.cuda.synchronize()
        buf = lambda t: pa.foreign_buffer(t.data_ptr(), t.numel() * t.element_size(), base=t)
        arrs = [pa.Array.from_buffers(pa.int64(), me, [None, buf(hk)]), pa.Array.from_buffers(pa.decimal128(12, 2) if dec else pa.float64(), me, [None, buf(hvv)])]
        batches = pa.table(arrs, names=["k", "v"]).to_batches(max_chunksize=1 << 22)

        def step_e2e():
            p = native.Plan(map_plan, [batches], config={"spark.comet.b200.chunkRows": str(1 << 26)}, device=DEVICE)
            p.execute_device()
            st = p.stats()
            recv, _ = comm.exchange(p)
            p.release()
            p2 = native.Plan(final_plan, [recv], config=cfg, device=DEVICE)
            out = p2.execute_device()
            cnt = out[0] if out else 0
            first = view(out[1][1].values, 16).cpu() if out and cnt else None   # a result read back: the first group's sum
            st2 = p2.stats()
            p2.release()
            recv.release()
            return st, st2, first
        step_e2e()
        env["barrier"]()
        t1 = time.perf_counter()
        h2d = 0
        for _ in range(args.e2e_steps):
            st, st2, _ = step_e2e()
            h2d += st["h2d_bytes"]
        env["barrier"]()
        el = env["max_over_ranks"](time.perf_counter() - t1)
        e2e = {"value": world * me * args.e2e_steps / el, "unit": "rows/s", "h2d_bytes_per_step": h2d // args.e2e_steps, "d2h_bytes_per_step": 16 + 64,
               "steps": args.e2e_steps, "ms_per_step": 1e3 * el / args.e2e_steps, "rows_per_gpu": me,
               "input": f"pinned host Arrow batches (int64 key + {'Decimal128' if dec else 'float64'} value, 4 Mi rows each) via ArrowArrayStream; bounded to {me} rows per GPU"}

    if rank == 0:
        peak, peak_src = measured_peak()
        in_bytes = 8 + w
        part_ms, part_launches = last["st"]["pipeline_ms"], max(last["st"]["pipeline_launches"], 1)
        rows_per_launch = n / part_launches
        # algorithmic bytes of the partial kernel (stream mode: clustered keys, one state row per run of equal adjacent keys, no key
        # table): the input columns once + per state row its key word and its two 16-byte accumulator words, written once
        gbytes = 8 + 32
        alg = in_bytes * n + gbytes * last["rows_state"]
        achieved = alg / (part_ms * 1e-3) / 1e9
        xs = last["xs"]
        line = {
            "metric": GROUPBY_METRIC, "value": world * n * args.steps / elapsed, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i128" if dec else "f64", "data": "synthetic",
            "config": {"workload": f"GROUP BY l_orderkey SUM(l_extendedprice), {n} rows per GPU (SF1000 lineitem / 8), ~4 clustered lines per order, {'DECIMAL(12,2)' if dec else 'DOUBLE'}; "
                                   "columns resident in HBM; Partial hash aggregate -> hash partition (murmur3 seed 42, pmod N) -> NCCL exchange inside the library -> Final hash aggregate",
                       "rows_per_gpu": n, "state_rows_per_gpu": last["rows_state"], "groups_per_gpu_after_exchange": last["n_out"],
                       "parallelism": f"hash-repartition x{world} (cb200_exchange: one ncclAllGather of counts + one grouped send/recv per state column; {native.nccl_info()})",
                       "l2": f"inputs ({in_bytes * n / 1e9:.1f} GB per GPU) and the hash table exceed L2; no flush needed", "checks": checks},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "kernel": "cb_pipeline_agg [CB_HASH, CB_STREAM] (fused scan + run-combining partial aggregate)", "ms_per_launch": part_ms / part_launches,
                         "rows_per_launch": rows_per_launch, "algorithmic_bytes": f"{in_bytes} B/row input + {gbytes} B per state row (key + accumulator words)",
                         "peak_source": peak_src},
            "phases_ms": {"partial_kernels": part_ms, "final_kernels": last["st2"]["pipeline_ms"], "exchange_payload": xs["payload_ms"]},
            "exchange": {"bytes_sent_per_gpu": xs["bytes_sent"], "bytes_received_per_gpu": xs["bytes_received"], "payload_ms": xs["payload_ms"],
                         "GBps_per_gpu": xs["bytes_sent"] / max(xs["payload_ms"], 1e-6) / 1e6, "nvlink_peak_GBps_per_direction": 900.0},
            "gpu_launches": sum(o["st"]["kernel_launches"] + o["st2"]["kernel_launches"] for o in outs), "clocks": clocks, "step_ms": env["step_ms"],
        }
        if e2e:
            line["e2e"] = e2e
        print(json.dumps(line))


# =====================================================================================================================
# Config 1 (filter + project) and Q6 (3-predicate filter + sum): BASELINE.json configs[0] / configs[2] on resident columns
# =====================================================================================================================
def workload_select_or_q6(args, env):
    import numpy as np
    import pyarrow as pa
    torch, native, rank, world, device = env["torch"], env["native"], env["rank"], env["world"], env["device"]
    from comet_b200 import proto as P, tpch
    variant = args.variant
    n = args.rows if args.rows != SF100_ROWS else (1_000_000_000 if args.workload == "config1" else SF100_ROWS)
    g = torch.Generator(device=device)
    g.manual_seed(7 + rank)
    ri = lambda lo, hi, dt=torch.int64: torch.randint(lo, hi, (n,), generator=g, device=device, dtype=dt)
    qty_units = ri(1, 51)
    price = qty_units * ri(90000, 210001)
    qty = qty_units * 100
    del qty_units
    ship = ri(8036, 10562, torch.int32)
    mk = (lambda c: to_dec128(torch, c)) if variant == "dec" else (lambda c: (c.to(torch.float64) / 100.0))
    m = tpch.D12 if variant == "dec" else P.DOUBLE
    w = 16 if variant == "dec" else 8
    t = native.DeviceTable(n)
    if args.workload == "config1":
        q_, p_ = mk(qty), mk(price)
        del qty, price
        t.add(m, q_.data_ptr(), w, keep=q_).add(m, p_.data_ptr(), w, keep=p_).add(P.DATE, ship.data_ptr(), 4, keep=ship)
        plan = tpch.config1_plan(variant)
        sel = float((ship < tpch.DATE_1998_09_02).float().mean().item())
        bytes_row = 4 + 2 * w + sel * w
        metric = "rows/sec on filter+project (Config 1: SELECT l_quantity*l_extendedprice WHERE l_shipdate < '1998-09-02')"
        kernel = "cb_select_count + k_scan + cb_pipeline_select (two streaming passes, stable compaction)"
    else:
        disc = ri(0, 11)
        q_, p_, d_ = mk(qty), mk(price), mk(disc)
        del qty, price, disc
        t.add(m, q_.data_ptr(), w, keep=q_).add(m, p_.data_ptr(), w, keep=p_).add(m, d_.data_ptr(), w, keep=d_).add(P.DATE, ship.data_ptr(), 4, keep=ship)
        plan = tpch.q6_partial_plan(variant)
        bytes_row = 4 + 3 * w
        metric = "rows/sec on TPC-H Q6 filter+sum"
        kernel = "cb_pipeline_agg (ungrouped)"
    cfg = {"spark.comet.b200.chunkRows": str(1 << 31)}

    def step():
        with native.Plan(plan, [t], config=cfg, device=DEVICE) as p:
            out = p.execute_device()
            st = p.stats()
            rows = out[0] if out else 0
        return rows, st
    sampler = ClockSampler(env["local_rank"])
    if rank == 0:
        sampler.start()
    elapsed, outs = timed_region(env, sampler if rank == 0 else None, step, args.warmup, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        peak, peak_src = measured_peak()
        pipe_ms = sum(o[1]["pipeline_ms"] for o in outs) / len(outs)
        achieved = bytes_row * n / (pipe_ms * 1e-3) / 1e9
        line = {"metric": metric, "value": world * n * args.steps / elapsed, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "i128" if variant == "dec" else "f64", "data": "synthetic",
                "config": {"workload": f"{args.workload} over {n} resident rows per GPU, variant {variant}", "rows_per_gpu": n, "rows_out": outs[-1][0], "parallelism": f"replicas x{world}",
                           "l2": "inputs exceed L2; no flush needed"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "kernel": kernel,
                             "ms_pipeline_kernels_per_step": pipe_ms, "spec_peak": 8000.0, "frac_of_spec_peak": achieved / 8000.0, "algorithmic_bytes_per_row": bytes_row,
                             "peak_source": peak_src},
                "gpu_launches": sum(o[1]["kernel_launches"] for o in outs), "clocks": clocks, "step_ms": env["step_ms"]}
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="q1", choices=["q1", "groupby", "config1", "q6"],
                    help="q1 = BASELINE.json configs[1] (the driver's default); groupby = configs[3] (hash-repartition across GPUs); config1 / q6 = configs[0] / [2] kernels on resident columns")
    ap.add_argument("--variant", default="dec", choices=["dec", "f64"])
    ap.add_argument("--rows", type=int, default=int(os.environ.get("CB200_BENCH_ROWS", SF100_ROWS)))
    ap.add_argument("--ref-rows", type=int, default=60_000_000)
    ap.add_argument("--chunk-rows", type=int, default=1 << 30)
    ap.add_argument("--groupby-chunk-rows", type=int, default=1 << 28)
    ap.add_argument("--groupby-e2e-rows", type=int, default=1 << 28)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-batch-rows", type=int, default=1 << 22)
    ap.add_argument("--e2e-chunk-rows", type=int, default=1 << 26, help="rows per device batch of the Parquet e2e leg (upload of batch k+1 overlaps decode+aggregate of batch k)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="do not move the rank next to its GPU's NUMA node while pinned host buffers are allocated")
    ap.add_argument("--e2e-input", default="parquet", choices=["parquet", "arrow", "both"])
    ap.add_argument("--parquet-files", type=int, default=16)
    ap.add_argument("--parquet-dictionary", default="all", choices=["all", "flags"],
                    help="all = writer default of Spark/parquet-mr and pyarrow (dictionary-encode every column, PLAIN fallback); flags = PLAIN numerics")
    ap.add_argument("--parquet-compression", default="NONE", choices=["NONE", "SNAPPY"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the Q1 result of the last timed step as DIR/<output>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "q1"):
        ap.error("--dump-outputs writes the result of the b200 q1 workload")
    if os.environ.get("CB200_BENCH_TRACE_S"):          # debugging aid: dump every thread's Python stack every N seconds to stderr
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["CB200_BENCH_TRACE_S"]), repeat=True)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    private_jit_cache()
    env = setup(args)
    if args.workload == "q1":
        workload_q1(args, env)
    elif args.workload == "groupby":
        workload_groupby(args, env)
    else:
        workload_select_or_q6(args, env)
    if env["comm"] is not None:
        env["comm"].destroy()
    if env["world"] > 1:
        env["dist"].destroy_process_group()


if __name__ == "__main__":
    main()
