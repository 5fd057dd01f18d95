"""bench.py — samples/sec of the DLRM-Criteo train step (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" = one pass of the hot path over one synthetic Criteo batch: KJT scan -> (bucketize + all-to-all at
N>1) -> pooled gather -> DLRM dot interaction + dense towers -> BCE loss -> backward with the fused sparse
Adagrad update -> dense Adam step.  fp32 everywhere (TF32 off, as the reference's default train.proto:14).
Workload at N=1: BASELINE.json configs[1] (examples/dlrm_criteo.config, full hash sizes, row-wise, B=65536
per rank) — it fits one GPU (12.2 GiB tables + 12.2 GiB Adagrad state).

N>1 (torchrun): tables sharded --sharding {row_wise,table_wise,mixed}, exchange over peer memory (default) or NCCL;
the line then carries `verify` (the sharded step against its unsharded twin, run inside this process) and an NVLink
roofline.  Other models of BASELINE.json: --model deepfm_criteo | mmoe_taobao | multi_tower_din_taobao.

Prints ONE JSON line (see DESIGN.md §7 for every field).
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

if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the ONE JSON line (NCCL prints its version banner there)
os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")   # CPU baseline: idle OpenMP workers must not spin
os.environ.setdefault("GOMP_SPINCOUNT", "0")
if "--impl" in sys.argv and "reference" in sys.argv:
    # the CPU arm uses all the host threads it can use; torchrun's blanket OMP_NUM_THREADS=1 is a launcher default,
    # not a user choice (libgomp reads the variable once, when torch loads it below)
    if "OMP_NUM_THREADS" not in os.environ or "TORCHELASTIC_RUN_ID" in os.environ or "LOCAL_RANK" in os.environ:
        os.environ["OMP_NUM_THREADS"] = str(min(os.cpu_count() or 1, 32))

import torch  # noqa: E402

METRIC = "samples/sec (DLRM-Criteo synth, train step fwd+bwd+optimizer)"
UNIT = "samples/s"
# DLRM-Criteo (F=26, L=1, D=16) per-sample algorithmic bytes, SURVEY.md §8d — computed from the layout at run time:
#   gather 1664 rows + 1664 pooled write + 208 ids + 104 lengths = 3640 B; backward 1664 grad + 26*4*64 RMW + 208 = 8528 B
NVLINK_GBS = 900.0     # NVLink 5, per direction per GPU (nominal; B200_PROFILING.md) — the N>1 roofline's denominator


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused backward's / the gather's kernels, as
    written by scripts/ncu_traffic.py from an `ncu --set full` capture of THIS build (the file carries a hash of the
    kernel sources it was taken on; a stale file is ignored)."""
    import hashlib

    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None
    try:
        d = json.load(open(path))
        h = hashlib.sha256()
        for fn in ("tzk_bwd.cu", "tzk_gather.cu", "tzk_common.cuh"):
            h.update(open(os.path.join(ROOT, "torcheasyrec_b200", "csrc", fn), "rb").read())
        return d if d.get("source_sha16") == h.hexdigest()[:16] else None
    except Exception:
        return None


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-size", type=int, default=65536, help="per-rank batch (data_config.batch_size)")
    ap.add_argument("--model", default="dlrm_criteo")
    ap.add_argument("--id-dist", default="uniform", choices=["uniform", "zipf"])
    ap.add_argument("--max-rows", type=int, default=0, help="cap every table (0 = full hash sizes)")
    ap.add_argument("--ring", type=int, default=8, help="distinct input batches rotated through the steps")
    ap.add_argument("--cpu-batch", type=int, default=8192, help="samples per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-zipf", action="store_true", help="skip the second (Zipf-id) timing of the same step")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the measurement-only extras (blocking-loss-read e2e variant)")
    ap.add_argument("--sharded-mode", default="auto", choices=["auto", "graph", "eager"],
                    help="N>1: 'graph' = fixed-capacity exchange captured in one CUDA graph, 'eager' = step by step "
                         "(auto: graph unless the model has sequence features)")
    ap.add_argument("--static-capacity", type=float, default=1.25,
                    help="head-room of the fixed-capacity wire buffers over the expected ids per destination")
    ap.add_argument("--exchange", default="peer", choices=["nccl", "peer"],
                    help="sharded runs: the peer-memory kernels of csrc/tzk_peer.cu (default), or NCCL all-to-alls")
    ap.add_argument("--sharding", default="row_wise", choices=["row_wise", "table_wise", "mixed"],
                    help="placement of the tables at N>1 (BASELINE configs: dlrm row_wise, deepfm table_wise, mmoe mixed)")
    ap.add_argument("--rw-min-rows", type=int, default=200000, help="mixed: tables with at least this many rows go row-wise")
    ap.add_argument("--trace", default="", help="after the timed runs: chrome trace of 3 steps of rank 0 (torch.profiler) "
                                                "written to this path — diagnosis only, never a reported number")
    ap.add_argument("--no-verify", action="store_true",
                    help="N>1: skip the in-process parity check of the sharded step against its unsharded twin")
    ap.add_argument("--force-sharded", action="store_true",
                    help="N=1 only: still go through bucketize / all-to-all / owner gather (1-rank process group)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps: what the last timed step left for its caller (loss, dense parameters, "
                         "a fixed sample of rows of every table and of its optimizer state) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus > 1 or args.force_sharded):
        ap.error("--dump-outputs: single-GPU unsharded runs of --impl ours only")
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0) -> None:
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) >= 8 and r[4 + j] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ---------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the same step on host cores
# ---------------------------------------------------------------------------------------------------------
def cpu_step_rate(model: str, batch: int, steps: int, warmup: int, max_rows: int, id_dist: str):
    """Times the CPU restatement of the step (torch-CPU dense towers + oracle sparse path)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_backend import OracleKernels

    from torcheasyrec_b200 import functional as Fn
    from torcheasyrec_b200.engine import Pipeline

    # thread scan on a 128-core host (scripts/cpu_threads.py, profiles/README.md): 8 -> 237k, 16 -> 307k,
    # 32 -> 313k, 64 -> 271k, 128 -> 31k samples/s; beyond 32 the two OpenMP pools fight each other
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    os.environ["OMP_NUM_THREADS"] = str(cores)
    pipe = Pipeline(model, device="cpu", max_rows=max_rows or None)
    batches = [pipe.synthetic_batch(batch, seed=100 + i, id_dist=id_dist) for i in range(2)]
    backend = OracleKernels(use_c=True)   # C/OpenMP restatement when oracle/libtzk_oracle.so is built
    with Fn.use_backend(backend):
        for i in range(warmup):
            pipe.eager_step(batches[i % 2])
        t0 = time.perf_counter()
        for i in range(steps):
            pipe.eager_step(batches[i % 2])
        dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps * 1e3, cores, backend.name


def run_reference(args):
    """The reference's CPU path of the same step (`kind: "port"`: tzrec's own path needs the torchrec / fbgemm wheels,
    which cannot be installed offline — DESIGN.md §7): this repo's Pipeline / model shells stepped with the oracle
    (oracle/tzk_oracle.c, OpenMP) as the sparse backend and torch-CPU dense towers, on all the host threads that help
    (capped at 32: measured scan in profiles/README.md).  Honours --steps / --warmup; every step is a bounded sample of
    --cpu-batch samples of the workload (a 65536-sample step takes ~0.25 s on 32 threads)."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    import psutil

    # full hash sizes need 2 x 12.2 GiB of host RAM (tables + Adagrad state); cap them if the box is small
    max_rows = args.max_rows
    note = f"tables capped at {max_rows} rows" if max_rows else "full hash sizes"
    if not max_rows and psutil.virtual_memory().available < 40 * 2 ** 30:
        max_rows, note = 4_000_000, "tables capped at 4M rows (host RAM < 40 GiB)"
    steps, warm = max(1, args.steps), max(1, min(args.warmup, 5))
    rate, ms, cores, kind = cpu_step_rate(args.model, args.cpu_batch, steps, warm, max_rows, args.id_dist)
    extras = {}
    try:    # BASELINE.json configs[0]: DeepFM, 1k-row tables, batch 512 (the reference's own CPU-runnable case)
        r0, ms0, c0, _ = cpu_step_rate("deepfm_criteo", 512, max(steps, 10), 2, 1000, "uniform")
        extras["configs0_deepfm_1k_rows_b512"] = {"value": r0, "unit": UNIT, "ms_per_step": ms0, "cores": c0,
                                                  "note": "examples/deepfm_criteo.config, every table 1000 rows, "
                                                          "batch 512, world_size 1, oracle port"}
    except Exception as e:   # noqa: BLE001
        extras["configs0_deepfm_1k_rows_b512"] = {"failed": repr(e)[:200]}
    try:
        extras["embedding_bag_stock_cpu"] = _embedding_bag_line(args.cpu_batch, max_rows)
    except Exception as e:   # noqa: BLE001
        extras["embedding_bag_stock_cpu"] = {"failed": repr(e)[:200]}
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model}: examples/{args.model}.config, {note}, sparse Adagrad lr=1e-3 fused in "
                               f"backward + dense Adam, ids {args.id_dist}",
                   "per_step_samples": args.cpu_batch,
                   "note": "bounded sample: each step is --cpu-batch samples of the GPU arm's per-rank batch"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{steps} steps of {args.cpu_batch} samples ({warm} warm-up); this repo's model shells + "
                                   "torch-CPU dense towers + oracle/ sparse path (C/OpenMP restatement); the reference's "
                                   "own path needs torchrec/fbgemm wheels that are not installable offline"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "extras": extras,
    }
    _print_line(line)


def _embedding_bag_line(batch: int, max_rows: int):
    """The 'best stock CPU kernel' line BASELINE.md §3 promised: torch.nn.functional.embedding_bag (sum) over the 26
    Criteo tables, forward only, same ids as the oracle's pooled lookup timed beside it."""
    import numpy as np

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_backend import OracleKernels

    from torcheasyrec_b200.engine import Pipeline

    pipe = Pipeline("dlrm_criteo", device="cpu", max_rows=min(max_rows or 4_000_000, 4_000_000))
    ebc = pipe.model.sparse_collections()[0]
    b = pipe.synthetic_batch(batch, seed=5)
    kjt = ebc._select(b.sparse_features[sorted(b.sparse_features)[0]])
    ids, off = kjt.values(), kjt.offsets()
    tabs = [ebc.table_weight(t) for t in range(len(ebc._configs))]
    F = len(tabs)

    def stock():
        return torch.cat([torch.nn.functional.embedding_bag(ids[f * batch:(f + 1) * batch], tabs[f],
                                                            torch.arange(batch), mode="sum") for f in range(F)], dim=1)

    k = OracleKernels(use_c=True)

    def ours():
        return k.pooled_gather_fwd(ebc.weights.data, ebc.layout, ids, off, batch)

    assert np.array_equal(stock().numpy(), ours().numpy())
    res = {}
    for name, fn in (("F.embedding_bag", stock), ("oracle pooled_lookup", ours)):
        fn()
        t0 = time.perf_counter()
        n = 5
        for _ in range(n):
            fn()
        dt = (time.perf_counter() - t0) / n
        res[name] = {"ms": dt * 1e3, "lookups_per_s": F * batch / dt}
    res["note"] = f"pooled lookup only (forward), 26 tables (<= 4M rows each), {batch} samples, {torch.get_num_threads()} threads"
    return res


# ---------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------
def time_kernel(fn, iters: int):
    """Average duration (ms) of `fn` launches, CUDA events on the launching (current) stream."""
    for i in range(3):          # untimed: lazy module loads, first-touch allocations of the outputs
        fn(i)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    torch.cuda.synchronize()
    for i in range(iters):
        ev[i][0].record()
        fn(i)
        ev[i][1].record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / iters


def run_ours(args):
    rank, local_rank, world = dist_env()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    sharded = world > 1 or args.force_sharded
    if sharded:
        import torch.distributed as dist

        if world == 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29533")
            dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
        else:
            dist.init_process_group("nccl", device_id=dev)
    from torcheasyrec_b200.engine import GraphedTrainStep, Pipeline
    from torcheasyrec_b200.kernels import default_kernels

    B, K, W = args.batch_size, args.steps, max(args.warmup, 3)
    # ---- N>1: the sharded step against its unsharded twin, inside this process (small tables, same plan / exchange) --
    verify = None
    if sharded and world > 1 and not args.no_verify:
        from torcheasyrec_b200.verify import verify_sharded

        try:
            worst = verify_sharded(args.model, dev, args.sharding, rw_min_rows=300 if args.sharding == "mixed" else 0,
                                   static_capacity=max(args.static_capacity, 2.5), exchange=args.exchange,
                                   max_rows=2000, batch=256)
            verify = {"status": "ok", "max_abs_dev": worst,
                      "what": "unsharded twin on the concatenated batch vs this sharded step (2000-row tables, 256 "
                              "samples per rank, 2 steps): logits, loss, every table, every dense parameter"}
        except Exception as e:   # noqa: BLE001 — reported in the line; the timing below still runs
            verify = {"status": "FAILED", "error": repr(e)[:400]}
        torch.cuda.synchronize()
    probe = Pipeline(args.model, device="cpu", max_rows=8) if args.sharded_mode == "auto" else None
    has_seq = bool(probe and any(f.is_sequence for f in probe.features))
    mode = args.sharded_mode if args.sharded_mode != "auto" else ("eager" if has_seq else "graph")
    graphed = mode == "graph"
    args._mode = mode
    pipe = Pipeline(args.model, device=dev, max_rows=args.max_rows or None,
                    sharding=args.sharding if sharded else None, rw_min_rows=args.rw_min_rows,
                    static_capacity=args.static_capacity if (sharded and (graphed or args.exchange == "peer")) else None,
                    exchange=args.exchange if sharded else "nccl")
    host = [pipe.synthetic_batch(B, seed=20260923 + rank * 1000 + i, id_dist=args.id_dist).pin_memory()
            for i in range(args.ring)]
    ring = [hb.to(dev) for hb in host]
    kern = default_kernels()
    if graphed:
        step = GraphedTrainStep(pipe, host[0], warmup=3)
        launches_before = kern.launches
        # count this step's own kernels once (eager replica of the captured step on the static inputs)
        step._fresh_kjt_caches()
        pipe.eager_step(step.static)
        launches_per_step = kern.launches - launches_before
    else:
        # variable-shape steps (sequence features; dynamic all-to-all splits) run eagerly instead of as one CUDA graph
        class EagerStep:
            def __init__(self):
                self.cur = None

            def load(self, batch, non_blocking=True):
                self.cur = batch.to(dev, non_blocking=non_blocking) if not batch.labels[pipe.labels[0]].is_cuda else batch
                for k, kjt in batch.sparse_features.items():
                    self.cur.sparse_features[k]._length_per_key = kjt._length_per_key

            def replay(self):
                return pipe.eager_step(self.cur)

        step = EagerStep()
        step.load(ring[0])
        launches_before = kern.launches
        step.replay()
        launches_per_step = kern.launches - launches_before
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM (device ring, D2D into the graph's static buffers) -----------------
    for i in range(W):
        step.load(ring[i % len(ring)])
        step.replay()
    barrier()
    clocks = ClockSampler(local_rank).start() if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step.load(ring[i % len(ring)])
        loss = step.replay()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs:      # before anything below steps the model again
        dump_outputs(args.dump_outputs, pipe, loss)
    # ---- e2e: pinned host batch -> H2D -> step -> loss back on the host, every step --------------------------
    # The H2D of batch i+1 runs on the copy stream while step i computes (graphed steps); the loss of EVERY step
    # reaches the host inside the timed region through a pinned D2H copy + event, read one step later so that the
    # host keeps enqueueing (what TrainPipelineSparseDist's progress() does with its batch queue).
    pin = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    evs = [torch.cuda.Event() for _ in range(2)]
    for i in range(2):
        step.load(host[i % len(host)])
        step.replay()
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    last = 0.0
    if graphed:
        step.prefetch(host[0])
    for i in range(K):
        if graphed:
            step.commit()
            step.prefetch(host[(i + 1) % len(host)])
        else:
            step.load(host[i % len(host)], non_blocking=True)
        loss = step.replay()
        pin[i % 2].copy_(loss, non_blocking=True)
        evs[i % 2].record()
        if i:
            evs[(i - 1) % 2].synchronize()
            last = float(pin[(i - 1) % 2])
    evs[(K - 1) % 2].synchronize()
    last = float(pin[(K - 1) % 2])
    g1.record()
    barrier()
    ms_e2e = g0.elapsed_time(g1)
    # ---- second id distribution (SURVEY.md §8d reports both): the same captured step on Zipf(1.05) ids -------
    zipf = None
    if args.id_dist == "uniform" and not args.no_zipf and not sharded:   # (row-wise blocks + Zipf overflow a fixed wire capacity)
        zring = [pipe.synthetic_batch(B, seed=20260923 + rank * 1000 + 500 + i, id_dist="zipf").to(dev)
                 for i in range(min(args.ring, 4))]
        for i in range(3):
            step.load(zring[i % len(zring)])
            step.replay()
        barrier()
        z0, z1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        z0.record()
        for i in range(K):
            step.load(zring[i % len(zring)])
            step.replay()
        z1.record()
        barrier()
        zipf = z0.elapsed_time(z1)
        del zring
    clk = clocks.stop() if clocks else None
    if args.trace:             # kernel timeline of a few steps (all ranks step, rank 0 records)
        from torch.profiler import ProfilerActivity, profile

        barrier()
        if rank == 0:
            with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
                for i in range(3):
                    step.load(ring[i % len(ring)])
                    step.replay()
                torch.cuda.synchronize()
            prof.export_chrome_trace(args.trace)
        else:
            for i in range(3):
                step.load(ring[i % len(ring)])
                step.replay()
        barrier()
    pipe.check_overflow()      # fixed-capacity exchange: no peer needed more than its wire capacity
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([ms_total, ms_e2e, zipf or 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e, zz = t.tolist()
        zipf = zz if zipf is not None else None
    args._zipf_ms = zipf
    args._verify = verify

    roofline, cpu = None, None
    if sharded:
        # ---- N>1 roofline: the requester-side gather against NVLink (rank 0 times it alone: no collective in it) ----
        try:
            if rank == 0:
                roofline = _peer_roofline(pipe, kern, ring, B, world, max(K, 10), ms_total / K)
        except Exception as e:   # noqa: BLE001
            roofline = {"failed": repr(e)[:300]}
        barrier()               # peers keep their symmetric buffers mapped until rank 0 is done
        if rank == 0:
            _emit(args, world, B, K, W, ms_total, ms_e2e, host, last, launches_per_step, clk, roofline, cpu, len(ring))
        return
    if rank != 0:
        return

    # ---- roofline of the dominant kernels (rank 0, standalone launches on the same inputs) -----------------
    ebc = pipe.model.sparse_collections()[0]
    lay = ebc.layout
    dg = sorted(ring[0].sparse_features)[0]
    kjts = [ebc._select(b.sparse_features[dg]) for b in ring]
    offs = [kern.lengths_to_offsets(k.lengths()) for k in kjts]
    ids = [k.values() for k in kjts]
    out = torch.empty((B, lay.total_dim), device=dev)
    grad = torch.randn((B, lay.total_dim), device=dev) * 1e-3
    R = len(ring)
    it = max(K, 10)
    # algorithmic bytes per sample of THIS collection and batch (SURVEY.md §8d): rows + pooled write + ids + lengths;
    # backward: gradient read + weight/state read+write of every looked-up row + ids.  Two variants of the backward
    # figure: U = every lookup hits a distinct row (SURVEY's upper bound, 26 rows/sample for Criteo) and U = the rows
    # this batch really touches (counted on the device below).
    lpk = kjts[0].length_per_key()
    nnz_f = [float(lpk[f]) / B for f in range(lay.num_features)]
    row_b = sum(l * d * 4 for l, d in zip(nnz_f, lay.dim))
    gather_b = row_b + sum(d * 4 for d in lay.dim) + sum(l * 8 for l in nnz_f) + 4 * lay.num_features
    spec = ebc.optimizer
    state_mult = {0: 2, 1: 4, 2: 2}[spec.kind]          # SGD w r+w; Adagrad w+state r+w; row-wise: w r+w (+8 B/row)
    fixed_b = sum(d * 4 for d in lay.dim) + sum(l * 8 for l in nnz_f)      # gradient read + ids
    bwd_b = fixed_b + state_mult * row_b + (8 * sum(nnz_f) if spec.kind == 2 else 0)
    uniq_row_bytes = 0.0                                  # sum over unique (table,row) of D*4, averaged over the ring
    for kj in kjts:
        o = 0
        for f in range(lay.num_features):
            n = lpk[f]
            uniq_row_bytes += float(torch.unique(kj.values()[o:o + n]).numel()) * lay.dim[f] * 4 / R
            o += n
    bwd_b_actual = fixed_b + (state_mult * uniq_row_bytes + (8 * uniq_row_bytes / (lay.dim[0] * 4) if spec.kind == 2 else 0)) / B
    fwd_ms = time_kernel(lambda i: kern.pooled_gather_fwd(ebc.weights.data, lay, ids[i % R], offs[i % R], B, out), it)
    bwd_ms = time_kernel(lambda i: kern.fused_bwd(spec.kind, True, grad, ebc.weights.data, ebc.opt_state, lay,
                                                  ids[i % R], offs[i % R], B, spec.lr, spec.eps, 1.0), it)
    # the same backward in its two halves: the id-only half (linearize + radix sort) runs on a side stream during
    # the forward pass inside the step, the gradient half is what sits on the step's critical path
    ws_b = torch.empty(kern.fused_bwd_workspace_bytes(lay, ids[0].numel()), dtype=torch.uint8, device=dev)
    sort_ms = time_kernel(lambda i: kern.fused_bwd_sort(True, lay, ids[i % R], offs[i % R], B, ws_b), it)
    kern.fused_bwd_sort(True, lay, ids[0], offs[0], B, ws_b)
    apply_ms = time_kernel(lambda i: kern.fused_bwd_apply(spec.kind, True, grad, ebc.weights.data, ebc.opt_state, lay,
                                                          offs[0], ids[0].numel(), B, spec.lr, spec.eps, 1.0, ws_b), it)
    peak, peak_src = measured_peak_gbs()
    fwd_gbs = gather_b * B / (fwd_ms * 1e-3) / 1e9
    bwd_gbs = bwd_b * B / (bwd_ms * 1e-3) / 1e9
    bwd_gbs_actual = bwd_b_actual * B / (bwd_ms * 1e-3) / 1e9
    dominant = ("tzk_fused_bwd (id half: linearize + radix sort + run lists; gradient half: fused_apply_kernel over the short-run list + long-run chunks)" if bwd_ms > fwd_ms
                else "pooled_gather_fwd_kernel")
    ach = bwd_gbs if bwd_ms > fwd_ms else fwd_gbs
    # dram__bytes_read.sum + dram__bytes_write.sum per launch, all kernels of the dominant op, from the ncu --set full
    # capture scripts/ncu_traffic.py took on this build (profiles/ncu_traffic.json; null when absent or stale)
    std = (args.model == "dlrm_criteo" and B == 65536 and not args.max_rows and args.id_dist == "uniform")
    nt = ncu_traffic() if std else None
    traffic = None
    if nt:
        traffic = nt.get("fused_bwd_bytes") if bwd_ms > fwd_ms else nt.get("pooled_gather_fwd_bytes")
    kernels = {
        "pooled_gather_fwd": {"ms": fwd_ms, "algorithmic_GBps": fwd_gbs, "frac": fwd_gbs / peak,
                              "row_read_GBps": row_b * B / (fwd_ms * 1e-3) / 1e9, "bytes_per_sample": gather_b},
        "fused_bwd": {"ms": bwd_ms, "algorithmic_GBps": bwd_gbs, "frac": bwd_gbs / peak, "bytes_per_sample": bwd_b,
                      "frac_upper_bound_U": bwd_gbs / peak, "frac_actual_U": bwd_gbs_actual / peak,
                      "bytes_per_sample_actual_U": bwd_b_actual,
                      "unique_rows_per_sample": uniq_row_bytes / (lay.dim[0] * 4) / B,
                      "sort_ms": sort_ms, "apply_ms": apply_ms,
                      "apply_frac": bwd_b * B / (apply_ms * 1e-3) / 1e9 / peak,
                      "note": "sort_ms overlaps the forward pass inside the step (side stream); apply_ms is the part on "
                              "the critical path; frac uses SURVEY §8d's upper bound (every lookup a distinct row), "
                              "frac_actual_U the rows this batch really touches"},
    }
    if args.model == "dlrm_criteo":
        Ns, D = lay.num_features, lay.dim[0]
        N = Ns + 1
        P = N * (N - 1) // 2
        dense16 = torch.randn(B, D, device=dev)
        sp = torch.randn(B, Ns * D, device=dev)
        d_out = torch.randn(B, P + 1 + D + Ns * D, device=dev)
        if_ms = time_kernel(lambda i: kern.dot_interact_fwd(dense16, sp, Ns, D, True, True, 4, 1), it)
        ib_ms = time_kernel(lambda i: kern.dot_interact_bwd(dense16, sp, d_out, Ns, D, True, True, 1), it)
        if_b = (N * D + P + D + Ns * D) * 4           # X in, [P | D | Ns*D] out  (SURVEY §8d: 1728 + 3132)
        ib_b = (N * D) * 4 * 2 + (P + D + Ns * D) * 4  # X in, d_out in, dX out
        kernels["dot_interact_fwd"] = {"ms": if_ms, "algorithmic_GBps": if_b * B / (if_ms * 1e-3) / 1e9,
                                       "frac": if_b * B / (if_ms * 1e-3) / 1e9 / peak, "bytes_per_sample": if_b}
        kernels["dot_interact_bwd"] = {"ms": ib_ms, "algorithmic_GBps": ib_b * B / (ib_ms * 1e-3) / 1e9,
                                       "frac": ib_b * B / (ib_ms * 1e-3) / 1e9 / peak, "bytes_per_sample": ib_b}
    roofline = {
        "bound": "hbm", "kernel": dominant, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
        "traffic": traffic,
        "traffic_note": (f"dram read+write bytes per launch summed over the kernels of the dominant op "
                         f"({', '.join(nt.get('kernels', []))}), ncu --set full via scripts/ncu_traffic.py "
                         f"({nt.get('when', '?')})" if traffic else
                         "null: no profiles/ncu_traffic.json taken on this build (scripts/ncu_traffic.py writes it)"),
        "peak_source": peak_src,
        "kernels": kernels,
        "share_of_step": {k: v["ms"] / (ms_total / K) for k, v in kernels.items()},
    }
    if not args.no_cpu_baseline and world == 1:
        try:
            steps_cpu = 2
            cpu_rows = args.max_rows or (4_000_000 if _small_host() else 0)
            rate, ms_cpu, cores, _ = cpu_step_rate(args.model, args.cpu_batch, steps_cpu, 1, cpu_rows, args.id_dist)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{steps_cpu} steps of {args.cpu_batch} samples of the same workload through the oracle "
                             f"restatement ({ms_cpu:.0f} ms/step)"}
        except Exception as e:  # the baseline is reported, never required
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    # ---- measurement-only extras (N=1): not part of value / e2e / roofline, and never allowed to fail the run ----
    if not args.no_extras and graphed:
        extras = {"note": "measurement-only; no reported number above depends on these"}
        try:
            extras["e2e_blocking"] = _e2e_blocking(step, host, K, B)
        except Exception as e:
            extras["e2e_blocking"] = {"failed": repr(e)[:200]}
        args._extras = extras
    _emit(args, world, B, K, W, ms_total, ms_e2e, host, last, launches_per_step, clk, roofline, cpu, len(ring))


DUMP_ROWS_PER_TABLE = 4096
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, pipe, loss: torch.Tensor) -> None:
    """Writes what a train step hands its caller, as of the last timed step: the loss and the model it updated — every
    dense parameter in full and, of every embedding table, the weights and optimizer state of a fixed sample of rows
    (all rows of a table up to DUMP_ROWS_PER_TABLE rows; otherwise that many draws of a generator seeded per table)."""
    import numpy as np

    out = {"loss": loss.detach().reshape(1)}
    dense = {id(p) for p in pipe.model.dense_parameters()}
    for name, p in pipe.model.named_parameters():
        if id(p) in dense:
            out[f"dense.{name}"] = p.detach()
    for c, coll in enumerate(pipe.model.sparse_collections()):
        for t in sorted(coll._table_off):
            n_rows = coll._table_rows[t]
            if n_rows <= DUMP_ROWS_PER_TABLE:
                rows = torch.arange(n_rows)
            else:
                gen = torch.Generator().manual_seed(1000 * c + t)
                rows = torch.randint(n_rows, (DUMP_ROWS_PER_TABLE,), generator=gen).unique()
            rows = rows.to(coll.weights.device)
            name = f"sparse{c}.{coll._configs[t].name}"
            out[f"{name}.weight"] = coll.table_weight(t).index_select(0, rows)
            state = coll.table_state(t)
            if state is not None:
                out[f"{name}.state"] = state.index_select(0, rows)
    arrays = {k: v.float().cpu().numpy() for k, v in out.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a.astype(np.float32, copy=False))


def _peer_roofline(pipe, kern, ring, B, world, iters, step_ms):
    """N>1: the requester-side gather reads (W-1)/W of its rows over NVLink — algorithmic NVLink bytes per launch over
    the CUDA-event time of standalone launches, against 900 GB/s per direction; and the same rows against HBM."""
    from torcheasyrec_b200.distributed import ShardedEmbeddingBagCollection

    sm = next((m for m in pipe.sharded if isinstance(m, ShardedEmbeddingBagCollection)), None)
    states = getattr(sm, "_peer_states", None) if sm is not None else None
    if not states:
        return None
    st = max(states, key=lambda s: s.g.total_dim)
    g = st.g
    dg = sorted(ring[0].sparse_features)[0]
    kjts = [g.local._select(b.sparse_features[dg]) for b in ring]
    offs = [kern.lengths_to_offsets(k.lengths()) for k in kjts]
    ids = [k.values() for k in kjts]
    R = len(ring)
    ms = time_kernel(lambda i: st.gather(ids[i % R], offs[i % R]), iters)
    lay = g.local.layout
    row_bytes = float(sum(kjts[0].length_per_key()[f] * lay.dim[f] * 4 for f in range(lay.num_features)))
    nvl = row_bytes * (world - 1) / world
    peak, peak_src = measured_peak_gbs()
    ach = nvl / (ms * 1e-3) / 1e9
    return {"bound": "nvlink", "kernel": "peer_pooled_gather_fwd_kernel (requester-side gather over peer memory)",
            "achieved": ach, "peak": NVLINK_GBS, "unit": "GB/s", "frac": ach / NVLINK_GBS, "traffic": None,
            "peak_source": "nominal NVLink 5 per direction per GPU (B200_PROFILING.md)",
            "ms": ms, "nvlink_bytes_per_launch": nvl, "row_bytes_per_launch": row_bytes,
            "share_of_step": ms / step_ms,
            "note": "algorithmic inbound NVLink bytes = embedding-row bytes x (W-1)/W (uniform ids; 64-B reads); "
                    "timed on rank 0 alone after the run (idle peers), CUDA events"}


def _e2e_blocking(step, host, K, batch):
    """The e2e feed with a BLOCKING loss read (`loss.item()`) between steps — the host cannot enqueue step i+1 before
    step i has finished.  Kept as a measurement-only comparison for the reported (pipelined-read) e2e."""
    for i in range(2):
        step.load(host[i % len(host)])
        step.replay()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    step.prefetch(host[0])
    last = 0.0
    for i in range(K):
        step.commit()
        step.prefetch(host[(i + 1) % len(host)])
        last = float(step.replay().item())
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    return {"value": batch * K / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / K, "last_loss": last,
            "note": "same H2D feed, loss.item() after every step (host and device serialised)"}


def _emit(args, world, B, K, W, ms_total, ms_e2e, host, last, launches_per_step, clk, roofline, cpu, ring_len):
    global_batch = B * world
    h2d = host[0].nbytes()
    sharded = world > 1 or args.force_sharded
    mode = getattr(args, "_mode", "graph")
    shard_txt = {"row_wise": "row-wise", "table_wise": "table-wise", "mixed": f"mixed (row-wise from {args.rw_min_rows} rows)"}
    if not sharded:
        exch = "none"
    elif args.exchange == "peer":
        exch = (f"peer-memory kernels over NVLink (requester-side gather, owner-side pull of keys + in-place gradient "
                f"reads, 4 flag barriers, dense gradients summed from peer buffers): no collective call in the step; "
                f"wire capacity {args.static_capacity}x")
    else:
        exch = (f"static capacity {args.static_capacity}x, in-graph NCCL all-to-all" if mode == "graph"
                else "dynamic splits (host read per step), NCCL all-to-all")
    line = {
        "metric": METRIC if args.model == "dlrm_criteo" else METRIC.replace("DLRM-Criteo", args.model),
        "value": global_batch * K / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model}: examples/{args.model}.config, "
                               f"{'full hash sizes' if not args.max_rows else f'tables capped at {args.max_rows} rows'}, "
                               f"{shard_txt[args.sharding] + ' over ' + str(world) + ' rank(s)' if sharded else 'one GPU'}, "
                               f"per-rank batch {B}, sparse Adagrad lr=1e-3 fused in backward + dense Adam, "
                               f"ids {args.id_dist}",
                   "global_batch": global_batch,
                   "parallelism": (f"{ {'row_wise': 'rw', 'table_wise': 'tw', 'mixed': 'tw+rw'}[args.sharding] }{world}+dp{world}"
                                   if sharded else "1 gpu"),
                   "l2": f"inputs rotate over {ring_len} distinct batches; tables + optimizer state >> 126 MB L2",
                   "cuda_graph": bool(mode == "graph"),
                   "exchange": exch},
        "e2e": {"value": global_batch * K / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K, "last_loss": last,
                "note": "pinned host batch -> H2D (copy stream) -> step -> loss D2H into pinned memory, every step, all "
                        "inside the timed region; the host reads step i-1's loss while step i runs"},
        "zipf_ids": (None if getattr(args, "_zipf_ms", None) is None else
                     {"value": global_batch * K / (args._zipf_ms * 1e-3), "unit": UNIT,
                      "ms_per_step": args._zipf_ms / K, "note": "same step, ids ~ Zipf(1.05) clipped to each table"}),
        "gpu_launches": launches_per_step * K,
        "gpu_launches_per_step": launches_per_step,
        "clocks": clk,
        "roofline": roofline,
        "cpu_baseline": cpu,
    }
    if getattr(args, "_verify", None) is not None:
        line["verify"] = args._verify["status"].lower() if args._verify["status"] == "ok" else "FAILED"
        line["verify_detail"] = args._verify
    if getattr(args, "_extras", None):
        line["extras"] = args._extras
    _print_line(line)


def _small_host() -> bool:
    try:
        import psutil

        return psutil.virtual_memory().available < 40 * 2 ** 30
    except Exception:
        return True


_REAL_STDOUT = None


def _quiet_stdout():
    """Everything that libraries print to fd 1 while the benchmark runs (NCCL's version banner, cuBLAS notices) goes
    to stderr; the ONE JSON line is written to the real stdout by _print_line()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _print_line(line: dict) -> None:
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    _quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    if torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
