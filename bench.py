#!/usr/bin/env python
"""bench.py -- DIFFormer propagation-layer throughput on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (headline workload)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path (oracle/_ref, else the oracle port)
  python bench.py --workload {sigmoid_cora,layer,segmented,fwdbwd}   # the other SURVEY 8 rows, one JSON line each (1 GPU)
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also write what the last timed step computed, DIR/out.npy

Headline workload ("simple")
  step      = one `full_attention_conv(q, k, v, 'simple')` forward (pass 1 reduce -> [all-reduce] -> pass 2 apply) over
              one batch of synthetic [N,H,D] fp32 node tensors.
  config A  = BASELINE configs[2]: N=132 534 (ogbn-proteins shape), H=4, D=64, fp32.  With G>1 ranks every rank holds
              132 534 rows of a G*132 534-node graph (WEAK scaling); the pass-1 partials (67.6 KB) are all-reduced inside
              the pass-1 kernel tail over peer-mapped NVLink memory (or by NCCL, --collective nccl).
  value     = node-updates/s with Q,K,V resident in HBM (inputs + output 543 MB > 126 MB L2; `cold` = same with an L2
              flush between steps); e2e = same through the public Python API with pinned HOST tensors (H2D of Q,K,V and
              D2H of the output inside the timed region).
  parity    = on the exact bench inputs, EVERY rank: out, S, z, u, |Q|, |K|, q^S^, q^z^ against the fp64 oracle of the
              GLOBAL problem (max over ranks); the run fails when any exceeds 1e-3.
  cfg_b     = BASELINE configs[3]: N=1 632 803 (pokec shape) rows sharded over the G ranks (STRONG scaling), same
              kernels, own parity; reported as an extra object in the same JSON line.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import time

sys.dont_write_bytecode = True      # the tree may be read-only, and a run leaves nothing in it
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_NODES, HEADS, DIM = 132534, 4, 64
N_CFG_B = 1632803
METRIC = "DIFFormer-layer node-updates/sec (full_attention_conv 'simple', N=132534 H=4 D=64 fp32 per GPU)"
UNIT = "node-updates/s"
TOL = 1e-3


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1466.2)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md 6.65 TB/s, 1.4 PFLOP/s sustained)"


class ClockSampler:
    """Samples SM clock + clock-event reasons with an `nvidia-smi -lms 20` side process while the
    timed region runs (a Python thread starves behind the launch loop's GIL)."""

    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        import subprocess
        self.proc, self.t0, self.t1 = None, None, None
        try:
            ident = str(dev.index if dev.index is not None else 0)
            try:
                ident = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
            except Exception:
                pass
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ident, f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.proc.stdout.readline()          # first sample: the tool is up
        except Exception:
            self.proc = None

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def summary(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            text, _ = self.proc.communicate(timeout=5)
        except Exception:
            return out
        clocks, reasons, mx = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in text.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if self.t0 is not None and not (self.t0 - 0.02 <= ts <= self.t1 + 0.02):
                    continue
                clocks.append(int(float(f[1])))
                mx = int(float(f[2]))
                for nm, val in zip(names, f[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        clocks.sort()
        out.update({"sm_mhz": clocks[len(clocks) // 2] if clocks else None, "sm_max_mhz": mx, "samples": len(clocks),
                    "reasons": sorted(reasons)})
        return out


def bind_to_gpu_numa_node(dev):
    """Multi-GPU e2e: pin this rank's threads (and with them its pinned host buffers: first touch) to the CPUs of the NUMA node its
    GPU hangs off, so that 8 ranks do not push their H2D / D2H traffic through one socket's memory and the inter-socket link."""
    try:
        props = torch.cuda.get_device_properties(dev)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        cpus = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
            return f"cpus {cpus} (NUMA node {open(f'/sys/bus/pci/devices/{bdf}/numa_node').read().strip()})"
    except Exception as exc:  # noqa: BLE001
        return f"not bound ({type(exc).__name__})"
    return "not bound"


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own full_attention_conv on the host cores (oracle/_ref, vendored
# unmodified by oracle/build_ref.py), else the oracle's op-for-op port of it
# ------------------------------------------------------------------------------------------------
def cpu_reference_fn():
    from oracle import difformer_oracle as O
    try:
        from oracle.ref_shim import load_reference_v1, reference_available
        if reference_available():
            ref = load_reference_v1()
            return (lambda q, k, v: ref.full_attention_conv(q, k, v, "simple")), "reference", \
                "the reference's own full_attention_conv (node classification/difformer.py:10-61, unmodified copy under oracle/_ref)"
    except Exception:
        pass
    return O.simple_attention_reference_chain, "port", "oracle transcription of the einsum chain difformer.py:18-39"


def cpu_reference_rate(steps, warmup, budget_s, rows=None, threads=None):
    from oracle import difformer_oracle as O
    fn, kind, what = cpu_reference_fn()
    ncpu = os.cpu_count() or 1
    q, k, v = O.synthetic_qkv(N_NODES, HEADS, DIM, seed=123)
    with torch.no_grad():
        if threads is None:
            # MKL/OpenMP do not always scale to every hardware thread: give the reference its best thread count
            cands = sorted({c for c in (ncpu, 64, 32, 16, 8) if c <= ncpu}, reverse=True)
            best = (None, float("inf"))
            for c in cands:
                torch.set_num_threads(c)
                fn(q[:32768], k[:32768], v[:32768])
                t0 = time.perf_counter()
                fn(q[:32768], k[:32768], v[:32768])
                dt = time.perf_counter() - t0
                if dt < best[1]:
                    best = (c, dt)
            threads = best[0]
        torch.set_num_threads(threads)
        if rows is None:
            t0 = time.perf_counter()
            fn(q, k, v)
            t_full = time.perf_counter() - t0
            frac = min(1.0, budget_s / max(t_full * (steps + warmup), 1e-9))
            rows = max(4096, int(N_NODES * frac))
        rows = min(rows, N_NODES)
        qs, ks, vs = q[:rows].contiguous(), k[:rows].contiguous(), v[:rows].contiguous()
        for _ in range(warmup):
            fn(qs, ks, vs)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn(qs, ks, vs)
        dt = (time.perf_counter() - t0) / steps
    torch.set_num_threads(ncpu)
    return rows / dt, dt, rows, threads, kind, what


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    rate, dt, rows, threads, kind, what = cpu_reference_rate(args.steps, args.warmup, budget_s=120.0)
    sample = f"{rows} of {N_NODES} rows per step (cost is linear in rows), H={HEADS} D={DIM} fp32, {what}, torch CPU, {threads} threads"
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(max(args.gpus, 1)),
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(world):
    """Identical for both arms (the driver compares the dicts)."""
    return {"workload": f"full_attention_conv('simple') N={N_NODES} H={HEADS} D={DIM} fp32 per GPU (BASELINE configs[2])",
            "rows_per_gpu": N_NODES, "global_rows": N_NODES * world}


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
class Problem:
    """One row-sharded 'simple' problem: this rank's rows of Q, K, V on the device + the step through the C ABI."""

    def __init__(self, rows, n_total, seed, dev, group, comm, collective):
        from difformer_b200 import ops
        from oracle import difformer_oracle as O
        self.ops, self.O = ops, O
        self.rows, self.n_total, self.dev, self.group, self.comm, self.collective = rows, float(n_total), dev, group, comm, collective
        gen = torch.Generator(device=dev).manual_seed(seed)
        # SURVEY 8d: Q, K, V ~ N(0,1) fp32, generated on the device (seeded per rank)
        self.q, self.k, self.v = (torch.randn(rows, HEADS, DIM, generator=gen, device=dev, dtype=torch.float32) for _ in range(3))
        self.plen = int(ops.lib.dif_simple_partials_len(HEADS, HEADS, DIM, DIM))
        self.T = rows * HEADS * DIM * 4

    def reduce(self):
        """pass 1 (+ all-reduce) -> (reduced partials, prepared operand image or None)"""
        ops = self.ops
        if self.comm is not None:          # pass 1 + all-reduce over peer-mapped NVLink memory in ONE kernel
            ex = self.comm.exchange(self.plen, self.dev)
            fused = ex.fused_reduce(self.q, self.k, self.v)
            if fused is not None:
                return fused
            return ex.allreduce(ops.simple_partials(self.q, self.k, self.v)), None
        partials, prepared = ops.simple_partials(self.q, self.k, self.v, with_prepared=True)
        if self.group is not None:
            import torch.distributed as dist
            dist.all_reduce(partials, group=self.group)
            prepared = None       # the pass-2 operand image only matches the un-reduced partials
        return partials, prepared

    one_kernel = True      # dif_simple_forward: pass 1 + (all-)reduce + pass 2 in one cooperative launch (--path twopass: off)

    def step(self):
        if self.one_kernel and (self.group is None or self.comm is not None):
            ex = self.comm.exchange(self.plen, self.dev) if self.comm is not None else None
            res = self.ops.simple_forward(self.q, self.k, self.v, self.n_total, ex)
            if res is not None:
                return res[0]
        partials, prepared = self.reduce()
        return self.ops.simple_apply(self.q, partials, self.n_total, HEADS, DIM, prepared=prepared)

    def parity(self, oracle_device):
        """out and the BASELINE.md 4.4 intermediates of THIS rank against the fp64 oracle of the GLOBAL problem."""
        import torch.distributed as dist
        O, ops = self.O, self.ops
        H, D = HEADS, DIM
        qd, kd, vd = (t.to(oracle_device, torch.float64) for t in (self.q, self.k, self.v))
        wp = O.simple_partials(qd, kd, vd)
        flat = torch.cat([wp["S"].reshape(-1), wp["z"].reshape(-1), wp["u"].reshape(-1), wp["sq"].reshape(1), wp["sk"].reshape(1)])
        if self.group is not None:           # oracle partials are additive over the row shards too
            flat = flat.to(self.dev)
            dist.all_reduce(flat, group=self.group)
            flat = flat.to(oracle_device)
        nS, nz = H * D * D, H * D
        want = {"S": flat[:nS].reshape(H, D, D), "z": flat[nS:nS + nz].reshape(H, D), "u": flat[nS + nz:nS + 2 * nz].reshape(H, D),
                "sq": flat[-2], "sk": flat[-1], "n": torch.tensor(self.n_total, dtype=torch.float64)}
        want_out, parts = O.simple_apply(qd, want, self.n_total, return_parts=True)
        got_out = self.step()
        got = self.reduce()[0].double().to(oracle_device)
        err = {"out": O.rel_err(got_out, want_out),
               "S": O.rel_err(got[:nS].reshape(H, D, D), want["S"]), "z": O.rel_err(got[nS:nS + nz].reshape(H, D), want["z"]),
               "u": O.rel_err(got[nS + nz:nS + 2 * nz].reshape(H, D), want["u"]),
               "normQ": abs(float(got[-2].sqrt() / want["sq"].sqrt()) - 1.0), "normK": abs(float(got[-1].sqrt() / want["sk"].sqrt()) - 1.0)}
        # q^S^ and q^z^ through pass 2 itself with edited partials and a small n_total (at n_total = N the fp32 denominator
        # q^z^ + N swallows q^z^ -- in the reference too):  u := 0, z := 0, n := 1 -> out = q^S^ ;  S := 0, u := 1 -> out = 1/(q^z^ + n)
        red = self.reduce()[0]
        only_s = red.clone()
        only_s[nS:nS + 2 * nz] = 0
        err["qS"] = O.rel_err(ops.simple_apply(self.q, only_s, 1.0, H, D), parts["qS"])
        only_z = red.clone()
        only_z[:nS] = 0
        only_z[nS + nz:nS + 2 * nz] = 1
        nz_ = 2.0 ** -13                      # comparable to |q^z^| (~1e-4 for N(0,1) inputs): no cancellation in 1/out - n
        qz = 1.0 / ops.simple_apply(self.q, only_z, nz_, H, D).double() - nz_
        err["qz"] = O.rel_err(qz[..., 0], parts["qz"])
        t = torch.tensor([err[k_] for k_ in sorted(err)], dtype=torch.float64, device=self.dev)
        if self.group is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        out = {k_: float(x) for k_, x in zip(sorted(err), t.tolist())}
        out["max"] = max(out.values())
        out["ok"] = bool(out["max"] < TOL)
        out["what"] = "max over ranks of the rel. error vs the fp64 oracle of the global problem; tolerance 1e-3"
        return out


def timed(fn, steps, barrier, dev, group):
    """-> (ms per step, what the last of the `steps` timed calls of fn returned)"""
    import torch.distributed as dist
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    ev[0].record()
    for _ in range(steps - 1):
        fn()
    last = fn()
    ev[1].record()
    barrier()
    t = torch.tensor([ev[0].elapsed_time(ev[1]) / steps], dtype=torch.float64, device=dev)
    if group is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item()), last


DUMP_ROWS = 32768       # rows of the [N, H, D] output --dump-outputs keeps (32 MiB in fp32)


def dump_outputs(out_dir, out):
    """Writes out_dir/out.npy: a fixed sample (DUMP_ROWS rows drawn once with seed 0, in ascending order) of `out`, the [N, H, D]
    result of the last timed step, in float32.  The same arguments give the same inputs, so two builds compare output for output."""
    import numpy as np
    rows = torch.randperm(out.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "out.npy"), out.index_select(0, rows.to(out.device)).float().cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    group = None
    numa = bind_to_gpu_numa_node(dev) if world > 1 else "single GPU: not bound"
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        group = dist.group.WORLD

    from difformer_b200 import ops
    from difformer_b200.sharded import shard_rows
    from oracle import difformer_oracle as O
    if args.simple_impl:
        ops.set_simple_impl(args.simple_impl)

    Problem.one_kernel = args.path == "fused"
    ops.set_fused_forward(args.path == "fused")
    comm, collective = None, args.collective if world > 1 else None
    if group is not None and args.collective == "nvlink":
        from difformer_b200.sharded import RowShardComm
        comm = RowShardComm(group)

    def barrier():
        if group is not None:
            dist.barrier(group=group)
        torch.cuda.synchronize(dev)

    prob = Problem(N_NODES, N_NODES * world, 123 + rank, dev, group, comm, collective)
    T = prob.T

    # ---- parity on the exact bench inputs, every rank (fp64 oracle on the host cores)
    parity = prob.parity(torch.device("cpu"))

    for _ in range(max(args.warmup, 3) + 20):      # W warm-up steps plus 20 more: clocks and caches settle before the timed K steps
        prob.step()
    barrier()
    if comm is not None:
        # watchdog (common.cuh): a rank whose kernel gave up waiting for a peer reports it here; then every rank switches
        # to the NCCL all-reduce of the partials so that the run still produces a valid number
        bad = torch.tensor([1.0 if comm.exchange(prob.plen, dev).timed_out() else 0.0], dtype=torch.float32, device=dev)
        dist.all_reduce(bad, op=dist.ReduceOp.MAX, group=group)
        if float(bad.item()) > 0:
            comm, collective = None, "nccl"
            prob.comm = None
            if rank == 0:
                print("bench: the NVLink exchange timed out waiting for a peer; falling back to NCCL", file=sys.stderr)
            for _ in range(3):
                prob.step()
            barrier()
    sampler = ClockSampler(dev)
    barrier()
    sampler.begin()
    ms, out = timed(prob.step, args.steps, barrier, dev, group)
    sampler.end()
    value = N_NODES * world / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    del out

    # ---- cold-cache number (SURVEY 8d): L2 flushed (256 MB written) before every step, each step timed on its own
    cold_ms = None
    if world == 1:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        pairs = []
        for _ in range(min(args.steps, 20)):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            prob.step()
            e1.record()
            pairs.append((e0, e1))
        torch.cuda.synchronize(dev)
        ts = sorted(a.elapsed_time(b) for a, b in pairs)
        cold_ms = ts[len(ts) // 2]
        del flush

    # ---- end to end through the public API with pinned host buffers
    import difformer
    q, k, v = prob.q, prob.k, prob.v
    qh, kh, vh = (x.cpu().pin_memory() for x in (q, k, v))
    oh = torch.empty((N_NODES, HEADS, DIM), dtype=torch.float32).pin_memory()
    rs = None
    if group is not None:
        from difformer_b200.sharded import RowShardedAttention
        rs = RowShardedAttention(N_NODES * world, group, nvlink=(collective == "nvlink"))

    # Double-buffered, three streams: the upload of step i+1 (copy engine, H2D) overlaps the kernels of step i and the
    # download of step i-1 (second copy engine, D2H).  Every step still uploads its own Q, K, V from pinned host
    # memory and downloads its own result; PCIe is full duplex, so the steady state is bound by the larger of the two.
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    dbuf = [tuple(torch.empty_like(x) for x in (q, k, v)) for _ in range(2)]
    ohs = [oh, torch.empty_like(oh).pin_memory()]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_cmp = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    live = [None, None]                       # keeps a step's device result alive until its download has been queued twice over

    def e2e_step(i):
        b = i & 1
        cur = torch.cuda.current_stream(dev)
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_cmp[b])        # the kernels of step i-2 have finished reading this input buffer
            for dst, src in zip(dbuf[b], (qh, kh, vh)):
                dst.copy_(src, non_blocking=True)
            ev_in[b].record(s_in)
        cur.wait_event(ev_in[b])
        with torch.no_grad():
            o = rs(*dbuf[b]) if rs is not None else difformer.full_attention_conv(*dbuf[b], "simple")
        ev_cmp[b].record(cur)
        o.record_stream(s_out)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_cmp[b])
            ohs[b].copy_(o, non_blocking=True)
            ev_out[b].record(s_out)
        live[b] = o

    def e2e_drain():
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(ev_out[0])
        cur.wait_event(ev_out[1])

    e2e_steps = max(3, min(args.steps, 20))
    for i in range(4):
        e2e_step(i)
    e2e_drain()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(e2e_steps):
        e2e_step(i)
    e2e_drain()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1) / e2e_steps
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if group is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    e2e_ms = float(t.item())
    e2e_out_err = O.rel_err(ohs[(e2e_steps - 1) & 1], prob.step())      # the downloaded result is the kernels' result
    del dbuf, ohs, qh, kh, vh, live

    # ---- BASELINE configs[3]: N = 1 632 803 rows sharded over the ranks (strong scaling), own parity (fp64 oracle on the GPU)
    cfg_b = None
    if not args.no_cfg_b:
        b0, b1 = shard_rows(N_CFG_B, rank, world)
        pb = Problem(b1 - b0, N_CFG_B, 1000 + rank, dev, group, prob.comm, collective)
        par_b = pb.parity(dev)
        for _ in range(3):
            pb.step()
        ms_b, _ = timed(pb.step, max(5, min(args.steps, 20)), barrier, dev, group)
        cfg_b = {"workload": f"full_attention_conv('simple') N={N_CFG_B} H={HEADS} D={DIM} fp32 row-sharded over {world} GPU(s) (BASELINE configs[3])",
                 "scaling": "strong", "rows_this_rank": b1 - b0, "ms_per_step": ms_b, "value": N_CFG_B / (ms_b * 1e-3), "unit": UNIT,
                 "roofline_frac": 4 * N_CFG_B * HEADS * DIM * 4 / (ms_b * 1e-3) / 1e9 / (measured_peaks()[0] * world), "parity": par_b}
        del pb

    launches_per_step = 3 if args.simple_impl == "generic" else (1 if (args.path == "fused" and (world == 1 or collective == "nvlink")) else 2)
    if world > 1 and collective == "nccl":
        launches_per_step += 1
    # ---- 16-bit I/O (bf16): same workload, half the algorithmic bytes (2048 B/node), own parity (1 GPU)
    lp16 = None
    if world == 1 and not args.no_lp16:
        qb, kb, vb = (t.to(torch.bfloat16) for t in (q, k, v))
        res = ops.simple_forward(qb, kb, vb)
        if res is not None:
            ob, pb_ = res
            wp = O.simple_partials(qb.double(), kb.double(), vb.double())          # fp64 oracle on the rounded inputs, on the GPU
            want = O.simple_apply(qb.double(), wp)
            nS, nz = HEADS * DIM * DIM, HEADS * DIM
            par = {"S": O.rel_err(pb_[:nS].reshape(HEADS, DIM, DIM), wp["S"]), "z": O.rel_err(pb_[nS:nS + nz].reshape(HEADS, DIM), wp["z"]),
                   "u": O.rel_err(pb_[nS + nz:nS + 2 * nz].reshape(HEADS, DIM), wp["u"]),
                   "normQ": abs(float(pb_[-2].double().sqrt() / wp["sq"].sqrt()) - 1.0), "normK": abs(float(pb_[-1].double().sqrt() / wp["sk"].sqrt()) - 1.0),
                   "out_vs_oracle_rounded_to_bf16": O.rel_err(ob.double(), want.to(torch.bfloat16).double()), "out": O.rel_err(ob.double(), want)}
            par["ok"] = bool(max(par["S"], par["z"], par["u"], par["normQ"], par["normK"]) < TOL and par["out"] < 2.0 ** -8)
            del wp, want
            for _ in range(5):
                ops.simple_forward(qb, kb, vb)
            ms16, _ = timed(lambda: ops.simple_forward(qb, kb, vb), args.steps, barrier, dev, None)
            lp16 = {"dtype": "bf16", "ms_per_step": ms16, "value": N_NODES / (ms16 * 1e-3), "unit": UNIT,
                    "roofline": {"bound": "hbm", "achieved": 2 * T / (ms16 * 1e-3) / 1e9, "peak": measured_peaks()[0], "unit": "GB/s",
                                 "frac": 2 * T / (ms16 * 1e-3) / 1e9 / measured_peaks()[0], "algorithmic_bytes_per_step": 2 * T},
                    "parity": par, "what": "same workload with bf16 node tensors in and out (simple_lp_kernel): TMA -> tcgen05 without a conversion pass"}
            del qb, kb, vb, ob

    if rank == 0:
        peak, _, peak_src = measured_peaks()
        alg_bytes = 4 * T                      # read Q,K,V once + write out once (SURVEY.md 8d)
        achieved = alg_bytes / (ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src,
                "kernel": ("simple_fused_kernel: pass 1 + grid-wide [+ cross-GPU] sum + pass 2 in ONE cooperative launch per step" if launches_per_step == 1 else
                           "simple op = pass 1 (reduce, cross-CTA [+cross-GPU] sum fused) + pass 2 (apply): one launch sequence per step"),
                "algorithmic_bytes_per_step": alg_bytes}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.isfile(tp):
            try:
                tj = json.load(open(tp))
                roof["traffic"] = tj.get("simple_step_dram_bytes")
                roof["traffic_source"] = "ncu --set full capture committed under profiles/ (not re-measured in this run): " + str(tj.get("source", ""))[:160]
            except Exception:
                pass
        if cold_ms is not None:
            roof["cold"] = {"ms_per_step": cold_ms, "frac": alg_bytes / (cold_ms * 1e-3) / 1e9 / peak,
                            "what": "median of per-step CUDA-event times with the L2 flushed (256 MB memset) before every step"}
        torch_gpu = None
        if world == 1:
            # the reference's own op chain (einsums + materialised broadcasts) on the same B200, CUDA tensors
            fn, kind, what = cpu_reference_fn()
            with torch.no_grad():
                for _ in range(5):
                    fn(q, k, v)
                torch.cuda.synchronize(dev)
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                for _ in range(20):
                    fn(q, k, v)
                g1.record()
                torch.cuda.synchronize(dev)
            tg = g0.elapsed_time(g1) / 20
            torch_gpu = {"value": N_NODES / (tg * 1e-3), "unit": UNIT, "ms_per_step": tg, "kind": kind,
                         "what": f"{what} in PyTorch eager on the same GPU"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            rate, dt, rows, threads, kind, what = cpu_reference_rate(steps=8, warmup=2, budget_s=20.0)
            r1, dt1, rows1, _, _, _ = cpu_reference_rate(steps=3, warmup=1, budget_s=5.0, rows=16384, threads=1)
            cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": kind,
                   "sample": f"{rows} of {N_NODES} rows x 8 steps, {what}, torch CPU fp32 (host has {os.cpu_count()} hardware threads)",
                   "one_thread": {"value": r1, "unit": UNIT, "cores": 1, "sample": f"{rows1} rows x 3 steps"}}
        cfg = workload_config(world)      # identical in both arms; everything specific to this arm goes to `notes`
        notes = {"parallelism": "single GPU" if world == 1 else (
                     f"row-shard x{world}, one all-reduce of 16898 fp32 per step: " +
                     ("fused into the pass-1 kernel tail, LL push over peer-mapped NVLink memory (no NCCL call)" if collective == "nvlink" else "NCCL")),
                 "l2": "inputs 407 MB + output 136 MB per step exceed the 126 MB L2; no flush between steps (roofline.cold: flushed)",
                 "simple_impl": args.simple_impl or "auto", "path": args.path, "host_numa_binding_rank0": numa}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": cfg, "notes": notes,
                "roofline": roof, "cpu_baseline": cpu, "torch_gpu_baseline": torch_gpu,
                "e2e": {"value": N_NODES * world / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": 3 * T, "d2h_bytes_per_step": T, "steps": e2e_steps, "result_rel_err_vs_device_run": e2e_out_err,
                        "api": "difformer.full_attention_conv(q, k, v, 'simple') on pinned host tensors; double-buffered (upload of step i+1 overlaps download of step i-1)"},
                "gpu_launches": launches_per_step * args.steps,
                "clocks": sampler.summary(), "parity": parity, "cfg_b": cfg_b, "lp16": lp16}
        print(json.dumps(line), flush=True)
    ok = parity["ok"] and (cfg_b is None or cfg_b["parity"]["ok"]) and (lp16 is None or lp16["parity"]["ok"])
    if group is not None:
        dist.destroy_process_group()
    if not ok:
        raise SystemExit("bench.py: PARITY FAILURE (see the `parity` objects of the JSON line): the timing above is void")


# ------------------------------------------------------------------------------------------------
# the other SURVEY 8 rows (1 GPU), one JSON line each
# ------------------------------------------------------------------------------------------------
def run_extra(args):
    import difformer
    from difformer_b200 import ops
    from oracle import difformer_oracle as O
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    hbm, tens, src = measured_peaks()

    def timeit(fn, iters):
        for _ in range(max(args.warmup, 3)):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    steps = min(args.steps, 200)
    w = args.workload
    line = {"workload": w, "n_gpus": 1, "steps": steps, "data": "synthetic", "peak_source": src}
    if w == "sigmoid_cora":          # BASELINE configs[1]: Cora shape
        n, h, d = 2708, 1, 64
        q, k, v = (t.to(dev) for t in O.synthetic_qkv(n, h, d, seed=1))
        q, k = q * 0.3, k * 0.3
        ms = timeit(lambda: difformer.full_attention_conv(q, k, v, "sigmoid"), steps)
        qg, kg, vg = (t.clone().requires_grad_(True) for t in (q, k, v))

        def fb():
            o = difformer.full_attention_conv(qg, kg, vg, "sigmoid")
            o.backward(torch.ones_like(o))
        ms_fb = timeit(fb, steps)
        out = difformer.full_attention_conv(q, k, v, "sigmoid")
        want = O.sigmoid_attention(q.double().cpu(), k.double().cpu(), v.double().cpu())
        flops = 4.0 * n * n * h * d
        line.update({"metric": "node-updates/s, full_attention_conv('sigmoid') N=2708 H=1 D=64 fp32 (Cora shape)", "value": n / (ms * 1e-3),
                     "unit": UNIT, "ms_per_step": ms, "fwd_bwd_ms": ms_fb, "dtype": "f32 (bf16x3 split on the tensor cores)",
                     "roofline": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": tens, "unit": "TFLOP/s",
                                  "frac": flops / (ms * 1e-3) / 1e12 / tens, "flops": flops},
                     "parity": {"out": O.rel_err(out, want)}})
    elif w == "layer":               # a-4/a-5: attention + gcn + head mean + residual, no grad, config A with E = 17 N
        n, h, d = N_NODES, HEADS, DIM
        q, k, v = (t.to(dev) for t in O.synthetic_qkv(n, h, d, seed=3))
        ei = O.synthetic_graph(n, 8 * n, seed=4).to(dev)
        E = ei.shape[1]
        csr = ops.graph_csr(ei, None, n)
        prev = torch.randn(n, d, device=dev)

        def layer():
            vb_ = torch.empty((n, d), dtype=torch.float32, device=dev)
            part, prep = ops.simple_partials(q, k, v, with_prepared=True, vbar=vb_)
            if args.layer_gcn == "epilogue":     # the gcn term gathered by the pass-2 epilogue itself: never written to HBM (measured slower)
                ep = ops.make_epilogue(0.5 / h, [(prev, 0.5)], gcn=(csr, vb_, 0.5))
            else:                                # SpMM on mean_h V (L2-resident), its [N,D] result is an addend of the epilogue
                g = ops.spmm(csr, vb_.view(n, 1, d)).view(n, d)
                ep = ops.make_epilogue(0.5 / h, [(g, 0.5), (prev, 0.5)])
            return ops.simple_apply(q, part, float(n), h, d, ep, prepared=prep)
        ms = timeit(layer, steps)
        alg = n * (3 * h * d * 4 + 2 * d * 4) + E * 8 + (n + 1) * 4
        attn = O.simple_attention(q.double().cpu(), k.double().cpu(), v.double().cpu())
        gcn = O.gcn_conv(v.double().cpu(), ei.cpu(), None)
        want = 0.5 * (attn + gcn).mean(1) + 0.5 * prev.double().cpu()      # alpha = 0.5, graph_weight < 0 (difformer.py:137-140, 200-201)
        line.update({"metric": f"node-updates/s, fused propagation layer (attention + gcn E={E} + head mean + residual) N={n} H=4 D=64 fp32",
                     "value": n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "dtype": "f32",
                     "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                  "frac": alg / (ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes_per_step": alg},
                     "parity": {"out": O.rel_err(layer(), want)}})
    elif w == "layer_x":             # f-1: one whole DIFFormerConv layer from its input x [N, 64] (Linears included), no grad, config A, E = 17 N
        from difformer_b200 import module as M_
        n, h, d = N_NODES, HEADS, DIM
        torch.manual_seed(11)
        conv = difformer.DIFFormerConv(d, d, num_heads=h, kernel="simple", use_graph=True, use_weight=True).to(dev)
        ln = torch.nn.LayerNorm(d).to(dev)
        x = torch.randn(n, d, device=dev)
        prev = torch.randn(n, d, device=dev)
        ei = O.synthetic_graph(n, 8 * n, seed=4).to(dev)
        E = ei.shape[1]
        ops.graph_csr(ei, None, n)

        def layer():
            with torch.no_grad():
                return M_._conv_forward(conv, x, x, ei, None, x, False, residual=(0.5, prev), layer_norm=ln)[0]
        res, host = {}, {}
        for fold in (False, True):
            ops.set_projection_folding(fold)
            res[fold] = timeit(layer, steps)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                layer()
            host[fold] = (time.perf_counter() - t0) / steps * 1e3        # enqueue cost of one layer (no sync): the floor the GPU time must stay above
            torch.cuda.synchronize()
        # the same folded layer as a CUDA graph: what the GPU needs once the host enqueue (several small launches, two streams) is out of the way
        ops.set_projection_folding(True)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            layer()
        torch.cuda.current_stream().wait_stream(side)
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            out_g = layer()
        ms_graph = timeit(cg.replay, steps)
        xd = x.double().cpu()
        qd, kd, vd = (torch.nn.functional.linear(xd, l.weight.double().cpu(), l.bias.double().cpu()).view(n, h, d) for l in (conv.Wq, conv.Wk, conv.Wv))
        body = (O.simple_attention(qd, kd, vd) + O.gcn_conv(vd, ei.cpu(), None)).mean(1)          # difformer.py:137-140
        want = torch.nn.functional.layer_norm(0.5 * body + 0.5 * prev.double().cpu(), (d,), ln.weight.double().cpu(), ln.bias.double().cpu(), ln.eps)
        par = {}
        for fold in (False, True):
            ops.set_projection_folding(fold)
            par["folded" if fold else "unfolded"] = O.rel_err(layer(), want)
        cg.replay()
        par["folded_graphed"] = O.rel_err(out_g, want)
        ms = res[True]
        alg = n * (3 * d * 4) + E * 8 + (n + 1) * 4        # x read (pass 1; pass 2 and the vbar GEMM re-read it from L2), prev, out
        line.update({"metric": f"node-updates/s, DIFFormerConv layer from x (Wq/Wk/Wv + attention + gcn E={E} + head mean + residual + LayerNorm) N={n} H=4 hidden=64 fp32",
                     "value": n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "ms_per_step_graphed": ms_graph, "ms_per_step_unfolded": res[False], "host_enqueue_ms": host[True],
                     "host_enqueue_ms_unfolded": host[False], "dtype": "f32",
                     "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                  "frac": alg / (ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes_per_step": alg},
                     "parity": par})
    elif w == "model":               # the reference's ogbn-proteins model (run.sh:37-39) on the full graph, inference: 3 layers, hidden 64, 1 head
        from difformer_b200 import GraphedForward
        n, cin, cout = N_NODES, 8, 112
        torch.manual_seed(3)
        m = difformer.DIFFormer(cin, 64, cout, num_layers=3, num_heads=1, kernel="simple", use_bn=True, use_residual=True, use_weight=True,
                                use_graph=True).to(dev).eval()
        x = torch.randn(n, cin, device=dev)
        ei = O.synthetic_graph(n, 8 * n, seed=4).to(dev)
        E = ei.shape[1]

        def fwd():
            with torch.no_grad():
                return m(x, ei)
        res = {}
        for fold in (False, True):
            ops.set_projection_folding(fold)
            res[fold] = timeit(fwd, steps)
        out_plain = None
        par = {}
        sd = {k_: v_.double().cpu() for k_, v_ in m.state_dict().items()}
        want = O.difformer_forward(sd, x.double().cpu(), ei.cpu(), None, hidden_channels=64, num_layers=3, num_heads=1, kernel="simple", use_bn=True, use_residual=True,
                                   use_weight=True, use_graph=True)
        for fold in (False, True):
            ops.set_projection_folding(fold)
            par["folded" if fold else "explicit"] = O.rel_err(fwd(), want)
        gf = GraphedForward(m, x, ei)                    # CUDA-graph replay of the folded forward: no host enqueue cost
        ms_graph = timeit(lambda: gf(x, ei), steps)
        par["graphed"] = O.rel_err(gf(x, ei), want)
        ms = res[True]
        line.update({"metric": f"node-updates/s, DIFFormer model forward (ogbn-proteins config: 3 layers, hidden 64, 1 head, bn + residual + gcn E={E}) N={n} fp32, inference",
                     "value": n / (ms_graph * 1e-3), "unit": UNIT, "ms_per_step": ms_graph, "ms_eager_folded": ms, "ms_eager_explicit": res[False],
                     "dtype": "f32", "parity": par})
    elif w == "segmented":           # BASELINE configs[4]: B = 8192 graphs, n_g ~ U[10,40], H = 1, D = 64
        gen = torch.Generator().manual_seed(5)
        nn_ = torch.randint(10, 41, (8192,), generator=gen)
        tot = int(nn_.sum())
        qs, ks, vs = (t.to(dev) for t in O.synthetic_qkv(tot, 1, 64, seed=6))
        nn_d = nn_.to(dev)
        ms = timeit(lambda: ops.segmented_full_attention(qs, ks, vs, "simple", nn_d), steps)
        qsg, ksg, vsg = (t.clone().requires_grad_(True) for t in (qs, ks, vs))
        gs = torch.randn(tot, 1, 64, device=dev)

        def fb3():
            qsg.grad = ksg.grad = vsg.grad = None
            o = ops.segmented_full_attention(qsg, ksg, vsg, "simple", nn_d)
            o.backward(gs)
        ms_fb = timeit(fb3, steps)
        want = O.segmented_simple_attention(qs.double().cpu(), ks.double().cpu(), vs.double().cpu(), nn_)
        alg = 4 * tot * 64 * 4
        line.update({"metric": f"node-updates/s, batched-graph 'simple' (difformer-v2) B=8192 sumN={tot} H=1 D=64 fp32", "value": tot / (ms * 1e-3),
                     "unit": UNIT, "ms_per_step": ms, "fwd_bwd_ms": ms_fb, "dtype": "f32",
                     "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / hbm,
                                  "algorithmic_bytes_per_step": alg},
                     "parity": {"out": O.rel_err(ops.segmented_full_attention(qs, ks, vs, "simple", nn_d), want)}})
    elif w == "fwdbwd":              # a-1 + a-1b at config A through torch.autograd
        n, h, d = N_NODES, HEADS, DIM
        q, k, v = (t.to(dev) for t in O.synthetic_qkv(n, h, d, seed=3))
        qg, kg, vg = (t.clone().requires_grad_(True) for t in (q, k, v))
        go = torch.randn(n, h, d, device=dev)

        def fb2():
            qg.grad = kg.grad = vg.grad = None
            o = difformer.full_attention_conv(qg, kg, vg, "simple")
            o.backward(go)
        ms = timeit(fb2, steps)
        dq, dk, dv = O.simple_attention_backward(q.double().cpu(), k.double().cpu(), v.double().cpu(), go.double().cpu())
        alg = (4 + 11) * n * h * d * 4     # fwd 4T; bwd: pass 1 reads q,g,out (3T), dq/dk/dv read 2T+2T+1T and write 3T
        line.update({"metric": f"node-updates/s, full_attention_conv('simple') forward+backward N={n} H=4 D=64 fp32", "value": n / (ms * 1e-3),
                     "unit": UNIT, "ms_per_step": ms, "dtype": "f32",
                     "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / hbm,
                                  "algorithmic_bytes_per_step": alg},
                     "parity": {"dq": O.rel_err(qg.grad, dq), "dk": O.rel_err(kg.grad, dk), "dv": O.rel_err(vg.grad, dv)}})
    else:
        raise SystemExit(f"unknown workload {w}")
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="simple", choices=["simple", "sigmoid_cora", "layer", "layer_x", "model", "segmented", "fwdbwd"])
    ap.add_argument("--simple-impl", default=None, choices=[None, "auto", "generic", "tcgen05"])
    ap.add_argument("--path", default="fused", choices=["fused", "twopass"], help="'simple' forward: one cooperative kernel, or pass 1 / pass 2 as two launches")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lp16", action="store_true", help="skip the bf16-I/O leg")
    ap.add_argument("--layer-gcn", default="spmm", choices=["spmm", "epilogue"], help="--workload layer: where the gcn term is computed")
    ap.add_argument("--no-cfg-b", action="store_true", help="skip the BASELINE configs[3] (N=1.6M strong-scaling) leg")
    ap.add_argument("--collective", default="nvlink", choices=["nvlink", "nccl"], help="multi-GPU all-reduce of the partials")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help=f"headline workload: after the timed steps write DIR/out.npy, {DUMP_ROWS} fixed rows (seed 0) of the [N, H, D] fp32 "
                         "output of the last timed step (rank 0's rows with several GPUs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "simple"):
        ap.error("--dump-outputs covers the headline workload (--impl ours --workload simple)")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload != "simple":
        run_extra(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
