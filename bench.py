#!/usr/bin/env python
"""bench.py -- consensus windows/s of the B200 window-consensus engine on a synthetic 40x pile.

One "step" = one pass of the hot path (the dcu_* C ABI) over all windows of this rank's shard of A-reads.
  value  : windows/s with windows, slices and the packed read DB already resident in HBM (kernel launches only)
  e2e    : the same through the read-level C ABI with HOST buffers: overlaps + trace points in (what the reference's
           HandleContext::operator() is handed, src/HandleContext.hpp:1699-1715), corrected bases out
           (dcu_pile + dcu_launch + dcu_vote + dcu_get_corrected; H2D and D2H inside the timed region)
  e2e_descriptors : dcu_run with host window / slice descriptors in and result records out (the window-level entry point)
  --impl reference : the CPU oracle (restatement of gt1/daccord; the upstream binary cannot be built here) on all
                     host threads over a bounded sample of the same windows -- window consensus only (no piling, no vote),
                     so the e2e ratio against it is conservative for the GPU side; an upper bound against real daccord
                     all the same (libmaus2's SIMD aligners are not reproduced).
Multi-GPU (torchrun): rank r processes the reads of `-J r,N` (reference src/daccord.cpp:1156-1184); --scaling weak
(default) makes the dataset N times larger, --scaling strong keeps --mb as the total (BASELINE config 3); the packed DB
is broadcast once over NCCL; no collective during compute.  Other BASELINE configs: --k (config 4), --coverage /
--depth-cap / --maxinput / --repeat-frac (config 5 and the shallow tail).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np


def j_shard(nreads, i, j):
    """reference -J i,j arithmetic (src/daccord.cpp:1156-1184)"""
    part = (nreads + j - 1) // j
    lo = min(i * part, nreads)
    return lo, min(lo + part, nreads)


def algorithmic_bytes(win, sl, res):
    """SURVEY 8d: sum over attempted windows of  sum_j ceil(len_j/4) + 8*MAo + 16 + (clen + 16)"""
    att = res["status"] != 0
    sl_bytes = (sl["len"].astype(np.int64) + 3) // 4 + 8
    cs = np.concatenate([[0], np.cumsum(sl_bytes)])
    b = win["slice_begin"].astype(np.int64)
    e = b + win["slice_cnt"].astype(np.int64)
    per = cs[e] - cs[b] + 16 + res["clen"].astype(np.int64) + 16
    return int(per[att].sum()), int(att.sum())


class ClockSampler(threading.Thread):
    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.stop_flag, self.sm, self.reasons, self.smmax = gpu, False, [], set(), None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.sm.append(float(f[0])); self.smmax = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smmax, "reasons": sorted(self.reasons)}


def full_compare(a, b):
    """bit-exact comparison of two (res, cons, ops) triples (what tests/common.compare_results does, vectorised):
    per window True where the result record differs, or -- for windows with a consensus -- the consensus bytes or the placement trace"""
    ra, ca, oa = a[:3]
    rb, cb, ob = b[:3]
    n = len(ra)
    bad = ra != rb
    ok = (ra["status"] == 1) & ~bad
    ca = np.asarray(ca).reshape(n, 64); cb = np.asarray(cb).reshape(n, 64); oa = np.asarray(oa).reshape(n, 128); ob = np.asarray(ob).reshape(n, 128)
    step = 1 << 18
    for i in range(0, n, step):
        j = min(n, i + step)
        mc = np.arange(64)[None, :] < ra["clen"][i:j, None]
        mo = np.arange(128)[None, :] < ra["nops"][i:j, None]
        bad[i:j] |= ok[i:j] & (((ca[i:j] != cb[i:j]) & mc).any(1) | ((oa[i:j] != ob[i:j]) & mo).any(1))
    return bad


DUMP_WINDOWS, DUMP_SEGMENTS, DUMP_BASES = 1 << 15, 1 << 16, 1 << 20      # sample sizes of --dump-outputs: at most about 45 MB of .npy files


def dump_outputs(path, win_out, reads_out):
    """--dump-outputs: what a caller of the timed paths receives, as DIR/<name>.npy in float32 / float64, so that two builds can be compared
    output for output.  win_out = (res, cons, ops) of the last step of the device-resident leg: the result records of a fixed sample of windows,
    with the consensus bytes and placement trace a window has (status 1: the first clen / nops bytes; zeros elsewhere, as those bytes are
    undefined).  reads_out = (seg, chars) of the last e2e step, or None when that leg did not run: the segment records and the corrected bases,
    both sampled when larger than the sample.  Each sample is a seeded function of the array's length alone."""
    rng = np.random.default_rng(20240601)

    def sample(n, k):
        return np.arange(n) if n <= k else np.unique(rng.integers(0, n, k))
    res, cons, ops = win_out
    n = len(res)
    wi = sample(n, DUMP_WINDOWS)
    r = res[wi]
    ok = r["status"] == 1
    c = np.asarray(cons).reshape(n, 64)[wi]
    o = np.asarray(ops).reshape(n, 128)[wi]
    arrays = {"window_index": wi.astype(np.float64),
              "window_consensus": np.where(ok[:, None] & (np.arange(64)[None, :] < r["clen"][:, None]), c, 0).astype(np.float32),
              "window_placement": np.where(ok[:, None] & (np.arange(128)[None, :] < r["nops"][:, None]), o, 0).astype(np.float32)}
    arrays.update(("window_" + f, r[f].astype(np.float64)) for f in res.dtype.names)
    if reads_out is not None:
        seg, chars = reads_out
        si, bi = sample(len(seg), DUMP_SEGMENTS), sample(len(chars), DUMP_BASES)
        arrays["read_segment_index"] = si.astype(np.float64)
        arrays.update(("read_segment_" + f, seg[si][f].astype(np.float64)) for f in seg.dtype.names)
        arrays["read_base_index"] = bi.astype(np.float64)
        arrays["read_bases"] = chars[bi].astype(np.float32)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def effective_cpus():
    """CPUs this process may really use: affinity mask and cgroup quota (os.cpu_count() ignores both)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def best_oracle_threads(run_oracle, p, packed, win, sl):
    """the CPU arm uses whatever thread count is fastest on this box (probed on a small sample)"""
    cand = sorted({max(1, effective_cpus() // 4), max(1, effective_cpus() // 2), effective_cpus(), min(os.cpu_count() or 1, 2 * effective_cpus())})
    best, rate = 1, 0.0
    for t in cand:
        n = min(len(win), 1000 + 300 * t)
        _, _, _, dt = run_oracle(p, packed, win[:n].copy(), sl, t)
        if n / max(dt, 1e-9) > rate:
            best, rate = t, n / max(dt, 1e-9)
    return best


def bind_to_gpu_numa_node(local):
    """keep this rank's host threads and pinned buffers on the NUMA node its GPU hangs off (best effort; returns the node or None)"""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        if bus is None:
            return None
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def maxalign_of(args):
    return args.depth_cap if args.depth_cap > 0 else 2**64 - 1


def build_workload(args, rank, world, keep_truth=False):
    from daccord_b200.host import Dataset
    total_mb = args.mb * (world if args.scaling == "weak" else 1)
    genome = int(total_mb * 1e6 / args.coverage)
    t0 = time.time()
    ds = Dataset.simulate(genome, read_len=args.read_len, coverage=args.coverage, repeat_frac=args.repeat_frac, seed=args.seed, keep_truth=keep_truth)
    lo, hi = j_shard(ds.nreads, rank, world)
    t1 = time.time()
    nthreads = max(1, effective_cpus() // (1 if getattr(args, "bound", False) else world))
    batch = ds.pile(lo, hi, w=args.w, a=args.a, maxalign=maxalign_of(args), maxinput=args.maxinput, nthreads=nthreads)
    t2 = time.time()
    info = {"reads_total": int(ds.nreads), "overlaps": int(ds.novl), "shard": [int(lo), int(hi)], "sim_s": round(t1 - t0, 2), "pile_s": round(t2 - t1, 2), "pile_threads": nthreads}
    return ds, batch, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--mb", type=float, default=50.0, help="sum of A-read lengths per GPU in Mb (BASELINE config 2: 50)")
    ap.add_argument("--coverage", type=float, default=40.0)
    ap.add_argument("--read-len", type=int, default=10000)
    ap.add_argument("--w", type=int, default=40)
    ap.add_argument("--a", type=int, default=10)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-sample-s", type=float, default=12.0)
    ap.add_argument("--k", type=int, default=8, help="k-mer size (BASELINE config 4 sweeps 6..14)")
    ap.add_argument("--depth-cap", type=int, default=0, help="-d: at most this many sequences per window (0 = unlimited; BASELINE config 5: 200)")
    ap.add_argument("--maxinput", type=int, default=5000, help="-D: overlaps kept per A-read")
    ap.add_argument("--repeat-frac", type=float, default=0.0, help="fraction of the genome covered by tandem repeats (BASELINE config 5: 0.2)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: --mb is the total over all GPUs (BASELINE config 3)")
    ap.add_argument("--truth-reads", type=int, default=400, help="corrected reads compared with the simulated truth (0 = off)")
    ap.add_argument("--cli", type=int, default=1, help="N=1 only: also time the `daccord` binary on the same data as .las / .db files (wall clock of the whole process)")
    ap.add_argument("--cli-oracle-reads", type=int, default=24, help="A-reads on which the oracle's file driver (all threads) is run beside the binary for a byte comparison of the FastA (0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (window results of a fixed sample of windows, corrected reads) as DIR/<name>.npy, rank 0's shard")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a sample whose size depends on the host's speed, so it has no fixed outputs to write")
    args.warmup = max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and os.environ.get("OMP_NUM_THREADS") == "1":
        # torchrun pins every rank to one OpenMP thread; the host sides of the ABI (validation, piling of the setup, host vote check) are OpenMP code:
        # give every rank its share of the host cores instead (set before the libraries that read it are loaded)
        os.environ["OMP_NUM_THREADS"] = str(max(1, effective_cpus() // world))
    workload = "%g Mb synthetic %gx pile %s (%d kb reads, 15%% error%s, LAS-equivalent overlaps with tspace=100 trace points), -w%d -a%d -k%d%s%s" % (
        args.mb, args.coverage, "per GPU" if args.scaling == "weak" else "in total, -J sharded", args.read_len // 1000,
        (", %.0f%% of the genome in tandem repeats" % (100 * args.repeat_frac)) if args.repeat_frac else "", args.w, args.a, args.k,
        (" -d%d" % args.depth_cap) if args.depth_cap else "", (" -D%d" % args.maxinput) if args.maxinput != 5000 else "")
    base = {"metric": "consensus_windows_per_s", "unit": "windows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "u32/u64 + f64", "data": "synthetic"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        from common import run_oracle, default_params
        ds, batch, info = build_workload(args, 0, 1)
        pi, pd, cor = ds.profile()
        p = default_params(w=args.w, k_lo=args.k, k_hi=args.k, p_i=pi, p_d=pd, est_cor=cor)
        packed = np.array(ds.packed(), copy=True)
        win_all, sl = batch.win, batch.sl
        threads = best_oracle_threads(run_oracle, p, packed, win_all, sl)
        # bounded sample: probe, then size each step to ~cpu_sample_s / steps of CPU work
        probe = min(len(win_all), 4000 * threads // 8 + 2000)
        _, _, _, t = run_oracle(p, packed, win_all[:probe].copy(), sl, threads)
        rate = probe / max(t, 1e-6)
        n = int(min(len(win_all), max(2000, rate * args.cpu_sample_s / max(args.steps + args.warmup, 1))))
        sample = win_all[:n].copy()
        for _ in range(args.warmup):
            run_oracle(p, packed, sample, sl, threads)
        tt, att = 0.0, 0
        for _ in range(args.steps):
            res, _, _, t = run_oracle(p, packed, sample, sl, threads)
            tt += t; att += int((res["status"] != 0).sum())
        v = att / tt
        out = dict(base, impl="reference", value=v, ms_per_step=1e3 * tt / args.steps, n_gpus=world,
                   config={"workload": workload, "sample": "first %d windows of the shard per step" % n, "threads": threads, "host_cpus": os.cpu_count(), "usable_cpus": effective_cpus(),
                           "what": "window consensus only (oracle_run_batch); CPU restatement of gt1/daccord with bit-parallel scoring, not the upstream binary: the ratio against it is an upper bound vs real daccord"},
                   cpu_baseline={"value": v, "unit": "windows/s", "cores": threads, "host_cpus": os.cpu_count(), "kind": "port", "sample": "first %d windows x %d steps" % (n, args.steps)},
                   e2e={"value": v, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        print(json.dumps(out))
        return 0

    import torch
    import daccord_b200 as d
    from daccord_b200.host import format_segments
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    args.bound = numa is not None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    total_mb = args.mb * (world if args.scaling == "weak" else 1)
    keep_truth = args.truth_reads > 0 and total_mb <= 260
    ds, batch, info = build_workload(args, rank, world, keep_truth=keep_truth)
    info["numa_node"] = numa
    pi, pd, cor = ds.profile()
    params = d.Params.default(w=args.w, k_lo=args.k, k_hi=args.k, p_i=pi, p_d=pd, est_cor=cor)
    eng = d.Engine(params, local)
    # packed read DB: one-time broadcast from rank 0 over NCCL (every rank needs the whole DB: B reads come from anywhere)
    packed_h = np.array(ds.packed(), copy=True)
    dbt = torch.empty(packed_h.size, dtype=torch.uint8, device="cuda")
    if rank == 0:
        dbt.copy_(torch.from_numpy(packed_h))
    if dist is not None:
        dist.broadcast(dbt, src=0)
    torch.cuda.synchronize()
    eng.set_reads_device(dbt.data_ptr(), dbt.numel())

    # pinned host staging of the step's inputs / outputs (the e2e legs copy them every step)
    win_p = torch.from_numpy(batch.win.view(np.uint8).copy()).pin_memory()
    sl_p = torch.from_numpy(batch.sl.view(np.uint8).copy()).pin_memory()
    win = win_p.numpy().view(d.WINDOW_DT); sl = sl_p.numpy().view(d.SLICE_DT)
    nwin = len(win)
    res_p = torch.empty(nwin * 16, dtype=torch.uint8).pin_memory(); cons_p = torch.empty(nwin * 64, dtype=torch.uint8).pin_memory(); ops_p = torch.empty(nwin * 128, dtype=torch.uint8).pin_memory()
    out = (res_p.numpy().view(d.RESULT_DT), cons_p.numpy(), ops_p.numpy())
    maxalign = maxalign_of(args)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg
    eng.upload(win, sl)
    for _ in range(args.warmup):
        eng.launch()
    sampler = ClockSampler(local); sampler.start()
    barrier()
    kms, launches, hard, second, lost = 0.0, 0, 0, 0, 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        kms += eng.launch()                 # CUDA-event time of the launch(es) on the engine's stream
        st = eng.stats(); launches += st["launches"]; hard += st["hard_windows"]; second += st["second_pass_windows"]; lost += st["lost_windows"]
    barrier()
    wall = time.perf_counter() - t0
    sampler.stop_flag = True
    res, cons, ops = eng.download(out)
    res_ref, cons_ref, ops_ref = res.copy(), cons.copy(), ops.copy()
    att = int((res["status"] != 0).sum()); okw = int((res["status"] == 1).sum())
    alg_bytes, _ = algorithmic_bytes(win, sl, res)
    tsec = kms / 1e3
    # ---- window-level entry point: dcu_run with host descriptors in, result records out
    for _ in range(1):
        eng.run(win, sl, out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.run(win, sl, out)
    barrier()
    desc_wall = time.perf_counter() - t0
    desc_same = not full_compare((res_ref, cons_ref, ops_ref), out).any()
    fasta, nseq = batch.vote(*out)           # host pile vote of the same results: the check of the GPU vote below
    corrected = sum(len(l) for l in fasta.split(b"\n") if l and not l.startswith(b">"))
    # ---- one stage earlier: overlaps + trace points in, trace reconstruction and slice extraction on the GPU (dcu_pile), result records out
    ovl, trace, boff, rlen = ds.overlaps(info["shard"][0], info["shard"][1], maxinput=args.maxinput)
    ovl_p = torch.from_numpy(ovl.view(np.uint8).copy()).pin_memory(); trace_p = torch.from_numpy(trace.view(np.uint8).copy()).pin_memory()
    ovl = ovl_p.numpy().view(ovl.dtype); trace = trace_p.numpy().view(np.uint16)
    gpu_pile = ds.tspace <= 128
    pile_wall, pile_same = None, None
    if gpu_pile:
        eng.pile(ovl, trace, ds.tspace, boff, rlen, advance=args.a, maxalign=maxalign); eng.launch(); eng.download(out)      # warm-up
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            eng.pile(ovl, trace, ds.tspace, boff, rlen, advance=args.a, maxalign=maxalign)
            eng.launch()
            eng.download(out)
        barrier()
        pile_wall = time.perf_counter() - t0
        pile_same = not full_compare((res_ref, cons_ref, ops_ref), out).any()
    # ---- e2e: the whole read-level path on the GPU: overlaps in, corrected bases out (dcu_pile + launch + dcu_vote); D2H = corrected bases only
    full_wall, full_same, full_d2h, truth, e2e_parts, reads_out = None, None, 0, None, None, None
    if gpu_pile:
        eng.pile(ovl, trace, ds.tspace, boff, rlen, advance=args.a, maxalign=maxalign); eng.launch(); seg, chars = eng.vote()      # warm-up
        chars_p = torch.empty(int(len(chars) * 1.02) + 4096, dtype=torch.uint8).pin_memory().numpy()     # pinned target of the corrected bases, like the other host buffers of the step
        barrier()
        t0 = time.perf_counter()
        tp = tl = tv = 0.0
        for _ in range(args.steps):
            ta = time.perf_counter()
            eng.pile(ovl, trace, ds.tspace, boff, rlen, advance=args.a, maxalign=maxalign)
            tb = time.perf_counter()
            eng.launch()
            tc = time.perf_counter()
            seg, chars = eng.vote(chars_out=chars_p)
            td = time.perf_counter()
            tp += tb - ta; tl += tc - tb; tv += td - tc
        barrier()
        full_wall = time.perf_counter() - t0
        e2e_parts = {"dcu_pile_ms": 1e3 * tp / args.steps, "dcu_launch_ms": 1e3 * tl / args.steps, "dcu_vote_and_get_corrected_ms": 1e3 * tv / args.steps}
        gfasta = format_segments(seg, chars)[0]
        if args.dump_outputs:
            reads_out = (seg.copy(), chars.copy())      # chars lies in chars_p, which the two-in-flight leg below writes again
        full_same = bool(gfasta == fasta)
        full_d2h = int(chars.nbytes + seg.nbytes + 16 * nwin)       # + the window descriptors dcu_vote reads back to lay out the reads
        if keep_truth and rank == 0:
            # anchor outside the oracle: the corrected reads of the GPU path against the simulated genome (first reads of the shard)
            truth = ds.truth_eval(gfasta, max_read=info["shard"][0] + args.truth_reads)
    # ---- the same with two batches in flight (one Engine each, as the command line keeps three): the window passes of the two contexts
    # alternate on the GPU, piling and vote of one batch overlap the window kernel of the other; every step still copies its inputs in and
    # its corrected bases out
    pipe_wall = None
    if gpu_pile and args.steps >= 2 and getattr(args, "pipelined", 1):
        try:
            eng2 = d.Engine(params, local)
            eng2.share_reads(eng)
            chars_p2 = torch.empty(len(chars_p), dtype=torch.uint8).pin_memory().numpy()
            eng2.pile(ovl, trace, ds.tspace, boff, rlen, advance=args.a, maxalign=maxalign); eng2.launch(); eng2.vote(chars_out=chars_p2)      # warm-up of the second context
            todo = list(range(args.steps)); lock = threading.Lock(); errs = []

            def work(e, buf):
                try:
                    while True:
                        with lock:
                            if not todo:
                                return
                            todo.pop()
                        e.pile(ovl, trace, ds.tspace, boff, rlen, advance=args.a, maxalign=maxalign)
                        e.launch()
                        e.vote(chars_out=buf)
                except Exception as ex:      # noqa: BLE001
                    errs.append(repr(ex))
            torch.cuda.synchronize()               # (no collective inside this guarded leg: a rank that skips it must not leave the others waiting)
            t0 = time.perf_counter()
            th = [threading.Thread(target=work, args=(eng, chars_p)), threading.Thread(target=work, args=(eng2, chars_p2))]
            for t in th:
                t.start()
            for t in th:
                t.join()
            torch.cuda.synchronize()
            pipe_wall = None if errs else time.perf_counter() - t0
            eng2.close()
        except Exception as ex:      # noqa: BLE001 -- an extra leg must never cost the line
            pipe_wall = None
            print("two-in-flight leg skipped: %r" % (ex,), file=sys.stderr)
    e2e_wall = full_wall if full_wall else desc_wall

    vals = torch.tensor([tsec, e2e_wall, wall, pile_wall or 0.0, desc_wall, pipe_wall or 0.0], dtype=torch.float64, device="cuda")
    cnts = torch.tensor([att, nwin, okw, corrected, launches, hard, alg_bytes, win.nbytes + sl.nbytes, res_p.numel() + cons_p.numel() + ops_p.numel(), second, lost,
                         ovl.nbytes + trace.nbytes + boff.nbytes + rlen.nbytes, full_d2h], dtype=torch.float64, device="cuda")
    per_rank = torch.zeros(world, dtype=torch.float64, device="cuda"); per_rank[rank] = tsec
    per_rank_att = torch.zeros(world, dtype=torch.float64, device="cuda"); per_rank_att[rank] = att
    flags = torch.tensor([1.0 if desc_same else 0.0, 1.0 if (pile_same or pile_same is None) else 0.0, 1.0 if (full_same or full_same is None) else 0.0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX); dist.all_reduce(cnts, op=dist.ReduceOp.SUM); dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
        dist.all_reduce(per_rank_att, op=dist.ReduceOp.SUM); dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    tsec_max, e2e_wall, wall, pile_wall_max, desc_wall_max, pipe_wall_max = [float(x) for x in vals.tolist()]
    att_t, nwin_t, ok_t, corr_t, launches_t, hard_t, alg_t, h2d_desc, d2h_desc, second_t, lost_t, h2d_ovl, d2h_full = [float(x) for x in cnts.tolist()]
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    ach = (alg_bytes * args.steps) / tsec / 1e9           # this rank's kernel: algorithmic GB/s
    traffic = None; traffic_src = None; issue = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic = tj["dram_bytes_per_window"] * att
        traffic_src = "%d B / window x windows of the launch; %s" % (tj["dram_bytes_per_window"], tj.get("source", ""))
        issue = tj.get("issue")
    except Exception:
        pass
    value = att_t * args.steps / tsec_max
    ranks_ms = [1e3 * float(x) / args.steps for x in per_rank.tolist()]
    line = dict(base, value=value, ms_per_step=1e3 * tsec_max / args.steps,
                config={"workload": workload, "windows_per_step": int(nwin_t), "attempted_per_step": int(att_t), "consensus_per_step": int(ok_t),
                        "corrected_mbp_per_s": corr_t * args.steps / tsec_max / 1e6, "l2": "inputs %.0f MB per GPU, larger than L2 (126 MB)" % ((win.nbytes + sl.nbytes) / 1e6),
                        "parallelism": "-J r,%d by A-read, no data-path collective" % world, "setup": info},
                e2e=(None if not full_wall else {"value": att_t * args.steps / e2e_wall, "unit": "windows/s", "h2d_bytes_per_step": int(h2d_ovl), "d2h_bytes_per_step": int(d2h_full),
                                                 "what": "dcu_pile + dcu_launch + dcu_vote + dcu_get_corrected: overlaps and trace points in (pinned host memory), corrected bases out",
                                                 "corrected_mbp_per_s": corr_t * args.steps / e2e_wall / 1e6, "fasta_identical_to_host_vote": bool(flags[2].item()), "rank0_ms_per_step": e2e_parts}),
                e2e_two_in_flight=(None if not pipe_wall_max else {"value": att_t * args.steps / pipe_wall_max, "unit": "windows/s",
                                                                  "what": "the e2e path with two batches in flight per GPU (two contexts, one host thread each): every step still copies its overlaps in and its corrected bases out"}),
                e2e_descriptors={"value": att_t * args.steps / desc_wall_max, "unit": "windows/s", "what": "dcu_run: window / slice descriptors in, result records + consensus + placement out",
                                 "h2d_bytes_per_step": int(h2d_desc), "d2h_bytes_per_step": int(d2h_desc), "results_identical": bool(flags[0].item())},
                e2e_from_overlaps=(None if not pile_wall else {"value": att_t * args.steps / pile_wall_max, "unit": "windows/s", "what": "dcu_pile (trace reconstruction + slices on the GPU) + launch + download of the result records",
                                                               "h2d_bytes_per_step": int(h2d_ovl), "d2h_bytes_per_step": int(d2h_desc), "results_identical": bool(flags[1].item())}),
                per_gpu={"kernel_ms_per_step": [round(x, 3) for x in ranks_ms], "attempted": [int(x) for x in per_rank_att.tolist()],
                         "imbalance_max_over_mean": (max(ranks_ms) / (sum(ranks_ms) / len(ranks_ms))) if ranks_ms and sum(ranks_ms) > 0 else None},
                gpu_launches=int(launches_t), hard_windows=int(hard_t), second_pass_windows=int(second_t), lost_windows=int(lost_t),
                smem_pass={"warps_per_sm": st["smem_warps"], "bytes_per_warp": st["smem_bytes_per_warp"]},
                roofline={"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src,
                          "peak_source": peak_src, "bytes_per_window": alg_bytes / max(att, 1), "issue": issue,
                          "note": "integer / latency bound path (SURVEY 8d): the HBM fraction is reported as the contract asks; `issue` holds the instruction-issue figures of the same ncu capture"},
                accuracy=truth, clocks=sampler.summary(), wall_s_timed=wall)
    if not full_wall:       # -w not a multiple of -a: the GPU piler does not apply, the descriptor path is the end-to-end number
        line["e2e"] = dict(line["e2e_descriptors"])
    # ---- the command line itself: `daccord reads.las reads.db > fasta` on the same data as files (process start, DB + LAS ingest, CUDA context,
    # error-profile file, pipelined batches, FastA text); compared with the library path above and, on a read range, with the oracle's file driver
    if world == 1 and args.cli and full_wall:
        import tempfile
        exe = os.path.join(ROOT, "daccord_b200", "_build", "daccord")
        with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
            las, db = os.path.join(tmp, "b.las"), os.path.join(tmp, "b.db")
            ds.write(las, db)
            opts = ["-w%d" % args.w, "-a%d" % args.a, "-k%d" % args.k, "-D%d" % args.maxinput] + (["-d%d" % args.depth_cap] if args.depth_cap else [])
            subprocess.run([exe] + opts + ["-I0,3", las, db], capture_output=True)          # first touch: page in the binary and the files, build the .dcuidx index
            t0 = time.perf_counter()
            r = subprocess.run([exe] + opts + ["--device%d" % local, las, db], capture_output=True)
            cli_wall = time.perf_counter() - t0
            cli = {"value": att / cli_wall if r.returncode == 0 else None, "unit": "windows/s", "wall_s": cli_wall, "rc": r.returncode,
                   "what": "`daccord %s b.las b.db` as one process: DB + LAS load, CUDA context, tables, 3 batches in flight, FastA on stdout" % " ".join(opts),
                   "fasta_identical_to_library_path": bool(r.stdout == gfasta), "fraction_of_e2e": (att / cli_wall) / (att * args.steps / e2e_wall) if r.returncode == 0 else None}
            cli["laps"] = [l[4:] for l in r.stderr.decode(errors="replace").split("\n") if l.startswith("[T] ")]
            if r.returncode != 0:
                cli["stderr_tail"] = r.stderr.decode(errors="replace")[-400:]
            if args.cli_oracle_reads > 0 and r.returncode == 0:
                sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
                from make_golden import oracle_fasta
                from common import default_params
                last = min(args.cli_oracle_reads, int(ds.nreads)) - 1
                po = default_params(w=args.w, k_lo=args.k, k_hi=args.k, p_i=pi, p_d=pd, est_cor=cor)
                t0 = time.perf_counter()
                want, ost = oracle_fasta(po, las, db, 0, last, a=args.a, threads=effective_cpus()) if (not args.depth_cap and args.maxinput == 5000) else (None, None)
                cli["oracle_files_s"] = time.perf_counter() - t0
                if want is not None:
                    r2 = subprocess.run([exe] + opts + ["-I0,%d" % last, "--device%d" % local, las, db], capture_output=True)
                    cli["fasta_identical_to_oracle_file_driver"] = bool(r2.returncode == 0 and r2.stdout == want)
                    cli["oracle_reads"] = last + 1
        line["e2e_cli"] = cli
    # CPU baseline: the oracle on a bounded sample of the same windows, all host threads (rank 0, N=1 only); full comparison of the sample
    if world == 1 and args.cpu_sample_s > 0:
        from common import run_oracle, default_params
        p = default_params(w=args.w, k_lo=args.k, k_hi=args.k, p_i=pi, p_d=pd, est_cor=cor)
        threads = best_oracle_threads(run_oracle, p, packed_h, batch.win, batch.sl)
        probe = min(nwin, 2000 + 500 * threads)
        r0, _, _, t = run_oracle(p, packed_h, batch.win[:probe].copy(), batch.sl, threads)
        n = int(min(nwin, max(probe, probe / max(t, 1e-6) * args.cpu_sample_s)))
        r1, c1, o1, t = run_oracle(p, packed_h, batch.win[:n].copy(), batch.sl, threads)
        diff = full_compare((r1, c1, o1), (res_ref[:n], cons_ref[:n * 64], ops_ref[:n * 128]))
        line["cpu_baseline"] = {"value": float((r1["status"] != 0).sum() / t), "unit": "windows/s", "cores": threads, "host_cpus": os.cpu_count(), "usable_cpus": effective_cpus(), "kind": "port",
                                "sample": "first %d windows of the step, %.1f s" % (n, t), "gpu_results_identical_on_sample": not diff.any(),
                                "compared": "result record, consensus bytes and placement trace of every sampled window", "differing_windows": int(diff.sum()),
                                "note": "CPU restatement of gt1/daccord (bit-parallel scoring, -march=x86-64-v3), not the upstream binary: GPU/CPU ratios are upper bounds vs real daccord"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, (res_ref, cons_ref, ops_ref), reads_out)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
