#!/usr/bin/env python
"""bench.py — parent-set local scores per second on B200 (BASELINE.json metric), one JSON line on rank 0.

Workload (default): BASELINE.json configs[3] — synthetic discrete BN p=60, n=1M, arity<=4, generating-graph skeleton
(stand-in for MMPC), `-p 12` (effective BIC cap 11), BIC + ScoreCache pruning.  It is the configuration the metric's
roofline target is quoted on and the largest discrete one that fits a single GPU; configs[0..2] are parity-test
cases (tests/), configs[4] needs 8 GPUs and wide masks (DESIGN.md).  `--workload cbic` runs configs[2]
(linear-Gaussian p=30, n=100k, cBIC lambda=2, exhaustive) instead.

A step = one pass of the hot path over every variable this rank owns (variables striped v % N as the reference
stripes its threads, score_main.cpp:136-139): score every candidate parent set, apply the store rule and the
subset-dominance prune, results left on the device.  `value` = sets scored by all ranks / max-over-ranks device
time.  `e2e` repeats the same through the public API with HOST buffers: the H2D copy of the data from pinned
memory and the D2H fetch of every variable's surviving (mask, score) list are inside the timed region.

--dump-outputs DIR: the timed steps drop their results on the device, so after them one more pass of the same step, outside
the timed region, reads every score cache back and writes it (dump_outputs).  The step is deterministic, so these are the
caches each timed step computed; two builds can be compared output for output on the same seeded inputs.

--impl reference times the CPU oracle's restatement of the reference path (oracle/, or oracle/_ref when the
reference's own sources were compiled) on the host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "parent-set local scores/sec"
UNIT = "sets/s"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return float(pk.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(kind):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture (profiles/traffic.json, written from the .ncu-rep by tools/traffic_from_ncu.py); None when absent."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(kind)
    return None


def load_k1_dram():
    """DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of EVERY K1 launch of one step, summed per kernel, from the
    committed ncu pass over `bench.py --one-pass` (profiles/r02_k1_dram.json, written by tools/k1_dram_from_ncu.py from the
    per-launch CSV next to it); None when absent."""
    path = os.path.join(ROOT, "profiles", "r02_k1_dram.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


def traffic_fields(kind):
    t = load_traffic(kind)
    if not t:
        return {"traffic": None}
    return {"traffic": t["dram_bytes_per_launch"], "traffic_detail": {k: t[k] for k in ("kernel", "grid", "launch_us_under_ncu", "dram_gbps_under_ncu", "report")}}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.reasons = set()
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nme, val in zip(names, f[2:6]):
                    if val.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------- workloads

BIC_NAME = ("configs[3]: synthetic discrete BN p=60 n=1e6 arity<=4 seed=4, generating-graph skeleton (2-hop), -p 12 -> cap 11, "
            "BIC + prune")


def bic_block(pkg, block):
    """block 0 is BASELINE configs[3] itself; block b > 0 has the same arities, DAG and skeleton with its own CPTs and rows"""
    return pkg.datagen.discrete_bn(p=60, n=1_000_000, seed=4, sample_seed=None if block == 0 else 1000 + block)


def make_bic_workload(pkg, blocks=1, codes=None, card=None):
    """`blocks` replicas of the config-4 network side by side in one data set of 60*blocks variables (block-diagonal
    skeleton).  codes/card may be passed in (multi-GPU: every rank generated one block and they were all-gathered)."""
    pb, n = 60, 1_000_000
    if codes is None:
        parts = [bic_block(pkg, b) for b in range(blocks)]
        codes = np.concatenate([q[0] for q in parts], axis=0)
        card = np.concatenate([q[1] for q in parts])
    _, _, edges0, _ = pkg.datagen.discrete_bn(p=pb, n=2, seed=4)  # the structure only (tiny sample)
    p = pb * blocks
    edges = [edges0[i % pb] << (pb * (i // pb)) for i in range(p)]
    K = pkg.effective_max_parents(12, pb, n, True)
    nbs = [pkg.two_hop_neighbors(edges, p, v) for v in range(p)]
    name = BIC_NAME if blocks == 1 else BIC_NAME + f"; weak scaling: {blocks} replicas of that network (own CPTs and rows) as one {p}-variable data set"
    return dict(kind="bic", p=p, n=n, codes=codes, card=np.asarray(card, dtype=np.int32), edges=edges, K=K, nbs=nbs, name=name, blocks=blocks)


def make_cbic_workload(pkg):
    p, n = 30, 100_000
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=3)
    nbs = [(1 << p) - 1] * p
    return dict(kind="cbic", p=p, n=n, x=x, K=p - 1, nbs=nbs, lam=2.0, blocks=1,
                name="configs[2]: synthetic linear-Gaussian SEM p=30 n=1e5 seed=3, cBIC lambda=2, all-ones skeleton (2^29 sets/variable), accept + prune")


def family_size(c, K):
    from math import comb
    return sum(comb(c, l) for l in range(0, min(c, K) + 1))


def sets_of(wl, v):
    c = bin(wl["nbs"][v] & ~(1 << v)).count("1")
    return family_size(c, wl["K"])


def owners_of(pkg, wl, world):
    """variable -> rank.  BIC: longest-processing-time-first on the predicted table cells (families differ by orders of
    magnitude); cBIC config 3: every family has the same size, the reference's striping v % N is already balanced."""
    D = importlib.import_module("urlearning-cpp_b200.distributed")
    if wl["kind"] != "bic" or world == 1:
        return [v % world for v in range(wl["p"])]
    costs = [D.family_cost(wl["card"], v, wl["nbs"][v], wl["K"]) for v in range(wl["p"])]
    return D.assign_lpt(costs, world)


# ---------------------------------------------------------------------------------------------- GPU arm

def run_gpu(args):
    import torch
    pkg = importlib.import_module("urlearning-cpp_b200")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # T contexts (streams) on this GPU, one host thread each: the reference's `-t T` worker threads (score_main.cpp:372-380)
    # pointed at one device.  Raises if the CUDA library or the device is missing: no fallback.
    is_bic = args.workload == "bic"
    T = max(1, args.threads_per_gpu) if is_bic else 1
    pool = pkg.EnginePool(local, T)
    eng = pool.engines[0]
    # one non-default stream for the timing events and the L2 flush (the legacy default stream would serialise with the engines' streams)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    if T == 1:
        eng.set_stream(stream.cuda_stream)
    weak = is_bic and args.scaling == "weak"

    # ---- inputs (SURVEY.md 8e).
    #   weak BIC (the default with N > 1): rank r owns replica r of the configs[3] network — same arities, DAG and skeleton, its
    #     own CPTs and rows — generates it, uploads only those 60 columns and scores its 60 variables; the per-variable caches
    #     are gathered to rank 0 over NCCL (inside the timed region of the e2e arm).  Work per GPU is fixed exactly.
    #   strong BIC (--scaling strong, and the `scaling_strong` sub-record of every N > 1 line): rank 0 generates configs[3], the
    #     packed codes are broadcast over NCCL, variables are dealt out by predicted cost (LPT), caches gathered to rank 0.
    #   cBIC: rank 0 forms the Gram, the p*p Gram is broadcast.
    D = importlib.import_module("urlearning-cpp_b200.distributed")

    def strong_inputs():
        wl_ = make_bic_workload(pkg, 1) if rank == 0 else None
        if world == 1:
            return wl_, None
        box = [None if wl_ is None else {k: v for k, v in wl_.items() if k != "codes"}]
        dist.broadcast_object_list(box, src=0)
        dev_ = torch.empty((box[0]["p"], box[0]["n"]), dtype=torch.uint8, device="cuda")
        if rank == 0:
            dev_.copy_(torch.from_numpy(wl_["codes"]))
        dist.broadcast(dev_, src=0)
        return (wl_ if rank == 0 else dict(box[0])), dev_

    dev = None
    shift, p_global = 0, None
    if is_bic:
        if world > 1 and weak:
            codes_b, card_b, _, _ = bic_block(pkg, rank)
            wl = make_bic_workload(pkg, 1, codes=codes_b, card=card_b)
            wl["name"] = BIC_NAME + f"; weak scaling: {world} replicas of that network (own CPTs and rows), replica r on GPU r"
            shift, p_global = 60 * rank, 60 * world
        else:
            wl, dev = strong_inputs()
    else:
        wl = make_cbic_workload(pkg) if rank == 0 else None
        if world > 1:
            box = [None if wl is None else {k: v for k, v in wl.items() if k != "x"}]
            dist.broadcast_object_list(box, src=0)
            wl = wl if rank == 0 else dict(box[0])
    p_global = p_global or wl["p"]
    flags = pkg.PRUNE_DOMINATED
    stype = pkg.BIC if is_bic else pkg.CBIC
    lam = wl.get("lam", 0.0)

    pinned = None
    if is_bic:
        if dev is not None:
            torch.cuda.synchronize()
            pool.set_discrete_device(dev.data_ptr(), wl["n"], wl["p"], wl["card"])
            pinned = dev.cpu().pin_memory()
            del dev
        else:
            pinned = torch.from_numpy(wl["codes"]).pin_memory()
            pool.set_discrete(pinned.numpy(), wl["card"])
    else:
        if rank == 0:
            pinned = torch.from_numpy(wl["x"]).pin_memory()
            eng.set_continuous(pinned.numpy())
            g = torch.from_numpy(eng.gram()).cuda()
        else:
            g = torch.empty((wl["p"], wl["p"]), dtype=torch.float64, device="cuda")
        if world > 1:
            dist.broadcast(g, src=0)
            if rank != 0:
                eng.set_gram(g.cpu().numpy(), wl["n"])

    if is_bic and world > 1 and weak:
        owner = [rank] * wl["p"]                       # local view: every variable of my replica is mine
        owner_global = [v // 60 for v in range(p_global)]
    else:
        owner = owners_of(pkg, wl, world)
        owner_global = owner
    mine = [v for v in range(wl["p"]) if owner[v] == rank]
    sets_mine = sum(sets_of(wl, v) for v in mine)
    items = [(v, wl["nbs"][v]) for v in mine]
    costs = [D.family_cost(wl["card"], v, wl["nbs"][v], wl["K"]) for v in mine] if is_bic else None
    words_global = pkg.mask_words_for(p_global)

    def to_global(masks):
        """local one-word masks [n, 1] -> [n, words_global] with every variable index shifted by `shift`"""
        m = np.ascontiguousarray(masks, dtype=np.uint64).reshape(len(masks), -1)
        if shift == 0 and m.shape[1] == words_global:
            return m
        out = np.zeros((len(m), words_global), dtype=np.uint64)
        w0, b = shift // 64, shift % 64
        out[:, w0] = m[:, 0] << np.uint64(b)
        if b and w0 + 1 < words_global:
            out[:, w0 + 1] = m[:, 0] >> np.uint64(64 - b)
        return out

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def step(fetch=False):
        """one pass of the hot path over this rank's variables (dealt to the pool's contexts by predicted cost).  fetch: read
        every surviving cache back to the host (into the context's page-locked result buffer, as a driver that formats each
        variable's block as it arrives would), software-pipelined one variable deep (v+1 is enqueued before v is read).
        Returns after every context has drained, so consecutive steps do not overlap."""
        flush.fill_(1)  # L2 flush between steps (inside the timed region: ~40 us of a step of hundreds of ms)
        stream.synchronize()
        if fetch and world > 1 and is_bic:
            # N > 1: the caches travel to rank 0 (the .pss writer) over NCCL inside the timed region
            if args.gather == "p2p":
                # the compacted caches go from every GPU straight into rank 0's device memory over NVLink (CUDA IPC mapping,
                # urlgpu_result_fetch_device), rank 0 reads the whole area back once
                t0_ = time.perf_counter()
                kept = pool.run(items, wl["K"], stype, lam=lam, flags=flags, fetch="keep", costs=costs)
                if os.environ.get("URLGPU_GATHER_TIMING"):
                    t1_ = time.perf_counter()
                    torch.cuda.synchronize()
                    t2_ = time.perf_counter()
                    print("[step rank %d] pool.run(keep) %.1f ms, device sync after it %.1f ms (wall %.3f)" % (rank, 1e3 * (t1_ - t0_), 1e3 * (t2_ - t1_), time.time() % 100), flush=True)
                try:
                    allc = D.gather_results_p2p(eng, kept, p_global, words_global, owner=owner_global, shift=shift, copy=False)
                except D.PeerMemoryUnavailable as ex:     # raised on every rank together: all switch to the NCCL gather
                    if rank == 0:
                        print("bench: peer memory unavailable (%s): using --gather nccl" % ex, file=sys.stderr)
                    args.gather = "nccl"
                    for r in kept.values():
                        r.free()
                    return step(fetch=True)
                nst_ = sum(r.count() for r in kept.values())
                for r in kept.values():
                    r.free()
            else:
                got = pool.run(items, wl["K"], stype, lam=lam, flags=flags, fetch=True, costs=costs)
                local = {v + shift: (to_global(m), sc) for v, (m, sc) in got.items()}
                allc = D.gather_caches(local, p_global, words_global, "cuda", owner=owner_global, copy=False)
                nst_ = sum(len(sc) for _, sc in got.values())
            if rank == 0:
                assert len(allc) == p_global
            return nst_
        out = pool.run(items, wl["K"], stype, lam=lam, flags=flags, fetch="pinned" if fetch else False, costs=costs)
        return sum(out.values()) if fetch else 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxed(ms):
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed(nsteps, fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = 0
        for _ in range(nsteps):
            out += fn()
        e1.record(stream)
        barrier()
        return maxed(e0.elapsed_time(e1)), out

    if args.one_pass:
        # for `ncu --profile-from-start off`: one warm pass, then exactly one pass of the step on ONE context between
        # cudaProfilerStart/Stop (the launches profiles/r02_k1_dram.* and the launch lists are made from); no JSON line
        step()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        pool.run(items, wl["K"], stype, lam=lam, flags=flags, fetch=False, costs=costs, contexts=1)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        if rank == 0:
            print(json.dumps({"one_pass": True, "sets": sets_mine, "launches": pool.stats()["launches_total"]}))
        pool.close()
        return

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    sampler.start()
    t16_warm = int(pool.stats().get("table16_fallbacks", 0))   # variables whose speculative 16-bit tables overflowed during the warm-up (remembered: 32-bit from then on)
    pool.reset_stats()
    ms, _ = timed(args.steps, step)
    launches_total = pool.stats()["launches_total"]
    # per-kernel device time for the roofline: one more pass of the same step on ONE context, so kernels run one at a time
    # and the library's CUDA events (recorded on the launching stream around every kernel family) do not overlap
    eng.reset_stats()
    eng.enable_timing(True)
    flush.fill_(1)
    stream.synchronize()
    pool.run(items, wl["K"], stype, lam=lam, flags=flags, fetch=False, costs=costs, contexts=1)
    st = eng.stats()
    eng.enable_timing(False)
    roof_steps = 1
    sampler.stop_flag = True
    sampler.join(timeout=2)

    total_sets = sets_mine
    if world > 1:
        t = torch.tensor([sets_mine], device="cuda", dtype=torch.int64)
        dist.all_reduce(t)
        total_sets = int(t.item())
    value = total_sets * args.steps / (ms / 1e3)

    # ---- e2e: the public API with HOST buffers: the H2D copy of the data from pinned memory (every rank uploads the columns
    # its variables need: its own replica in the weak arm), the D2H fetch of every surviving (mask, score) list and, with
    # N > 1, the NCCL gather of the caches to rank 0 are inside the timed region
    e2e = None
    if is_bic or world == 1:
        host = pinned.numpy()

        def e2e_step():
            t0 = time.perf_counter()
            if is_bic:
                pool.set_discrete(host, wl["card"])  # one upload per GPU; the pool's other contexts borrow the device copy
            else:
                pool.set_continuous(host)
            t1 = time.perf_counter()
            out = step(fetch=True)
            if os.environ.get("URLGPU_GATHER_TIMING"):
                print("[e2e_step rank %d] upload %.1f ms, step+gather %.1f ms" % (rank, 1e3 * (t1 - t0), 1e3 * (time.perf_counter() - t1)), flush=True)
            return out

        e2e_step()
        nst = max(1, min(args.steps, 3))
        ems, stored = timed(nst, e2e_step)
        h2d = (wl["n"] * wl["p"]) * (1 if is_bic else 8) * world   # per rank: the columns of its own data set
        if world > 1:
            t = torch.tensor([stored], device="cuda", dtype=torch.int64)
            dist.all_reduce(t)
            stored = int(t.item())
        words = pkg.mask_words_for(wl["p"])
        e2e = {"value": total_sets * nst / (ems / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int((8 * words + 4) * stored // nst), "steps": nst, "ms_per_step": ems / nst}
        if world > 1:
            e2e["gather_to_rank0"] = ("%s, inside the timed region: %d bytes per step" % (
                "device to device over NVLink into rank 0's memory (CUDA IPC peer mapping), then one D2H on rank 0" if args.gather == "p2p"
                else "NCCL gather of host-packed blocks", int((8 * words_global + 4) * stored // nst)))

    # ---- strong-scaling sub-record of every N > 1 weak line: configs[3] ITSELF split over the ranks (codes broadcast over NCCL,
    # variables dealt out by predicted cost, device-resident timing like `value`, then one e2e pass with the NCCL gather)
    strong = None
    if is_bic and world > 1 and weak:
        wl_s, dev_s = strong_inputs()
        torch.cuda.synchronize()
        pool.set_discrete_device(dev_s.data_ptr(), wl_s["n"], wl_s["p"], wl_s["card"])
        del dev_s
        owner_s = owners_of(pkg, wl_s, world)
        mine_s = [v for v in range(wl_s["p"]) if owner_s[v] == rank]
        items_s = [(v, wl_s["nbs"][v]) for v in mine_s]
        costs_s = [D.family_cost(wl_s["card"], v, wl_s["nbs"][v], wl_s["K"]) for v in mine_s]
        sets_s = sum(sets_of(wl_s, v) for v in range(wl_s["p"]))
        words_s = pkg.mask_words_for(wl_s["p"])

        def step_s(fetch=False):
            flush.fill_(1)
            stream.synchronize()
            if not fetch:
                pool.run(items_s, wl_s["K"], stype, flags=flags, fetch=False, costs=costs_s)
                return 0
            if args.gather == "p2p":
                kept = pool.run(items_s, wl_s["K"], stype, flags=flags, fetch="keep", costs=costs_s)
                try:
                    allc = D.gather_results_p2p(eng, kept, wl_s["p"], words_s, owner=owner_s, copy=False)
                except D.PeerMemoryUnavailable:
                    args.gather = "nccl"
                    for r in kept.values():
                        r.free()
                    return step_s(True)
                nst_ = sum(r.count() for r in kept.values())
                for r in kept.values():
                    r.free()
            else:
                got = pool.run(items_s, wl_s["K"], stype, flags=flags, fetch=True, costs=costs_s)
                allc = D.gather_caches(got, wl_s["p"], words_s, "cuda", owner=owner_s, copy=False)
                nst_ = sum(len(sc) for _, sc in got.values())
            if rank == 0:
                assert len(allc) == wl_s["p"]
            return nst_
        step_s()
        nss = max(1, min(args.steps, 5))
        sms, _ = timed(nss, step_s)
        step_s(True)
        ems_s, _ = timed(1, lambda: step_s(True))
        strong = {"workload": wl_s["name"], "scaling": "strong", "value": sets_s * nss / (sms / 1e3), "unit": UNIT, "steps": nss, "ms_per_step": sms / nss,
                  "e2e_gather_ms_per_step": ems_s, "sets_per_step": sets_s,
                  "parallelism": f"configs[3] itself: codes broadcast over NCCL, 60 variables dealt to {world} ranks by predicted cost (LPT), caches gathered to rank 0"}

    mem_free, mem_total = torch.cuda.mem_get_info()
    t16_fallbacks = int(pool.stats().get("table16_fallbacks", 0))   # timed regions (value, roofline pass, e2e), summed over the ranks
    if world > 1:
        t = torch.tensor([t16_fallbacks, t16_warm], device="cuda", dtype=torch.int64)
        dist.all_reduce(t)
        t16_fallbacks, t16_warm = int(t[0].item()), int(t[1].item())
    if args.dump_outputs:
        # the step is deterministic (integer counts, fixed-order reductions, bit-identical caches on every context), so one
        # more pass over the same inputs that reads the caches back returns what the last timed step left on the device
        dump_outputs(args.dump_outputs, pool.run(items, wl["K"], stype, lam=lam, flags=flags, fetch=True, costs=costs))
    if rank == 0:
        peak, peak_src = load_peaks()
        fam = {"count": st["ms_count"], "cube": st["ms_cube"], "tree": st["ms_tree"], "cbic": st["ms_cbic"], "accept": st["ms_accept"],
               "prune": st["ms_prune"]}
        dom = max(fam, key=fam.get)
        if is_bic:
            k1_ms = st["ms_count"] + st["ms_cube"] + st["ms_tree"]
            k1_launches = st["launches_count"] + st["launches_cube"] + st["launches_tree"]
            alg_gbs = st["algorithmic_bytes"] / (k1_ms / 1e3) / 1e9 if k1_ms > 0 else None
            issued = (st["k1_bytes_read"] + st["k1_bytes_written"]) / roof_steps
            # The admissible fraction: DRAM bytes the K1 kernels really moved (ncu dram__bytes_read+write summed over ALL K1
            # launches of one step, committed under profiles/) / the K1 kernel time measured live here / the measured HBM peak.
            # The algorithmic figure n*(|S|+1) per set (SURVEY 8d) is kept as effective_algorithmic_gbs: the cube path derives
            # most tables by marginalisation instead of re-reading rows, so that number exceeds the peak and is not a fraction.
            dram = load_k1_dram()
            dram_bytes = dram["k1_dram_bytes_per_step"] if dram else None
            achieved = dram_bytes / (k1_ms / roof_steps / 1e3) / 1e9 if dram_bytes and k1_ms > 0 else None
            dom_k = dram["dominant_kernel"] if dram else None
            roofline = {"bound": "hbm", "kernel": "K1 = bic_root_kernel (root tables counted from bucketed packed rows; fused roots hand their "
                                                  "children straight on) + cube_derive_kernel (every other table by marginalisation, scored in the same pass)",
                        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if achieved else None,
                        "traffic": dom_k["dram_bytes_per_launch"] if dom_k else None,
                        "traffic_detail": ({"dominant_kernel": dom_k, "per_kernel": dram["per_kernel"], "source": dram["source"]} if dram else None),
                        "definition": "achieved = DRAM bytes of all K1 launches of one step (ncu, profiles/r02_k1_dram.json) / K1 kernel ms of this run",
                        "limiter": (dram.get("limiter") if dram else None),
                        "peak_source": peak_src,
                        "effective_algorithmic_gbs": alg_gbs,
                        "algorithmic_bytes_per_step": st["algorithmic_bytes"] / roof_steps, "kernel_ms_per_step": k1_ms / roof_steps,
                        "launches_per_step": k1_launches / roof_steps, "share_of_step": k1_ms / roof_steps / (ms / args.steps),
                        "issued_bytes_per_step": issued,
                        "issued_frac_of_peak": issued / (k1_ms / roof_steps / 1e3) / 1e9 / peak if k1_ms > 0 else None,
                        "timed_on": "one extra pass of the step on a single context (kernels serial); value/e2e use all contexts, "
                                    "whose kernels overlap, so share_of_step is kernel time of the serial pass / step time of the concurrent one",
                        "note": "effective_algorithmic_gbs = sum over scored sets of n*(|S|+1) (SURVEY 8d) / K1 time: what a row-streaming "
                                "kernel would have to sustain; issued_* = bytes the K1 kernels load/store according to the host plan (L2 hits "
                                "included), an upper bound of the DRAM traffic.  The K1 kernels are bound by instruction issue (limiter): halving "
                                "their HBM bytes with 16-bit tables (round 2) cut DRAM traffic from 858 to 471 GB per step and the step by 4 %, so the "
                                "DRAM fraction FELL from 0.43 to 0.24 while the kernels got faster",
                        "family_ms": fam}
        else:
            k3_ms = st["ms_cbic"]
            achieved = st["algorithmic_flops"] / (k3_ms / 1e3) / 1e12 if k3_ms > 0 else None
            fp64 = eng.probe_fp64()
            roofline = {"bound": "fp64", "kernel": "K3 cbic sweep DFS", "achieved": achieved, "peak": fp64["dfma"], "unit": "TFLOP/s",
                        "frac": achieved / fp64["dfma"] if achieved else None, **traffic_fields("cbic"),
                        "peak_source": "measured in this run (urlgpu_probe_fp64: register-resident DFMA chains); DMMA m8n8k4: %.1f TFLOP/s" % fp64["dmma"],
                        "note": "achieved counts the per-set k^3/3+2k^2+2k flops of SURVEY 8d; the sweep DFS shares work between sets "
                                "(~4 FMAs per set), so it can exceed the FMA peak and is an equivalent-work figure, not a pipe utilisation",
                        "algorithmic_flops_per_step": st["algorithmic_flops"] / roof_steps, "kernel_ms_per_step": k3_ms / roof_steps,
                        "share_of_step": k3_ms / roof_steps / (ms / args.steps), "family_ms": fam}
        cpu = cpu_baseline(wl, args) if world == 1 and not args.no_cpu_baseline else None
        # the rest of BASELINE.json's metric ("BIC & cBIC ...; score-file wall time"), measured by the same default command
        extra = {}
        if world == 1 and is_bic and not args.no_subrecords:
            try:
                extra["other_scores"] = measure_other_scores(pkg, D, torch, pool, wl, flags)
            except Exception as ex:
                extra["other_scores"] = {"error": repr(ex)}
            pool.close()
            pool = None
            import tempfile
            try:
                extra["cbic"] = measure_cbic_subrecord(pkg, torch, local)
            except Exception as ex:  # reported, never hidden
                extra["cbic"] = {"error": repr(ex)}
            try:
                with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
                    extra["score_file"] = measure_score_file(pkg, wl, td)
            except Exception as ex:
                extra["score_file"] = {"error": repr(ex)}
        scaling = "weak" if weak else "strong"
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": "int32 counts / int64 fixed-point log-likelihood -> f32" if is_bic else "f64 -> f32",
                "data": "synthetic (seeded numpy generator, urlearning-cpp_b200/datagen.py)",
                "config": {"workload": wl["name"], "sets_per_step": total_sets,
                           "parallelism": (("replica r of the network on GPU r (its own 60 columns uploaded there), caches gathered to rank 0 over NCCL"
                                            if (weak and world > 1) else "variables dealt to ranks by predicted cost (LPT)") if is_bic
                                           else "variables striped v % N") + f", N={world}; "
                                          f"{T} context(s)/stream(s) per GPU, one host thread each (the reference's -t workers)",
                           "l2": "flushed between steps (256 MB write)", "dominant_family": dom,
                           "table16_fallbacks": t16_fallbacks, "table16_fallbacks_warmup": t16_warm,
                           "hbm_in_use_gb": round((mem_total - mem_free) / 1e9, 1)},
                "e2e": e2e, "gpu_launches": int(launches_total), "clocks": sampler.summary(), "roofline": roofline,
                "cpu_baseline": cpu, **extra, **({"scaling_strong": strong} if strong else {})}
        print(json.dumps(line))
    if world > 1:
        D.release_boards()
        dist.barrier()
        dist.destroy_process_group()
    if pool is not None:
        pool.close()



DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, caches, limit=DUMP_LIMIT, seed=0):
    """Write the per-variable score caches {variable: (masks uint64 [n, words], scores float32 [n])} as .npy files, one row
    per stored parent set, variables ascending and each cache in its canonical (|S|, mask) order:
      variable.npy  float64 [N]            the child variable
      parents.npy   float64 [N, 2*words]   every 64-bit parent-mask word as two exact 32-bit halves, low half first
      scores.npy    float32 [N]            the stored score
      index.npy     float64 [N]            the row's position in the full output
    When the full output exceeds `limit` bytes, a fixed seeded sample of rows (kept in order) is written instead."""
    vs = sorted(caches)
    masks = np.concatenate([np.asarray(caches[v][0], dtype=np.uint64) for v in vs])
    scores = np.concatenate([np.asarray(caches[v][1], dtype=np.float32) for v in vs])
    variable = np.concatenate([np.full(len(caches[v][1]), v, dtype=np.float64) for v in vs])
    index = np.arange(len(scores), dtype=np.int64)
    rows = (limit - 4 * 128) // (8 + 8 * 2 * masks.shape[1] + 4 + 8)   # 128: one .npy header
    if len(scores) > rows:
        index = np.sort(np.random.default_rng(seed).choice(len(scores), size=rows, replace=False))
    halves = np.stack([masks[index] & np.uint64(0xFFFFFFFF), masks[index] >> np.uint64(32)], axis=2).reshape(len(index), -1)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("variable", variable[index]), ("parents", halves.astype(np.float64)), ("scores", scores[index]),
                    ("index", index.astype(np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- sub-records of the default line

def fast_write_csv(path, codes):
    """codes uint8 [p, n] with single-digit values -> CSV, one record per line (numpy only: np.savetxt takes minutes at n = 1e6)"""
    p, n = codes.shape
    buf = np.empty((n, 2 * p), dtype=np.uint8)
    buf[:, 0::2] = codes.T + ord("0")
    buf[:, 1::2] = ord(",")
    buf[:, -1] = ord("\n")
    buf.tofile(path)


def measure_other_scores(pkg, D, torch, pool, wl, flags, steps=3):
    """SURVEY.md 8f-4: the other discrete scores on K1's counts, device-resident like `value`.  fNML: configs[3] itself (same
    kernels as BIC, the regret table as the per-configuration table).  BDeu (ess = 1): the configs[3] network sampled at
    n = 2e4 with -p 6 — BDeu runs on the direct-counting kernels (one table per set), at the sample sizes it is used with."""
    out = []
    small_codes, small_card, _, _ = pkg.datagen.discrete_bn(p=60, n=20_000, seed=4)
    items = [(v, wl["nbs"][v]) for v in range(wl["p"])]
    for name, codes, card, K, stype, lam, note in (
            ("fNML", wl["codes"], wl["card"], wl["K"], pkg.FNML, 0.0, "configs[3] data and skeleton, -p %d (fNML has no log-bound), prune" % wl["K"]),
            ("BDeu", small_codes, small_card, 6, pkg.BDEU, 1.0, "configs[3] network sampled at n=2e4, -p 6, ess=1, prune")):
        pool.set_discrete(np.ascontiguousarray(codes), card)
        costs = [D.family_cost(card, v, wl["nbs"][v], K) for v in range(wl["p"])]
        sets = sum(family_size(bin(wl["nbs"][v] & ~(1 << v)).count("1"), K) for v in range(wl["p"]))
        pool.run(items, K, stype, lam=lam, flags=flags, costs=costs)
        pool.reset_stats()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            pool.run(items, K, stype, lam=lam, flags=flags, costs=costs)   # returns after every context has drained
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out.append({"score": name, "workload": note, "sets_per_step": sets, "ms_per_step": ms, "value": sets / ms * 1e3, "unit": UNIT, "steps": steps,
                    "gpu_launches": int(pool.stats()["launches_total"])})
    return out


def measure_cbic_subrecord(pkg, torch, device):
    """BASELINE configs[2] next to the default line (the metric is "BIC & cBIC"): p=30, n=1e5, 2^29 sets per variable,
    acceptance + prune, results left on the device.  One warm-up step and two timed ones (CUDA events), then one pass with
    the library's per-family events."""
    wl = make_cbic_workload(pkg)
    eng = pkg.Engine(device)
    stream = torch.cuda.Stream()
    eng.set_stream(stream.cuda_stream)
    eng.set_continuous(wl["x"])
    sets = sum(sets_of(wl, v) for v in range(wl["p"]))

    def step():
        for v in range(wl["p"]):
            eng.score_variable(v, wl["nbs"][v], wl["K"], pkg.CBIC, lam=wl["lam"], flags=pkg.PRUNE_DOMINATED).free()
    step()
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nst = 2
    e0.record(stream)
    for _ in range(nst):
        step()
    e1.record(stream)
    stream.synchronize()
    ms = e0.elapsed_time(e1)
    eng.reset_stats()
    eng.enable_timing(True)
    step()
    st = eng.stats()
    fp64 = eng.probe_fp64()
    eng.close()
    return {"workload": wl["name"], "value": sets * nst / (ms / 1e3), "unit": UNIT, "steps": nst, "warmup": 1, "ms_per_step": ms / nst, "sets_per_step": sets,
            "family_ms": {"cbic": st["ms_cbic"], "accept": st["ms_accept"], "prune": st["ms_prune"], "gram": st["ms_gram"]},
            "fp64_peak_tflops_measured": fp64}


def measure_score_file(pkg, wl, tmpdir):
    """the other half of BASELINE.json's metric: wall time of `score` from a CSV on disk to a finished .pss.  (a) configs[0]
    hepatitis as the reference runs it; (b) configs[3] itself written as a 120 MB CSV, with its skeleton, -p 12, --prune (one worker
    thread: in a one-shot process several contexts on one GPU only multiply the first-use allocations, measured 0.53 s of scoring
    with -t 1 against 1.45 s with -t 4).  Times are the binary's own phase clocks plus the wall time of the
    whole process (CUDA context creation included)."""
    import re
    exe = os.path.join(ROOT, "urlearning-cpp_b200", "score")
    out = {}

    def run(tag, args, pss):
        t0 = time.perf_counter()
        r = subprocess.run([exe] + args + [pss, "--quiet"], capture_output=True, text=True)
        wall = time.perf_counter() - t0
        if r.returncode != 0:
            out[tag] = {"error": r.stderr[-300:]}
            return
        m = re.search(r"Scored (\d+) parent sets in ([\d.]+) s .*; parse ([\d.]+) s, init ([\d.]+) s, write ([\d.]+) s, total ([\d.]+) s wall", r.stdout)
        out[tag] = {"process_wall_s": wall, "sets_scored": int(m.group(1)), "score_s": float(m.group(2)), "parse_csv_s": float(m.group(3)),
                    "cuda_init_and_upload_s": float(m.group(4)), "write_pss_s": float(m.group(5)), "total_s": float(m.group(6)), "pss_bytes": os.path.getsize(pss), "args": " ".join(a if not a.startswith(tmpdir) else os.path.basename(a) for a in args)}

    hep = os.path.join(ROOT, "tests", "data", "hepatitis.clean.csv")
    run("configs[0] hepatitis -s -f BIC", [hep, "-s", "-f", "BIC"], os.path.join(tmpdir, "hep.pss"))
    csv, skel = os.path.join(tmpdir, "cfg3.csv"), os.path.join(tmpdir, "cfg3_skel.csv")
    fast_write_csv(csv, wl["codes"])
    pkg.datagen.write_skeleton_matrix(skel, wl["edges"], wl["p"])
    run("configs[3] p=60 n=1e6 -k skeleton -p 12 --prune", [csv, "-k", skel, "-f", "BIC", "-p", "12", "--prune"], os.path.join(tmpdir, "cfg3.pss"))
    out["csv_bytes"] = os.path.getsize(csv)
    for f in ("hep.pss", "cfg3.pss", "cfg3.csv", "cfg3_skel.csv"):
        try:
            os.remove(os.path.join(tmpdir, f))
        except OSError:
            pass
    return out


# ---------------------------------------------------------------------------------------------- config 5 (optional workload)

def degree_bounded_dag(p, seed, max_degree=16, max_indegree=8):
    """random DAG over a random topological order whose undirected skeleton has degree <= max_degree everywhere (BASELINE
    configs[4]: "skeleton degree <= 16"): node i draws up to max_indegree parents among its predecessors that still have
    room.  Non-local, so 2-hop neighbourhoods cover a large part of the network.  -> (order, parents, weights, edges)"""
    rng = np.random.default_rng(seed)
    order = rng.permutation(p)
    deg = np.zeros(p, dtype=np.int64)
    parents, weights = [[] for _ in range(p)], [[] for _ in range(p)]
    for pos, v in enumerate(order):
        want = int(rng.integers(1, max_indegree + 1))
        pool = [int(u) for u in order[:pos] if deg[u] < max_degree]
        k = min(want, len(pool), max_degree - int(deg[v]))
        if k > 0:
            pa = sorted(int(u) for u in rng.choice(pool, size=k, replace=False))
            parents[v] = pa
            weights[v] = [float(rng.uniform(0.3, 0.9) * rng.choice([-1.0, 1.0])) for _ in pa]
            for u in pa:
                deg[u] += 1
                deg[v] += 1
    edges = [0] * p
    for v in range(p):
        for u in parents[v]:
            edges[v] |= 1 << u
            edges[u] |= 1 << v
    return [int(v) for v in order], parents, weights, edges


def run_gpu_cbic5(args):
    """BASELINE configs[4]: linear-Gaussian p=200, n=1e7, skeleton degree <= 16, cBIC lambda=2, sharded by
    (variable, parent-set range) across the ranks.  A step = (1) row-sharded standardise + FP64 Gram (DMMA), moments and
    Gram partials all-gathered and summed in rank order; (2) every rank scores its contiguous piece of the concatenated
    family index space (urlgpu_score_range: 2-hop candidates, explicit -p 4 — the reference's default p-1 over the 2-hop set
    is astronomically large and p=200 does not fit its 64-bit varset, SURVEY Q3) into an NCCL buffer; (3) one all-to-all
    moves the raw scores to the variables' owners; (4) owners apply acceptance + prune (urlgpu_result_from_scores)."""
    import torch
    pkg = importlib.import_module("urlearning-cpp_b200")
    D = importlib.import_module("urlearning-cpp_b200.distributed")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    p, n_total, K, lam = 200, args.n5, args.k5, 2.0
    n_local = n_total // world
    n_total = n_local * world
    order, parents, weights, edges = degree_bounded_dag(p, 5)
    maxdeg = max(bin(e).count("1") for e in edges)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1000 + rank)     # same DAG and weights on every rank, rank-specific rows; generated on the device
    x = torch.randn((p, n_local), dtype=torch.float64, device="cuda", generator=gen)
    for v in order:
        for u, w in zip(parents[v], weights[v]):
            x[v] += w * x[u]
    nbs = [pkg.two_hop_neighbors(edges, p, v) for v in range(p)]
    cs = [bin(nb & ~(1 << v)).count("1") for v, nb in enumerate(nbs)]
    eng = pkg.Engine(local)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    sizes = [family_size(c, K) for c in cs]
    sets_total = sum(sizes)
    pieces, owner = D.plan_ranges(sizes, world)
    my_total = sum(c for _, _, c in pieces[rank])
    board = None
    if args.exchange == "p2p":
        try:
            board = D.PeerScoreBoard(eng, sizes, owner)
        except D.PeerMemoryUnavailable as ex:     # raised on every rank together
            if rank == 0:
                print("bench: peer memory unavailable (%s): using --exchange nccl" % ex, file=sys.stderr)
    score_buf = torch.empty(max(1, my_total), dtype=torch.float32, device="cuda") if board is None else None
    owned = [v for v in range(p) if owner[v] == rank]

    def allsum(a):
        if world == 1:
            return a
        t = torch.from_numpy(a).cuda()
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        out = parts[0].clone()
        for q in parts[1:]:   # fixed rank order: identical result on every rank and for every run
            out += q
        return out.cpu().numpy()

    stored_box = [0]

    def step(fetch=False):
        eng.shard_begin(x.data_ptr(), n_local, p)
        s1, _ = eng.shard_moments(None)
        mean = allsum(s1) / n_total
        a1, a2 = eng.shard_moments(mean)
        S1, S2 = allsum(a1), allsum(a2)
        dev = np.sqrt((S2 - S1 * S1 / n_total) / (n_total - 1.0))
        eng.shard_finish(mean, dev, n_total)
        g = allsum(eng.gram())
        eng.set_gram(g, n_total)
        if board is not None:
            # the K3 kernels store every piece straight into its owner's score board (peer memory over NVLink); a barrier follows
            for (v, first, count) in pieces[rank]:
                eng.score_range(v, nbs[v], K, pkg.CBIC, first, count, lam=lam, out_device_ptr=board.target(v, first))
            board.fence()
            full = {v: board.target(v) for v in owned}
        else:
            mine, off = {}, 0
            for (v, first, count) in pieces[rank]:
                t = score_buf[off:off + count]
                eng.score_range(v, nbs[v], K, pkg.CBIC, first, count, lam=lam, out_device_ptr=t.data_ptr())
                mine[(v, first, count)] = t
                off += count
            full = {v: t.data_ptr() for v, t in D.exchange_ranges(pieces, owner, sizes, mine, "cuda").items()}
        stored = 0
        prev = None
        for v, ptr in full.items():
            res = eng.result_from_scores(v, nbs[v], K, pkg.CBIC, ptr, n=sizes[v], flags=pkg.PRUNE_DOMINATED).prefetch()
            if prev is not None:
                stored += len(prev.fetch(pinned=True)[1]) if fetch else prev.count()
                prev.free()
            prev = res
        if prev is not None:
            stored += len(prev.fetch(pinned=True)[1]) if fetch else prev.count()
            prev.free()
        stored_box[0] = stored

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    sampler.start()
    eng.reset_stats()
    eng.enable_timing(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    stored = stored_box[0]
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        t = torch.tensor([stored], device="cuda", dtype=torch.int64)
        dist.all_reduce(t)
        stored = int(t.item())
    st = eng.stats()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    eng.enable_timing(False)

    # ---- e2e: the rows start in page-locked HOST memory: every step uploads this rank's n/N rows (H2D inside the timed region)
    # and reads every surviving (mask, score) list of the variables it owns back into the engine's page-locked result buffer
    x_host = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
    x_host.copy_(x)
    torch.cuda.synchronize()

    def e2e_step():
        x.copy_(x_host, non_blocking=True)
        step(fetch=True)

    e2e_step()
    nst = max(1, min(args.steps, 2))
    barrier()
    e0.record(stream)
    for _ in range(nst):
        e2e_step()
    e1.record(stream)
    barrier()
    ems = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ems], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ems = float(t.item())
    words = pkg.mask_words_for(p)
    e2e = {"value": sets_total * nst / (ems / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(p * n_total * 8),
           "d2h_bytes_per_step": int((8 * words + 4) * stored), "steps": nst, "ms_per_step": ems / nst,
           "note": "every surviving cache is read back on its owner rank (%d entries over all ranks); no gather" % stored}
    if rank == 0:
        gram_tf = st["gram_flops"] / (st["ms_gram"] / 1e3) / 1e12 if st["ms_gram"] > 0 else None
        fp64 = eng.probe_fp64()
        k3_rate = my_total * args.steps / (st["ms_cbic"] / 1e3) if st["ms_cbic"] > 0 else None
        line = {"metric": METRIC, "value": sets_total * args.steps / (ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64 -> f32", "data": "synthetic (seeded, generated on the device with torch)",
                "config": {"workload": f"configs[4]: linear-Gaussian p=200 n={n_total} (rows sharded over {world} GPU(s)), random DAG with skeleton degree<="
                                       f"{maxdeg}, 2-hop candidates ({min(cs)}..{max(cs)} per variable), explicit -p {K}, cBIC lambda=2, accept + prune",
                           "sets_per_step": sets_total, "stored_after_prune": stored,
                           "parallelism": f"rows sharded n/{world} for the Gram; scoring sharded by (variable, parent-set range): {world} contiguous pieces of the "
                                          f"concatenated family index space, " + ("every piece scored straight into its owner's memory over NVLink (CUDA IPC peer mapping), one barrier"
                                                                               if board is not None else "one all-to-all of raw scores to the variables' owners") + f", N={world}"},
                "e2e": e2e, "gpu_launches": int(st["launches_total"]), "clocks": sampler.summary(),
                "roofline": {"bound": "fp64", "kernel": "K2 gram_partial_kernel (TMA bulk copies -> shared memory -> DMMA m8n8k4.f64) + fixed-order combine", "achieved": gram_tf,
                             "peak": fp64["dmma"], "unit": "TFLOP/s", "frac": gram_tf / fp64["dmma"] if gram_tf else None, "traffic": None,
                             "peak_source": "measured in this run (urlgpu_probe_fp64: register-resident DMMA m8n8k4.f64 chains); DFMA: %.1f TFLOP/s" % fp64["dfma"],
                             "gram_ms_per_step_rank0": st["ms_gram"] / args.steps, "gram_flops_per_step_rank0": st["gram_flops"] / args.steps,
                             "k3_rank_sets_per_s_rank0": k3_rate,
                             "family_ms": {"moments+standardise": st["ms_standardise"], "gram": st["ms_gram"], "cbic": st["ms_cbic"], "accept": st["ms_accept"],
                                           "prune": st["ms_prune"]}},
                "cpu_baseline": None}
        print(json.dumps(line))
    if board is not None:
        board.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()

# ---------------------------------------------------------------------------------------------- CPU arms

def cpu_sample(wl, budget_s, threads, seed=0):
    """Time the oracle on a bounded sample: sets drawn uniformly from the whole workload's candidate families."""
    import oracle_lib as orc
    rng = np.random.default_rng(seed)
    p = wl["p"]
    fam = np.array([sets_of(wl, v) for v in range(p)], dtype=np.float64)
    t_used, n_done = 0.0, 0
    batch = 4 * threads
    z = None
    if wl["kind"] == "cbic":
        z = orc.standardise(wl["x"])
    while t_used < budget_s:
        v = int(rng.choice(p, p=fam / fam.sum()))
        cand = [i for i in range(p) if i != v and (wl["nbs"][v] >> i) & 1]
        masks = []
        for _ in range(batch):
            # uniform over the family: pick a layer with probability C(c,l)/family, then a uniform l-subset
            from math import comb
            w = np.array([comb(len(cand), l) for l in range(min(len(cand), wl["K"]) + 1)], dtype=np.float64)
            l = int(rng.choice(len(w), p=w / w.sum()))
            masks.append(sum(1 << int(i) for i in rng.choice(cand, size=l, replace=False)) if l else 0)
        t0 = time.perf_counter()
        if wl["kind"] == "bic":
            orc.bic_score_many(wl["codes"], wl["card"], v, np.array(masks, dtype=np.uint64), 0, threads)
        else:
            import concurrent.futures as cf
            with cf.ThreadPoolExecutor(threads) as ex:  # ctypes releases the GIL
                list(ex.map(lambda m: orc.cbic_residual(z, v, int(m), wl["lam"]), masks))
        t_used += time.perf_counter() - t0
        n_done += batch
    return n_done / t_used, n_done, t_used


def cpu_baseline(wl, args):
    threads = os.cpu_count() or 1
    rate, n_done, t_used = cpu_sample(wl, args.cpu_seconds, threads)
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_done} parent sets drawn uniformly from the workload's candidate families, {t_used:.1f} s, "
                      "oracle direct counting / per-set OLS refit (the reference's algorithmic structure), no pruning",
            "why_port": "the reference's own AD-tree code (oracle/_ref) cannot hold this workload: its leaf lists are n-bit sets per node "
                        "(SURVEY Q6; measured 640 sets/s at n=2e4, p=12 and ~1/n beyond), so the faster direct-counting port is the conservative CPU arm"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pkg = importlib.import_module("urlearning-cpp_b200")
    wl = make_bic_workload(pkg, 1) if args.workload == "bic" else make_cbic_workload(pkg)
    threads = os.cpu_count() or 1
    # each step = a bounded sample: the whole run ends within ~1.5 minutes unless --cpu-seconds asks for something else
    per_step = args.cpu_seconds if args.cpu_seconds_given else max(2.0, min(20.0, 90.0 / max(1, args.steps + args.warmup)))
    for i in range(args.warmup):
        cpu_sample(wl, per_step, threads, seed=100 + i)
    done, used = 0, 0.0
    for i in range(args.steps):
        r, n_done, t_used = cpu_sample(wl, per_step, threads, seed=i)
        done += n_done
        used += t_used
    value = done / used
    total_sets = sum(sets_of(wl, v) for v in range(wl["p"]))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": used / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak" if (wl["kind"] == "bic" and args.scaling == "weak") else "strong",
            "vs_baseline": None, "dtype": "int32 counts -> f32" if wl["kind"] == "bic" else "f64 -> f32",
            "data": "synthetic (seeded numpy generator, urlearning-cpp_b200/datagen.py)",
            "config": {"workload": wl["name"], "sets_per_step": total_sets,
                       "note": "each step = a bounded uniform sample of the workload's parent sets on the host cores"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{done} sampled parent sets in {used:.1f} s over {args.steps} steps"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="urlgpu", choices=["urlgpu", "reference"])
    ap.add_argument("--workload", default="bic", choices=["bic", "cbic", "cbic5"])
    ap.add_argument("--threads-per-gpu", type=int, default=4, help="BIC: contexts (streams) per GPU, one host thread each")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="BIC with N > 1 GPUs: weak = N replicas of the configs[3] network in one 60N-variable data set (per-GPU work "
                         "fixed); strong = configs[3] itself split over the ranks")
    ap.add_argument("--n5", type=int, default=10_000_000, help="total rows of the cbic5 workload")
    ap.add_argument("--k5", type=int, default=4, help="explicit parent limit (-p) of the cbic5 workload")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1, e2e arm: how the caches reach rank 0: p2p = written by every GPU straight into rank 0's device memory over "
                         "NVLink (urlgpu_result_fetch_device), nccl = fetched to the host, packed, NCCL gather")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="cbic5: how the raw scores reach their owners: p2p = scored straight into the owner's memory over NVLink "
                         "(CUDA IPC peer mapping, urlgpu_peer_*), nccl = local buffer + one all-to-all")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subrecords", action="store_true", help="skip the cBIC configs[2] and score-file wall-time sub-records of the default line")
    ap.add_argument("--one-pass", action="store_true", help="profiling aid: one warm pass, then one pass on one context inside cudaProfilerStart/Stop; no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, run the step once more, untimed, and write the score caches it reads back (every "
                         "variable's stored parent sets and scores) to DIR/*.npy, at most 64 MB (a seeded sample of rows beyond that); "
                         "bic and cbic, one GPU")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "urlgpu" or args.workload == "cbic5" or args.gpus != 1 or args.one_pass):
        ap.error("--dump-outputs needs --impl urlgpu, --workload bic or cbic, --gpus 1 and no --one-pass")
    args.cpu_seconds_given = any(a == "--cpu-seconds" or a.startswith("--cpu-seconds=") for a in sys.argv[1:])
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "cbic5":
        run_gpu_cbic5(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
