#!/usr/bin/env python
"""bench.py — paired-end reads mapped/sec on a synthetic hg38-scale reference (BASELINE.json configs[1]:
--preset chip, 3 Gbp synthetic reference, 2x50 bp pairs).

A "step" is one pass of the mapping hot path (trim -> minimizers -> index probe -> candidates -> mate
supplement / PE filter -> banded verification -> pairing -> sampling -> traceback -> MAPQ -> record) over
one batch of `--pairs-per-step` synthetic pairs, through the C ABI (include/chromap_b200.h).

  value : pairs/s with the batch already resident in HBM (records stay on the device)
  e2e   : pairs/s through the same call with HOST buffers (pinned), H2D of the reads and D2H of the
          records inside the timed region
  --impl reference : the UNMODIFIED reference binary (oracle/_ref/chromap) on the box's host cores, same
          reference / index / read distribution; each step = one 500 000-pair reference batch, timed by
          the reference's own per-batch "Mapped N read pairs in Xs" lines.

Prints ONE JSON line on rank 0.

  --dump-outputs DIR : after the timed steps, rank 0 writes what the headline (device) leg computed in its last step -- every
          field of the records and every count the call returns -- as DIR/<name>.npy in float64, so that two builds can be
          compared output for output on identical seeded inputs (see dump_outputs()).
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

K_MER, WINDOW = 17, 7
ACGT = b"ACGT"


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md 8(d) config 2), generated on the device with torch (plumbing, not the product)
def gen_reference(torch, dev, total_bp, n_seq, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    seq_len = total_bp // n_seq
    lut = torch.tensor(list(ACGT), dtype=torch.uint8, device=dev)
    ref = torch.empty(seq_len * n_seq, dtype=torch.uint8, device=dev)
    CH = 1 << 28
    for o in range(0, ref.numel(), CH):
        n = min(CH, ref.numel() - o)
        ref[o:o + n] = lut[torch.randint(0, 4, (n,), device=dev, generator=g, dtype=torch.int64)]
    # planted segmental repeats: per sequence one 5 kb segment x 50 copies (odd copies 1 % diverged)
    rep_len, rep_copies = 5000, 50
    if seq_len > 4 * rep_len * rep_copies:
        for s in range(n_seq):
            base = s * seq_len
            seg = lut[torch.randint(0, 4, (rep_len,), device=dev, generator=g)]
            starts = torch.randint(0, seq_len - rep_len, (rep_copies,), device=dev, generator=g)
            for ci in range(rep_copies):
                c = seg.clone()
                if ci % 2 == 1:
                    m = torch.rand(rep_len, device=dev, generator=g) < 0.01
                    c[m] = lut[torch.randint(0, 4, (int(m.sum()),), device=dev, generator=g)]
                st = base + int(starts[ci])
                ref[st:st + rep_len] = c
    # 300 bp family, ~1e5 copies genome-wide at 3 Gbp (exercises the f=500/1000 caps)
    fam_len = 300
    fam_copies = int(1e5 * total_bp / 3e9)
    if fam_copies > 0:
        fam = lut[torch.randint(0, 4, (fam_len,), device=dev, generator=g)]
        sid = torch.randint(0, n_seq, (fam_copies,), device=dev, generator=g)
        st = sid * seq_len + torch.randint(0, seq_len - fam_len, (fam_copies,), device=dev, generator=g)
        st = torch.sort(st).values
        keep = torch.ones_like(st, dtype=torch.bool)
        keep[1:] = (st[1:] - st[:-1]) >= fam_len  # a copy that would overlap its predecessor is dropped: the scatter below writes every base once (deterministic)
        st = st[keep]
        fam_copies = int(st.numel())
        idx = st[:, None] + torch.arange(fam_len, device=dev)[None, :]
        vals = fam[None, :].repeat(fam_copies, 1)
        m = torch.rand(fam_copies, fam_len, device=dev, generator=g) < 0.005
        vals[m] = lut[torch.randint(0, 4, (int(m.sum()),), device=dev, generator=g)]
        ref[idx.reshape(-1)] = vals.reshape(-1)
    # N runs, 0.1 %
    n_runs = int(total_bp * 0.001 / 100)
    if n_runs > 0:
        sid = torch.randint(0, n_seq, (n_runs,), device=dev, generator=g)
        ln = torch.randint(1, 200, (n_runs,), device=dev, generator=g)
        st = sid * seq_len + torch.randint(0, seq_len - 200, (n_runs,), device=dev, generator=g)
        ar = torch.arange(200, device=dev)[None, :]
        idx = (st[:, None] + ar)[ar < ln[:, None]]
        ref[idx] = ord("N")
    offsets = np.arange(n_seq + 1, dtype=np.uint64) * np.uint64(seq_len)
    return ref, offsets, seq_len


def gen_pairs(torch, ref, n_seq, seq_len, n_pairs, read_len, seed, dev):
    """2x read_len pairs: fragment length U[80,500], uniform origin, random strand, 1 % substitutions,
    0.1 % single-base indels, 5 % PCR duplicates (exact fragment copies), 1 % junk pairs."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    sid = torch.randint(0, n_seq, (n_pairs,), device=dev, generator=g)
    fl = torch.randint(80, 501, (n_pairs,), device=dev, generator=g)
    st = torch.randint(0, seq_len - 600, (n_pairs,), device=dev, generator=g)
    strand = torch.randint(0, 2, (n_pairs,), device=dev, generator=g)
    # duplicates copy an earlier fragment of the same batch
    dup = torch.rand(n_pairs, device=dev, generator=g) < 0.05
    src = (torch.rand(n_pairs, device=dev, generator=g) * torch.arange(n_pairs, device=dev)).long()
    sid = torch.where(dup, sid[src], sid); fl = torch.where(dup, fl[src], fl)
    st = torch.where(dup, st[src], st); strand = torch.where(dup, strand[src], strand)
    base = sid * seq_len + st
    ar = torch.arange(read_len, device=dev)[None, :]
    comp = torch.full((256,), ord("N"), dtype=torch.uint8, device=dev)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b

    def indel_index(n):
        # single-base deletion (skip one reference base) or insertion (repeat one index) in 0.1 %*L of reads
        p = torch.randint(1, read_len - 1, (n, 1), device=dev, generator=g)
        kind = torch.rand(n, 1, device=dev, generator=g)
        has = kind < 0.001 * read_len
        dele = kind < 0.0005 * read_len
        shift = torch.where(ar >= p, torch.where(dele, 1, -1), 0)
        return torch.where(has, shift, 0)

    left = ref[(base[:, None] + ar + indel_index(n_pairs))]                       # forward strand, 5' end
    ridx = base[:, None] + fl[:, None] - 1 - ar - indel_index(n_pairs)
    right = comp[ref[ridx].long()]                                                # reverse complement of 3' end
    fwd_first = (strand == 0)[:, None]
    r1 = torch.where(fwd_first, left, right)
    r2 = torch.where(fwd_first, right, left)
    lut = torch.tensor(list(ACGT), dtype=torch.uint8, device=dev)
    for r in (r1, r2):
        m = torch.rand(n_pairs, read_len, device=dev, generator=g) < 0.01
        r[m] = lut[torch.randint(0, 4, (int(m.sum()),), device=dev, generator=g)]
    junk = torch.rand(n_pairs, device=dev, generator=g) < 0.01
    nj = int(junk.sum())
    if nj:
        r1[junk] = lut[torch.randint(0, 4, (nj, read_len), device=dev, generator=g)]
        r2[junk] = lut[torch.randint(0, 4, (nj, read_len), device=dev, generator=g)]
    off = (torch.arange(n_pairs + 1, device=dev, dtype=torch.int64) * read_len).to(torch.int32)
    return r1.contiguous().view(-1), r2.contiguous().view(-1), off


def gen_whitelist(torch, dev, n_wl, n_cells, bc_len, seed):
    """BASELINE config 4: a 737 k-entry whitelist of distinct random 16-mers, reads drawn uniformly from 10 k "cells"."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    keys = torch.unique(torch.randint(0, 1 << (2 * bc_len), (int(n_wl * 1.05),), device=dev, generator=g, dtype=torch.int64))[:n_wl]
    keys = keys[torch.randperm(keys.numel(), device=dev, generator=g)]
    return keys, keys[:n_cells]


def gen_barcodes(torch, cell_keys, n, bc_len, seed, dev):
    """n barcodes (ASCII, bc_len bases each; key = 2 bits per base, first base in the high bits, utils.h:107-126) uniform over
    the cells, 2 % with one substituted base, Phred qualities U[2, 40]."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    key = cell_keys[torch.randint(0, cell_keys.numel(), (n,), device=dev, generator=g)]
    sh = (2 * (bc_len - 1 - torch.arange(bc_len, device=dev)))[None, :]
    codes = (key[:, None] >> sh) & 3
    mut = torch.rand(n, device=dev, generator=g) < 0.02
    pos = torch.randint(0, bc_len, (n,), device=dev, generator=g)
    add = torch.randint(1, 4, (n,), device=dev, generator=g)
    rows = torch.nonzero(mut).squeeze(1)
    codes[rows, pos[rows]] = (codes[rows, pos[rows]] + add[rows]) & 3
    lut = torch.tensor(list(ACGT), dtype=torch.uint8, device=dev)
    seq = lut[codes]
    qual = (torch.randint(2, 41, (n, bc_len), device=dev, generator=g) + 33).to(torch.uint8)
    return seq.contiguous().view(-1), qual.contiguous().view(-1)


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md), read in-process through NVML every
    20 ms (no fork, a few microseconds per read); falls back to one nvidia-smi query per second if NVML is missing.
    (Round 1 forked nvidia-smi every 0.1 s on every rank inside a 0.4 s timed region: the driver's N=8 leg lost 19 %
    to that and to unpinned host threads.)"""
    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.stop_flag = False
        self.sm = []
        self.sm_max = None
        self.reasons = set()
        self.how = "nvml"
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(visible_to_physical(gpu_index))
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            self.how = "nvidia-smi"

    def run(self):
        if self.nv is not None:
            nv = self.nv
            bits = [(name, getattr(nv, attr)) for name, attr in self.REASONS if hasattr(nv, attr)]
            while not self.stop_flag:
                try:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    for name, bit in bits:
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
                time.sleep(0.02)
            return
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(visible_to_physical(self.gpu)), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    r = [x.strip() for x in out.split(",")]
                    self.sm.append(float(r[0])); self.sm_max = float(r[1])
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(name)
            except Exception:
                pass
            for _ in range(10):
                if self.stop_flag:
                    break
                time.sleep(0.1)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unsampled"], "samples": 0, "how": self.how}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(sm), "how": self.how}


def visible_to_physical(i):
    """CUDA device index -> NVML / nvidia-smi index (CUDA_VISIBLE_DEVICES may renumber)."""
    v = os.environ.get("CUDA_VISIBLE_DEVICES")
    if v:
        ids = [x.strip() for x in v.split(",") if x.strip()]
        if i < len(ids) and ids[i].isdigit():
            return int(ids[i])
    return i


def bind_to_gpu_numa(gpu_index):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU (same NUMA node): the map call runs
    up to four launch threads per rank, and at N=8 unpinned threads migrate across sockets."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(visible_to_physical(gpu_index))
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {w * 64 + b for w, x in enumerate(words) for b in range(64) if (int(x) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception as e:  # no NVML / not permitted: run unpinned
        log("NUMA binding skipped:", repr(e))
    return 0


def host_description():
    """CPU model / sockets / NUMA layout of the box (so that reference-arm numbers from different boxes can be compared)."""
    d = {"logical_cpus": os.cpu_count(), "usable_cpus": len(os.sched_getaffinity(0))}
    try:
        out = subprocess.run(["lscpu"], capture_output=True, text=True, timeout=5).stdout
        for line in out.splitlines():
            k, _, v = line.partition(":")
            k = k.strip()
            if k in ("Model name", "Socket(s)", "Core(s) per socket", "Thread(s) per core", "NUMA node(s)", "CPU max MHz", "CPU MHz"):
                d[k.lower().replace("(s)", "s").replace(" ", "_")] = v.strip()
    except Exception:
        pass
    try:
        d["loadavg_1min"] = os.getloadavg()[0]
    except OSError:
        pass
    return d


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------
def setup_world():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def run_ours(a):
    import torch
    import torch.distributed as dist
    import chromap_b200 as cb
    rank, local, world = setup_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n_bound = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    total_bp = int(a.ref_gbp * 1e9)
    t0 = time.time()
    ref, offsets, seq_len = gen_reference(torch, dev, total_bp, a.n_seq, a.seed)
    torch.cuda.synchronize()
    log("rank %d: reference %.2f Gbp in %d sequences generated in %.1fs" % (rank, ref.numel() / 1e9, a.n_seq, time.time() - t0))
    params = cb.make_params(a.preset, max_read_length=max(64, a.read_len + 14))
    m = cb.Mapper(params, device=local)
    m.upload_reference_ptr(ref.data_ptr(), offsets)
    t0 = time.time()
    m.build_index(K_MER, WINDOW)
    info = m.index_info()
    t_index = time.time() - t0
    log("rank %d: index built on device in %.1fs: %s" % (rank, t_index, info))
    n = a.pairs_per_step
    bc_len = 16
    if a.barcodes:
        wl_keys, cell_keys = gen_whitelist(torch, dev, a.whitelist_size, a.cells, bc_len, a.seed + 17)
        # abundance table = the reference's pre-pass over the first barcodes (chromap.cc:492-548): here 2 M synthetic ones
        sb, _ = gen_barcodes(torch, cell_keys, 2000000, bc_len, a.seed + 19, dev)
        sh = (2 * (bc_len - 1 - torch.arange(bc_len, device=dev)))[None, :]
        lutc = torch.zeros(256, dtype=torch.int64, device=dev)
        for i_, ch in enumerate(ACGT):
            lutc[ch] = i_
        skey = (lutc[sb.view(-1, bc_len).long()] << sh).sum(1)
        uk, cnt = torch.unique(skey, return_counts=True)
        pos_ = torch.searchsorted(torch.sort(wl_keys).values, uk)
        wl_sorted = torch.sort(wl_keys).values
        ok_ = (pos_ < wl_sorted.numel()) & (wl_sorted[pos_.clamp(max=wl_sorted.numel() - 1)] == uk)
        counts = torch.zeros(wl_sorted.numel(), dtype=torch.int64, device=dev)
        counts[pos_[ok_]] = cnt[ok_]
        m.upload_barcode_whitelist(wl_sorted.cpu().numpy().astype(np.uint64), counts.cpu().numpy().astype(np.uint32), int(cnt[ok_].sum()), bc_len)
    pool = max(1, min(a.steps + a.warmup, a.pool))
    # weak scaling: every rank maps its own batches (batch b -> rank b mod world, SURVEY.md 8(e))
    dev_batches, host_batches = [], []
    for b in range(pool):
        gb = b * world + rank
        r1, r2, off = gen_pairs(torch, ref, a.n_seq, seq_len, n, a.read_len, a.seed * 1000003 + gb, dev)
        if a.barcodes:
            bq = gen_barcodes(torch, cell_keys, n, bc_len, a.seed * 7000003 + gb, dev)
            dev_batches.append((r1, r2, off) + bq)
            host_batches.append(tuple(t.cpu().pin_memory() for t in (r1, r2, off) + bq))
        else:
            dev_batches.append((r1, r2, off))
            host_batches.append(tuple(t.cpu().pin_memory() for t in (r1, r2, off)))
    torch.cuda.synchronize()
    mb = params.max_num_best_mappings
    out_dev = torch.empty(n * mb * 24, dtype=torch.uint8, device=dev)
    out_host = torch.empty(n * mb * 24, dtype=torch.uint8).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    rec_dtype = cb.PAIRS_RECORD if params.output_format == 5 else cb.PE_RECORD

    def step_device(i, out=None):
        b = dev_batches[i % pool]
        kw = dict(barcodes=b[3], barcode_quals=b[4], bc_len=bc_len) if a.barcodes else {}
        _, st = m.map_batch(b[0], b[2], b[1], b[2], first_read_id=(i * world + rank) * n, on_device=True, n_pairs=n,
                            out=out_dev if out is None else out, out_on_device=True, **kw)
        return st

    def step_host(i):
        b = host_batches[i % pool]
        kw = dict(barcodes=b[3].numpy(), barcode_quals=b[4].numpy(), bc_len=bc_len) if a.barcodes else {}
        _, st = m.map_batch(b[0].numpy(), b[2].numpy().view(np.uint32), b[1].numpy(), b[2].numpy().view(np.uint32),
                            first_read_id=(i * world + rank) * n, out=out_host.numpy().view(rec_dtype), **kw)
        return st

    # legs: "device" and "e2e" are the headline numbers (the library's default concurrency: the call's reference
    # batches run as overlapping lanes); "serial" repeats the device leg with one lane, i.e. every kernel alone on
    # one stream, so that per-kernel CUDA-event times are exclusive -- the roofline and kernel_ms_per_step come from it
    res = {}
    for name, fn, lanes, steps in (("device", step_device, a.lanes, a.steps), ("e2e", step_host, a.lanes, a.steps),
                                   ("serial", step_device, 1, min(a.steps, 10))):
        m.set_lanes(lanes)
        for i in range(a.warmup):
            fn(i)
        sampler = ClockSampler(local)
        barrier()
        sampler.start()
        t0 = time.perf_counter()
        stage = {}
        n_rec = n_map = launches = 0
        counters = {}
        for i in range(steps):
            st = fn(a.warmup + i)
            tm = m.timing()
            for k_, v in tm.items():
                if isinstance(v, list):
                    stage[k_] = [x + y for x, y in zip(stage.get(k_, [0] * len(v)), v)]
                else:
                    stage[k_] = stage.get(k_, 0) + v
            n_rec += st["n_records"]; n_map += st["n_mapped_pairs"]
        barrier()
        dt = time.perf_counter() - t0
        sampler.stop_flag = True
        sampler.join()
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        res[name] = dict(dt=dt, stage=stage, n_rec=n_rec, n_map=n_map, clocks=sampler.summary(), steps=steps)
        if name == "device" and a.dump_outputs:  # the last timed step's records, before the next leg overwrites out_dev
            last = (out_dev[:st["n_records"] * 24].cpu().numpy().view(rec_dtype), st)
    # ---- the one collective of the multi-GPU path (SURVEY.md 8e), outside the timed mapping region: duplicate removal over the
    # records of up to four mapped batches per rank: tuple pack -> ONE ncclAllGather -> radix sort + survivor rule on the GPU
    exchange = None
    if params.remove_pcr_duplicates and params.output_format != 5 and not a.no_exchange and not a.barcodes:  # (bulk records: the barcoded leg keeps its keys on the host)
        try:
            m.set_lanes(a.lanes)
            keep = []
            for i in range(min(4, pool)):
                o = torch.empty(n * mb * 24, dtype=torch.uint8, device=dev)
                st_ = step_device(a.warmup + i, out=o)
                keep.append(o[:st_["n_records"] * 24])
            mine = torch.cat(keep)
            n_loc = mine.numel() // 24
            uid = [m.comm_unique_id() if rank == 0 else None]
            if world > 1:
                dist.broadcast_object_list(uid, src=0)
            m.comm_init(world, rank, uid[0])
            surv = torch.empty_like(mine)
            barrier()
            n_out, xst = m.dedup_exchange(mine, n=n_loc, on_device=True, out=surv)   # warm-up (NCCL connection set-up)
            barrier()
            t0 = time.perf_counter()
            n_out, xst = m.dedup_exchange(mine, n=n_loc, on_device=True, out=surv)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            vals = torch.tensor([xst["pack_ms"], xst["allgather_ms"], xst["resolve_ms"], wall * 1e3], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(vals, op=dist.ReduceOp.MAX)
            pk, ag, rs, wl_ = (float(x) for x in vals.tolist())
            exchange = {"what": "cmx_dedup_exchange over the records of %d mapped batches per rank (outside the timed mapping region)" % len(keep),
                        "records_this_rank": n_loc, "records_global": int(xst["n_global"]), "survivors_this_rank": int(n_out),
                        "tuple_bytes_sent_per_rank": int(xst["bytes_sent"]), "tuple_bytes_received_per_rank": int(xst["bytes_received"]),
                        "pack_ms": round(pk, 3), "allgather_ms": round(ag, 3), "sort_resolve_ms": round(rs, 3), "call_ms": round(wl_, 3),
                        "allgather_GBps_per_rank": round(xst["bytes_received"] / (ag * 1e-3) / 1e9, 1) if ag > 0 else None,
                        "timing": "CUDA events on the exchange stream, max over ranks"}
            # the same step as a range shuffle (cmx_dedup_shuffle): every record travels once to the rank that owns its key
            # range, which runs the single-GPU post-processing on it
            try:
                cap = 2 * n_loc + 4096
                part = torch.empty(cap * 24, dtype=torch.uint8, device=dev)
                barrier()
                n_part, sst = m.dedup_shuffle(mine, n=n_loc, on_device=True, out=part, capacity=cap)   # warm-up
                barrier()
                t0 = time.perf_counter()
                n_part, sst = m.dedup_shuffle(mine, n=n_loc, on_device=True, out=part, capacity=cap)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                vals = torch.tensor([sst["partition_ms"], sst["shuffle_ms"], sst["postprocess_ms"], wall * 1e3, float(sst["n_received"])], device=dev,
                                    dtype=torch.float64)
                tot = torch.tensor([float(n_part)], device=dev, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(vals, op=dist.ReduceOp.MAX)
                    dist.all_reduce(tot, op=dist.ReduceOp.SUM)
                pt, sh, pp, wl2, nr_max = (float(x) for x in vals.tolist())
                exchange["shuffle"] = {"what": "cmx_dedup_shuffle over the same records: sample-sort partition -> grouped ncclSend/ncclRecv -> sort + "
                                               "duplicate rule on the owner of each key range",
                                       "records_out_global": int(tot.item()), "records_received_max_over_ranks": int(nr_max),
                                       "balance_max_over_mean": round(nr_max * world / max(1, int(sst["n_global"])), 3),
                                       "record_bytes_sent_this_rank": int(sst["bytes_sent"]), "record_bytes_received_this_rank": int(sst["bytes_received"]),
                                       "partition_ms": round(pt, 3), "shuffle_ms": round(sh, 3), "postprocess_ms": round(pp, 3), "call_ms": round(wl2, 3),
                                       "shuffle_GBps_per_rank": round(sst["bytes_received"] / (sh * 1e-3) / 1e9, 1) if sh > 0 and sst["bytes_received"] else None}
                del part
            except Exception as ex:
                exchange["shuffle"] = {"unavailable": repr(ex)[:200]}
            m.comm_destroy()
            del keep, mine, surv
        except Exception as ex:  # NCCL missing on the box: report, do not hide
            exchange = {"unavailable": repr(ex)[:200]}
    cpu_baseline = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        if a.barcodes or params.split_alignment:
            cpu_baseline = {"value": None, "unit": "pairs/s", "cores": os.cpu_count() or 1, "kind": "port",
                            "sample": "not timed for this leg (the default chip leg and --impl reference carry the CPU numbers)"}
        else:
            cpu_baseline = cpu_port_baseline(a, m, ref, offsets, seq_len, host_batches[0][:3])
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    dv, ee, sr = res["device"], res["e2e"], res["serial"]
    value = a.steps * n * world / dv["dt"]
    e2e = a.steps * n * world / ee["dt"]
    st = sr["stage"]
    ks = sr["steps"]
    kern = {k_: st[k_] / ks for k_ in ("front_ms", "cluster_ms", "seed_ms", "pair_candidates_ms", "verify_ms", "pairing_ms", "select_ms", "emit_ms")}
    kern["seed_overflow_tiers_ms"] = kern["seed_ms"] - kern["front_ms"] - kern["cluster_ms"]
    top = max((k_ for k_ in kern if k_ != "seed_ms"), key=kern.get)
    peaks, peak_src = measured_peaks()
    # Roofline of the index-probe kernel = the fused front end (seed_front_kernel: read bytes in, length filter, minimizers,
    # table probes, records out).  Algorithmic bytes of one launch, two definitions (DESIGN.md 4):
    #   layout : what OUR table layout needs: 16 B per probed slot + 12 B per minimizer record written + the read bytes +
    #            192 B of per-pair metadata written
    #   survey : SURVEY.md 8(d)'s count for the reference's khash: 12 B per probe step + 8 B per found value (+ the read bytes)
    read_bytes = 2.0 * a.read_len * n
    bytes_layout = (st["n_probe_steps"] * 16 + st["n_minimizers"] * 12) / ks + read_bytes + 192.0 * n
    bytes_survey = (st["n_probe_steps"] * 12 + st["n_found"] * 8) / ks + read_bytes
    fk = kern["front_ms"]
    achieved = bytes_layout / (fk * 1e-3) / 1e9 if fk > 0 else 0.0
    achieved_survey = bytes_survey / (fk * 1e-3) / 1e9 if fk > 0 else 0.0
    traffic = None  # dram bytes + executed warp instructions of one launch from the committed ncu --set full capture of this workload
    warp_inst = None
    tp = os.path.join(ROOT, "profiles", "front_kernel_ncu.json")
    if os.path.exists(tp):
        prof = json.load(open(tp))
        if prof.get("pairs_per_step") == n and abs(prof.get("ref_bp", 0) - int(ref.numel())) < 0.01 * ref.numel() and prof.get("preset") == a.preset:
            traffic = prof.get("dram_bytes_per_launch")
            warp_inst = prof.get("warp_instructions_per_launch")
    issue = None
    if warp_inst and fk > 0:
        sm_clock = (dv["clocks"].get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0) * 1e6
        peak_issue = 148 * 4 * sm_clock  # warp instructions per second: 148 SMs x 4 schedulers x 1 per clock
        issue = {"warp_instructions_per_launch": warp_inst, "achieved_per_s": warp_inst / (fk * 1e-3), "peak_per_s": peak_issue,
                 "frac": warp_inst / (fk * 1e-3) / peak_issue, "note": "the kernel is integer-issue bound (3 x Hash64 per k-mer), not HBM bound"}
    cells = (st["n_verified"] / ks) * a.read_len * (2 * params.error_threshold + 1)
    line = {
        "metric": "paired-end reads mapped/sec (hg38-scale, 2x50bp)", "value": value, "unit": "pairs/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": dv["dt"] / a.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "--preset %s%s, synthetic %.2f Gbp reference (%d seqs, planted repeats, N runs), 2x%d bp PE pairs, %d pairs/step/GPU"
                               % (a.preset, " + 16 bp cell barcodes (%d-entry whitelist)" % a.whitelist_size if a.barcodes else "", ref.numel() / 1e9, a.n_seq, a.read_len, n),
                   "preset": a.preset, "k": K_MER, "w": WINDOW, "pairs_per_step": n, "ref_bp": int(ref.numel()),
                   "index": {"keys": info["n_keys"], "occurrences": info["n_occ"], "table_slots": info["table_slots"], "build_s": round(t_index, 2)},
                   "l2": "inputs (%.0f MB reads/step) and the %.1f GB index exceed L2; distinct batches cycle through a pool of %d"
                         % (2 * a.read_len * n / 1e6, info["table_slots"] * 16 / 1e9, pool),
                   "sharding": "batch b -> rank b mod N, index+reference replicated per GPU, no data-path collective in the timed region",
                   "host": dict(host_description(), cpus_bound_to_gpu_numa_node=n_bound)},
        "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": int(2 * a.read_len * n + 8 * (n + 1) + (2 * bc_len * n if a.barcodes else 0)),
                "d2h_bytes_per_step": int(24 * ee["n_rec"] / a.steps), "ms_per_step": ee["dt"] / a.steps * 1e3},
        "gpu_launches": int(dv["stage"]["n_launches"]),
        "clocks": dv["clocks"], "clocks_e2e": ee["clocks"],
        "kernel_ms_per_step": {k_: round(v, 3) for k_, v in kern.items()},
        "kernel_ms_per_step_note": "one-lane pass: exclusive CUDA-event times of the stages, sum = %.2f ms/step" % (sr["dt"] / ks * 1e3),
        "lanes": a.lanes,
        "mapped_fraction": dv["n_map"] / (a.steps * n),
        "tier_pairs_per_step": [x / ks for x in st["tier_pairs"]],
        "roofline": {"kernel": "seed_front_kernel (index probe fused with length filter + minimizers, reads staged by cp.async.bulk)", "bound": "hbm",
                     "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                     "peak_source": peak_src, "traffic": traffic, "algorithmic_bytes_per_launch": bytes_layout,
                     "achieved_survey_8d": achieved_survey, "frac_survey_8d": achieved_survey / peaks["hbm_gbs"], "algorithmic_bytes_survey_8d": bytes_survey,
                     "kernel_ms": fk, "kernel_share_of_step": fk / (sr["dt"] / ks * 1e3), "top_stage": top, "issue": issue,
                     "timed": "%d steps with one lane (every kernel alone on one stream, %.2f ms/step); the headline legs run %d overlapping lanes" % (ks, sr["dt"] / ks * 1e3, a.lanes),
                     "probe_steps_per_pair": st["n_probe_steps"] / (ks * n), "minimizers_per_pair": st["n_minimizers"] / (ks * n),
                     "verified_candidates_per_pair": st["n_verified"] / (ks * n),
                     "cell_updates_per_s": cells / (kern["verify_ms"] * 1e-3) if kern["verify_ms"] > 0 else None},
    }
    if exchange is not None:
        line["dedup_exchange"] = exchange
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, *last)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(d, recs, stats):
    """One float64 .npy per record field and one per count of `stats`, all together under DUMP_BYTES: a larger output is reduced
    to a sample of its records drawn with a fixed seed; sample_index.npy holds the sampled positions (all of them when nothing
    was dropped)."""
    os.makedirs(d, exist_ok=True)
    n = len(recs)
    cap = (DUMP_BYTES - (64 << 10)) // (8 * (len(recs.dtype.names) + 1))  # 64 KB left for the counts and the .npy headers
    idx = np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
    np.save(os.path.join(d, "sample_index.npy"), idx.astype(np.float64))
    for f in recs.dtype.names:
        np.save(os.path.join(d, f + ".npy"), recs[f][idx].astype(np.float64))
    for k, v in stats.items():
        np.save(os.path.join(d, k + ".npy"), np.array([v], dtype=np.float64))
    log("outputs of the last timed step (%d of %d records) written to %s" % (len(idx), n, d))


def cpu_port_baseline(a, m, ref, offsets, seq_len, host_batch):
    """The CPU oracle (a port, oracle/) on a bounded sample of the same workload, all host cores."""
    from oracle import oracle_py as orc
    import psutil
    cores = os.cpu_count() or 1
    need = m.index_info()["n_keys"] * 2 * 16 * 2.2 + ref.numel() * 2
    if psutil.virtual_memory().available < need:
        log("cpu_baseline skipped: not enough host RAM for a second copy of the index")
        return None
    t0 = time.time()
    idx = m.download_index()
    oidx = orc.Index(arrays=idx, k=K_MER, w=WINDOW)
    del idx
    href = ref.cpu().numpy()
    oref = orc.Reference(seqs=[href[int(offsets[i]):int(offsets[i + 1])] for i in range(len(offsets) - 1)])
    log("cpu_baseline: index + reference copied to the host in %.1fs" % (time.time() - t0))
    r1, r2, off = (t.numpy() for t in host_batch)
    n = min(len(off) - 1, a.cpu_sample_pairs)
    L = a.read_len
    p = orc.make_params(a.preset)
    s1, s2, o = r1[:n * L], r2[:n * L], off[:n + 1].view(np.uint32)
    orc.map_pairs(p, oidx, oref, s1[:20000 * L], o[:20001], s2[:20000 * L], o[:20001], n_threads=cores)  # warm-up
    t0 = time.perf_counter()
    recs, _ = orc.map_pairs(p, oidx, oref, s1, o, s2, o, n_threads=cores)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": "%d pairs of step 0 through oracle/ (CPU restatement, OpenMP over taskloop chunks), same index arrays" % n}


# ------------------------------------------------------------------------------------------------------
def run_reference(a):
    """The unmodified reference binary on the host cores.  Needs a GPU only to synthesise the same data and
    to build the (identical-lookup) index in seconds; chromap itself runs on the CPU, untouched."""
    rank, local, world = setup_world()
    if rank != 0:
        return
    binp = os.path.join(ROOT, "oracle", "_ref", "chromap")
    if not os.path.exists(binp):
        emit({"impl": "reference", "unavailable": "oracle/_ref/chromap not built (needs /root/reference at build time)"})
        return
    import torch
    import chromap_b200 as cb
    dev = torch.device("cuda", local)
    torch.cuda.set_device(local)
    total_bp = int(a.ref_gbp * 1e9)
    ref, offsets, seq_len = gen_reference(torch, dev, total_bp, a.n_seq, a.seed)
    m = cb.Mapper(cb.make_params(a.preset, max_read_length=max(64, a.read_len + 14)), device=local)
    m.upload_reference_ptr(ref.data_ptr(), offsets)
    m.build_index(K_MER, WINDOW)
    work = a.workdir or ("/dev/shm/chromap_b200_bench" if os.path.isdir("/dev/shm") else "/tmp/chromap_b200_bench")
    os.makedirs(work, exist_ok=True)
    t0 = time.time()
    href = ref.cpu().numpy()
    with open(os.path.join(work, "ref.fa"), "wb") as f:
        for i in range(a.n_seq):
            f.write(b">chr%d\n" % (i + 1))
            href[int(offsets[i]):int(offsets[i + 1])].tofile(f)
            f.write(b"\n")
    # The index the reference binary loads.  Default: the device-built index written in the reference's file format (seconds);
    # tests/test_gpu_parity.py::test_device_built_index_has_the_content_of_the_reference_binarys_index shows that it holds
    # exactly what `chromap -i` builds (same occurrence table byte for byte, same key -> value map, same bucket count).
    # --reference-index chromap lets the reference binary build it itself (minutes at 3 Gbp, single-threaded).
    index_by = a.reference_index
    if index_by == "chromap":
        pr = subprocess.run([binp, "-i", "-r", os.path.join(work, "ref.fa"), "-o", os.path.join(work, "ref.index")], capture_output=True, text=True)
        if pr.returncode != 0:
            emit({"impl": "reference", "unavailable": "chromap -i failed: " + pr.stderr[-200:].replace("\n", " | ")})
            return
    else:
        idx = m.download_index()
        with open(os.path.join(work, "ref.index"), "wb") as f:  # index.cc:91-130 / khash.h:374-386 layout
            np.array([K_MER, WINDOW], dtype=np.int32).tofile(f)
            np.array([idx["n_keys"], idx["n_buckets"], idx["n_keys"], idx["n_keys"], int(idx["n_buckets"] * 0.77 + 0.5)], dtype=np.uint32).tofile(f)
            idx["flags"].tofile(f); idx["keys"].tofile(f); idx["vals"].tofile(f)
            np.array([len(idx["occ"])], dtype=np.uint32).tofile(f)
            idx["occ"].tofile(f)
        del idx
    n_batches = a.warmup + a.steps
    n = 500000  # one reference batch (chromap.h:182) per step
    L = a.read_len
    for which in (0, 1):
        with open(os.path.join(work, "read%d.fq" % (which + 1)), "wb") as f:
            for b in range(n_batches):
                r = gen_pairs(torch, ref, a.n_seq, seq_len, n, L, a.seed * 1000003 + b, dev)[which].cpu().numpy().reshape(n, L)
                rec = np.empty((n, 2 * L + 16), dtype=np.uint8)  # "@" + 9-digit id + "\n" + seq + "\n+\n" + qual + "\n"
                ids = np.char.zfill((np.arange(n) + b * n).astype(str), 9).astype("S9")
                rec[:, 0] = ord("@"); rec[:, 1:10] = np.frombuffer(ids.tobytes(), dtype=np.uint8).reshape(n, 9)
                rec[:, 10] = 10; rec[:, 11:11 + L] = r; rec[:, 11 + L] = 10; rec[:, 12 + L] = ord("+"); rec[:, 13 + L] = 10
                rec[:, 14 + L:14 + 2 * L] = ord("I"); rec[:, 14 + 2 * L] = 10
                rec[:, :15 + 2 * L].tofile(f)
    del ref, m
    torch.cuda.empty_cache()
    log("reference arm: inputs written to %s in %.1fs" % (work, time.time() - t0))
    cores = os.cpu_count() or 1
    cmd = [binp, "--preset", a.preset, "-x", os.path.join(work, "ref.index"), "-r", os.path.join(work, "ref.fa"),
           "-1", os.path.join(work, "read1.fq"), "-2", os.path.join(work, "read2.fq"), "-o", os.path.join(work, "out.bed"), "-t", str(cores)]
    t0 = time.time()
    pr = subprocess.run(cmd, capture_output=True, text=True)
    wall = time.time() - t0
    per_batch = []
    for line in pr.stderr.splitlines():
        if line.startswith("Mapped ") and "read pairs in" in line:
            per_batch.append(float(line.split(" in ")[1].rstrip("s.")))
    for f in ("ref.index", "ref.fa", "read1.fq", "read2.fq", "out.bed"):
        try:
            os.remove(os.path.join(work, f))
        except OSError:
            pass
    if pr.returncode != 0 or len(per_batch) < n_batches:
        emit({"impl": "reference", "unavailable": "reference run failed rc=%d: %s" % (pr.returncode, pr.stderr[-300:].replace("\n", " | "))})
        return
    timed = per_batch[a.warmup:a.warmup + a.steps]
    dt = sum(timed)
    v = a.steps * n / dt
    line = {"impl": "reference", "metric": "paired-end reads mapped/sec (hg38-scale, 2x50bp)", "value": v, "unit": "pairs/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": "--preset %s, synthetic %.2f Gbp reference (%d seqs), 2x%d bp PE pairs; reference chromap 0.3.3 -t %d, step = one 500000-pair batch (its own per-batch timer)"
                                   % (a.preset, total_bp / 1e9, a.n_seq, L, cores), "total_wall_s": round(wall, 1),
                       "index_built_by": "chromap -i (the reference binary)" if index_by == "chromap" else
                                         "cmx_build_index + cmx_download_index, reference file format (content == chromap -i, tests/test_gpu_parity.py)",
                       "per_batch_s": [round(x, 3) for x in timed], "host": host_description()},
            "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cores, "kind": "reference",
                             "sample": "%d batches of 500000 pairs, reference binary 'Mapped N read pairs in Xs' lines" % a.steps},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else any library prints (NCCL's version banner,
    torchrun notices) was redirected to stderr at start-up."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preset", default="chip")
    ap.add_argument("--ref-gbp", type=float, default=3.0)
    ap.add_argument("--n-seq", type=int, default=24)
    ap.add_argument("--read-len", type=int, default=50)
    ap.add_argument("--pairs-per-step", type=int, default=2000000)
    ap.add_argument("--pool", type=int, default=6)
    ap.add_argument("--lanes", type=int, default=4, help="overlapping lanes per call in the headline legs (cmx_set_lanes)")
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--cpu-sample-pairs", type=int, default=1000000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-exchange", action="store_true", help="skip the duplicate-removal exchange leg")
    ap.add_argument("--barcodes", action="store_true", help="scATAC leg (BASELINE config 4): 16 bp cell barcodes + whitelist correction")
    ap.add_argument("--whitelist-size", type=int, default=737000)
    ap.add_argument("--cells", type=int, default=10000)
    ap.add_argument("--workdir", default=None)
    ap.add_argument("--reference-index", default="ours", choices=["ours", "chromap"], help="--impl reference: who builds the index the reference binary loads")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's records and counts to DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if a.warmup < 3:
        a.warmup = 3
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
