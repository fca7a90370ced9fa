#!/usr/bin/env python
"""bench.py - SNP-pair observations/s into the Hansel matrix (+ haplotype recovery seconds).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
  python bench.py --impl reference ...                      (the reference's CPU way, timed on host cores)

Workload = BASELINE.json configs[2]: synthetic metagenomic gene region, 10k SNPs,
10M x 150 bp reads (the configuration the 1/2/4/8-GPU metric is quoted on; it fits one
GPU).  A "step" is one complete ingestion of the batch: zero the counts, pair-expand
every read into the banded matrix, and (N>1) sum the partial matrices with an NCCL
integer all-reduce.  Weak scaling: every rank ingests its own 10M-read shard of the
same metagenome (different reads, same strains/sites).

`value`   : observations/s with the packed reads already resident in HBM.
`e2e`     : the same metric from the north_star boundary: the packed (rank, off, codes) arrays in pinned HOST
            memory go through the public call (Hansel.ingest_packed -> hx_ingest_host), which
            copies them in a few chunks (each expanded while the next is in flight), folds into the working matrix
            and returns the totals - a new matrix every step.  `e2e.other_paths`: the dense wire format with the
            host-side encoder inside the clock, and with the chunks encoded before the clock (device-side limit).
`e2e_bam` : a synthetic coordinate-sorted BAM of the same reads (bounded sample) through util.load_from_bam:
            reads/s with the per-stage seconds (file read, inflate, record scan, depth cap, CIGAR walks, gather,
            GPU ingestion).

--dump-outputs DIR writes what the last timed step computed (see dump_outputs) as .npy files, so that two builds
can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: the bench leaves it as the build left it

import numpy as np  # noqa: E402

from gretel_b200 import synth  # noqa: E402

METRIC = "snp_pair_observations_per_sec"
UNIT = "obs/s"
DUMP_BYTES = 64 << 20                   # --dump-outputs: budget of all files together


def b_obs(k_mean):
    """Algorithmic bytes per observation, SURVEY.md section 8(d): one uint32 counter
    read-modify-write plus the read's amortised input."""
    return 8.0 + (k_mean + 12.0) / (k_mean * (k_mean - 1.0) / 2.0)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed regions (NVML, ~1 kHz)."""
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
            "hw_power_brake": 0x80}

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        self._on = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            if self._on.is_set():
                try:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    for name, bit in self.BITS.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:  # noqa: BLE001
                    pass
            time.sleep(0.001)

    def start(self):
        if self.nv is None:
            return
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()

    def region(self, on):
        (self._on.set if on else self._on.clear)()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self._stop.set()
        self._t.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def gdist_bounds(off, world):
    from gretel_b200 import dist as gdist
    return gdist.shard_bounds(off, world)


def workload_config(args, k_mean=None, n_reads=None):
    w = synth.WORKLOADS[args.workload]
    cfg = {"workload": "BASELINE.json configs[%d] %s: %d SNPs, %d x %s reads per GPU%s" % (
        w.config, w.name, w.n_snps, args.reads or w.n_reads,
        ("~%d bp ONT-like" % w.read_len) if w.long_reads else ("%d bp" % w.read_len),
        "" if not args.reads or args.reads == w.n_reads else " (reduced by --reads)"),
        "n_snps": w.n_snps, "reads_per_gpu": args.reads or w.n_reads, "seed": 20260000 + w.config + 1,
        "l2_policy": "inputs larger than L2 (packed reads are streamed once per step)"}
    if k_mean is not None:
        cfg["mean_snps_per_read"] = round(k_mean, 3)
    if n_reads is not None:
        cfg["reads_with_2plus_snps"] = int(n_reads)
    return cfg


# ----------------------------------------------------------------------------------- reference arm
def lumma_floor(rank, off, kernel_ms):
    """Tensor-core floor of the long-read kernel (ingest_lumma.cu): the reads sorted by (first 16-site block, blocks
    spanned) and cut into chunks of 32 per first block exactly as k_l2_scatter / k_l2_onehot do; a chunk spanning n
    blocks takes n(n+1)/2 MMAs of M=128, N=128, K=32 (int8, 64 cycles each at the 8192 MAC/clk/SM peak)."""
    k = np.diff(off)
    ok = k >= 2
    r, k = rank[ok].astype(np.int64), k[ok]
    if not len(r):
        return None
    sb, eb = (r + 1) >> 4, (r + k) >> 4
    order = np.lexsort((eb, sb))
    sb, eb = sb[order], eb[order]
    first = np.concatenate([[0], np.flatnonzero(np.diff(sb)) + 1])                 # start of every first block's reads
    within = np.arange(len(sb)) - np.repeat(first, np.diff(np.concatenate([first, [len(sb)]])))
    chunk_start = np.flatnonzero(within % 32 == 0)
    n = np.maximum.reduceat(eb, chunk_start) - sb[chunk_start] + 1
    mma = float((n * (n + 1) // 2).sum())
    floor_ms = mma * 64 / 148 / 1.965e6
    return {"mma_per_launch": mma, "cycles_per_mma": 64, "floor_ms": floor_ms, "frac": floor_ms / kernel_ms,
            "chunks": int(len(chunk_start)), "operand_slabs": int(n.sum()),
            "note": "one M=128,N=128,K=32 int8 MMA per (chunk of 32 reads, 16 first sites, 16 second sites) at the 8192 "
                    "MAC/clk/SM peak; measured in the kernel: ~140 cycles per MMA, because an MMA of this shape reads "
                    "8 KB of operands from shared memory (the whole 128 B/clk) while TMA refills 6 KB per MMA"}


def popc_floor(rank, off, kernel_ms):
    """The compute floor of the bit-sliced kernel: 16 POPC per (site pair x group of 32 same-rank reads), issued
    by whole warps over the t2-major pair prefix, on the quarter-rate XU pipe (15.5 lanes/clk/SM measured,
    profiles/r1_microbench.txt).  Returned beside the HBM figures: it is the hardware bound this kernel is
    closest to, and the kernel is still several times above it (issue slots / phase barriers, DESIGN.md 4)."""
    k = np.diff(off).astype(np.int64)
    R = len(rank)
    if R == 0:
        return None
    start = np.flatnonzero(np.r_[True, rank[1:] != rank[:-1]])
    pos = np.arange(R) - np.repeat(start, np.diff(np.r_[start, R]))
    gid = np.cumsum(np.r_[True, pos[1:] % 32 == 0]) - 1
    kg = np.zeros(int(gid[-1]) + 1, np.int64)
    np.maximum.at(kg, gid, k)
    lane_ops = int((16 * ((kg * (kg - 1) // 2 + 31) // 32) * 32).sum())
    lanes_per_clk_sm, sms, mhz = 15.5, 148, 1965.0
    floor_ms = lane_ops / (lanes_per_clk_sm * sms * mhz * 1e6) * 1e3
    return {"pipe": "xu (POPC)", "lane_ops_per_launch": lane_ops, "peak_lanes_per_clk_per_sm": lanes_per_clk_sm,
            "floor_ms": floor_ms, "frac": floor_ms / kernel_ms}


def run_reference(args):
    """The reference's own CPU implementation of the path (per-pair Python calls into a NumPy
    array, forked workers over read chunks: gretel/util.py:242-286, 294-326), restated in
    oracle/py_baseline.py because hanselx/pysam are not installable here."""
    rank_env = int(os.environ.get("RANK", "0"))
    if rank_env != 0:
        return 0
    from oracle import py_baseline as pb
    cores = os.cpu_count() or 1
    w = synth.WORKLOADS[args.workload]
    # bounded sample: about 3 s of work per step on all cores (~1 M obs/s/core)
    sample_reads = args.ref_sample or int(min(w.n_reads, 2_000_000, max(2000, 30_000 * cores)))
    d = synth.generate(synth.scaled(w, sample_reads))
    k = np.diff(d["off"])
    W = d["max_k"] - 1
    times, crumbs = [], 0
    for it in range(args.warmup + args.steps):
        crumbs, dt = pb.timed_ingest(d["rank"], d["off"], d["codes"], w.n_snps, W, n_procs=cores)
        if it >= args.warmup:
            times.append(dt)
    total_t = float(sum(times))
    value = crumbs * len(times) / total_t
    sample = "%d of %d reads (%d observations) of the same workload, %d forked workers" % (
        len(k), w.n_reads, crumbs, cores)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic", "config": workload_config(args, float(k.mean()), len(k)),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def recovery_cpu_baseline(device):
    """One haplotype on BASELINE.json configs[1] (HIV-like, ~1k SNPs) recovered by the literal Python
    restatement of gretel.py:102-189 + :79-98 over a dense Hansel (the reference's way: one Python call per
    branch / per pair), next to the same haplotype on the GPU.  The dense matrix is taken from the GPU
    ingestion so that the CPU side only pays for recovery."""
    from gretel_b200 import util
    from oracle import hansel_oracle as o
    w = synth.scaled(synth.WORKLOADS["hiv"], 20_000)
    d = synth.generate(w)
    N = w.n_snps
    h = util.load_from_packed(d["rank"], d["off"], d["codes"], N, band_w=d["max_k"] - 1, device=device)
    ho = o.OracleHansel.init_matrix(o.SYMBOLS, o.UNSYMBOLS, N)
    ho.m[...] = h.to_dense()
    ho.L = h.L
    horig = ho.copy()
    t0 = time.perf_counter()
    path, prob, mn = o.generate_path(N, ho, horig)
    t_gen = time.perf_counter() - t0
    t_rw = None
    if path is not None:
        t0 = time.perf_counter()
        o.reweight_hansel_from_path(ho, path, max(mn, 0.01))
        t_rw = time.perf_counter() - t0
    orig = h.copy()
    t0 = time.perf_counter()
    res = h.generate_path_codes(orig)
    if res[0] is not None:
        h.reweight_path_codes(res[0], max(res[3], 0.01))
    t_gpu = time.perf_counter() - t0
    same = (path is None and res[0] is None) or (path is not None and res[0] is not None and
                                                  [o.CODE[x] for x in path] == list(res[0]))
    return {"workload": "configs[1] hiv: %d SNPs, 20000 reads, L=%d" % (N, h.L), "cores": 1, "kind": "port",
            "generate_path_s": t_gen, "reweight_s": t_rw, "gpu_generate_plus_reweight_s": t_gpu,
            "same_haplotype": bool(same)}


# ----------------------------------------------------------------------------------- our arm
def dump_outputs(out_dir, h, N, W):
    """What the last timed step left in ``h``, as the caller of the ingestion receives it: ``totals.npy`` (slices,
    crumbs, covered SNPs, sentinel increments) and ``band.npy``, the step's counts as the float32 band [N+2][W][7][7]
    that Hansel.band() returns once they are folded into an empty matrix.  The counts are copied without folding
    them, so the rest of the run is unchanged.  A band over the budget keeps a fixed, seeded sample of its rows;
    ``band_rows.npy`` lists the rows kept."""
    import torch
    from gretel_b200 import dist as gdist
    totals = np.array(h.ingest_totals(), dtype=np.float64)
    cptr, cn, _, _ = h.counts_buffer()
    assert cn == (N + 2) * W * 49, "pending counts do not have the band's shape"
    cnt = torch.as_tensor(gdist._DevBuf(cptr, cn, "<i4"), device=torch.device("cuda", h.device)).cpu().numpy()
    cnt = cnt.view(np.uint32).reshape(N + 2, W, 7, 7)
    rows = np.arange(N + 2)
    fit = (DUMP_BYTES - (1 << 20)) // (W * 49 * 4)      # 1 MB left for the row list, the totals and the headers
    if fit < N + 2:
        rows = np.sort(np.random.default_rng(20260000).choice(N + 2, size=fit, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "band.npy"), cnt[rows].astype(np.float32))
    np.save(os.path.join(out_dir, "band_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "totals.npy"), totals)


def measure_other_config(name, args, device):
    """One more BASELINE.json ingestion config on this GPU: inputs resident, K steps of clear + pair expansion timed with
    CUDA events on the library's stream, then the independent per-row recount (as parity_probe)."""
    import torch
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    w = synth.WORKLOADS[name]
    d = synth.generate(w)
    N, W, R = w.n_snps, d["max_k"] - 1, len(d["rank"])
    dev = torch.device("cuda", device)
    t_rank, t_off, t_codes = (torch.from_numpy(d[k_]).to(dev) for k_ in ("rank", "off", "codes"))
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W, device=device)
    h.counts_buffer()
    stream = torch.cuda.ExternalStream(h.stream, device=dev)

    def step():
        h.reset_counts()
        h.ingest_device(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with torch.cuda.stream(stream):
        for a, b in ev:
            a.record(stream)
            step()
            b.record(stream)
    torch.cuda.synchronize()
    ms = float(sum(a.elapsed_time(b) for a, b in ev)) / args.steps
    kms = []
    for _ in range(3):
        step()
        h.ingest_totals()
        kms.append(h.kernel_ms("ingest"))
    rows_exp = torch.zeros(N + 2, dtype=torch.int64, device=dev)
    rows_got = torch.zeros(N + 2, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    h.probe_expected_rows(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R, rows_exp.data_ptr())
    h.counts_row_sums(rows_got.data_ptr())
    h.sync()
    pt = h.ingest_totals()
    ok = bool(torch.equal(rows_exp, rows_got)) and int(rows_got.sum().item()) == int(pt[1]) + int(pt[3])
    out = {"workload": workload_config(argparse.Namespace(workload=name, reads=0), float(np.diff(d["off"]).mean()), R)["workload"],
           "value": pt[1] / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "kernel_ms": float(np.mean(kms)),
           "observations_per_step": int(pt[1]), "reads": R, "band_w": W, "steps": args.steps, "parity_probe_ok": ok,
           "inputs": "resident in HBM; every step clears the counts and runs the whole ingestion"}
    if d["max_k"] > 52:
        out["tensor_floor"] = lumma_floor(d["rank"], d["off"], float(np.mean(kms)))
    h.close()
    return out


def run_ours(args):
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun (one process per GPU)" % args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    overlap = world > 1 and args.overlap_steps and args.exchange in ("allreduce", "auto") and args.scaling == "weak" and args.segments <= 1
    if world > 1:
        import torch.distributed as dist
        if overlap:
            os.environ.setdefault("NCCL_MAX_CTAS", str(args.comm_sms))   # the collective shares the GPU with the next step's kernel
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from gretel_b200 import dist as gdist, util
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS

    w = synth.WORKLOADS[args.workload]
    if args.reads:
        w = synth.scaled(w, args.reads)
    t0 = time.time()
    strong = args.scaling == "strong" and world > 1
    if strong:
        # BASELINE.json configs[2] as named: ONE read set, cut into contiguous chunks of the rank-sorted reads
        # balanced by pair count; every rank generates the same reads and keeps its chunk
        full = synth.generate(w, shard=0)
        bnd = gdist_bounds(full["off"], world)
        lo_r, hi_r = int(bnd[rank]), int(bnd[rank + 1])
        o0 = int(full["off"][lo_r])
        d = dict(full)
        d["rank"] = full["rank"][lo_r:hi_r].copy()
        d["off"] = (full["off"][lo_r:hi_r + 1] - o0).copy()
        d["codes"] = full["codes"][o0:int(full["off"][hi_r])].copy()
        del full
    else:
        d = synth.generate(w, shard=rank)
    gen_s = time.time() - t0
    N = w.n_snps
    k = np.diff(d["off"])
    R = len(k)
    # band width must agree on every rank
    W = d["max_k"] - 1
    if world > 1:
        tw = torch.tensor([W], device="cuda")
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        W = int(tw.item())
    n_obs_local = None

    # device-resident inputs for `value`
    dev = torch.device("cuda", local_rank)
    t_rank = torch.from_numpy(d["rank"]).to(dev)
    t_off = torch.from_numpy(d["off"]).to(dev)
    t_codes = torch.from_numpy(d["codes"]).to(dev)
    # pinned host inputs for `e2e`
    p_rank = torch.from_numpy(d["rank"]).pin_memory()
    p_off = torch.from_numpy(d["off"]).pin_memory()
    p_codes = torch.from_numpy(d["codes"]).pin_memory()
    # ... in the compact wire format the packer emits for the GPU path (uint16 SNP counts, nibble codes)
    klen, codes4, n_codes = util.compact_packed(d["off"], d["codes"])
    p_klen = torch.from_numpy(klen).pin_memory()
    p_codes4 = torch.from_numpy(codes4).pin_memory()
    h2d_bytes = p_rank.numel() * 4 + p_klen.numel() * 2 + p_codes4.numel()
    if args.e2e_format == "wide":
        h2d_bytes = p_rank.numel() * 4 + p_off.numel() * 8 + p_codes.numel()
    # ... or in the dense wire format (uint8 rank deltas and SNP counts, 2-bit alleles + exception list), in a
    # few chunks so that each chunk's copy overlaps the previous chunk's pair expansion
    dense_chunks = []
    dense_h2d = 0
    if args.e2e_format in ("dense", "auto"):
        _keep = []
        for c in util.dense_chunks(d["rank"], d["off"], d["codes"], args.e2e_chunks):
            pinned = torch.from_numpy(c.blob).pin_memory()
            _keep.append(pinned)
            dense_chunks.append(c.rebased(pinned.numpy()))
        dense_h2d = sum(c.nbytes for c in dense_chunks)
        if args.e2e_format == "dense":
            h2d_bytes = dense_h2d
        else:                                 # hx_ingest_host: allele bytes as they are + uint8 rank deltas and SNP counts
            packed_h2d = p_rank.numel() * 4 + p_off.numel() * 8 + p_codes.numel()
            slim = R >= 200000 and bool(np.all(np.diff(d["rank"]) >= 0))
            h2d_bytes = (p_codes.numel() + R * (1 + (1 if W + 1 < 256 else 2))) if slim else packed_h2d

    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W, device=local_rank)
    h.set_ingest_kernel(args.kernel)
    h.counts_buffer()                      # allocate the pending counts outside the timed region
    stream = torch.cuda.ExternalStream(h.stream, device=dev)

    pipe = None
    fused = None
    seam = None
    if strong and args.exchange in ("auto", "allreduce", "seam"):
        seam = gdist.SeamExchange(h, int(d["rank"][-1]) if R else -1)
    if world > 1 and args.exchange == "fused":
        fused = gdist.FusedExchange(h)
    elif world > 1 and args.segments > 1:
        pipe = gdist.PipelinedIngest(h, d["rank"], R, segments=args.segments)

    def step():
        if fused is not None:
            fused.reset()
            h.ingest_device(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R)
            fused.finish()
            return
        h.reset_counts()
        if pipe is not None:
            pipe.run(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr())
            return
        h.ingest_device(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R)
        if seam is not None:
            gdist.seam_exchange_counts(h, None, plan=seam)
        elif world > 1:
            if args.exchange == "reduce":
                gdist.reduce_counts(h, dst=0)
            elif args.exchange == "packed":
                gdist.allreduce_counts_packed(h)
            else:
                gdist.allreduce_counts(h)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1, weak scaling: consecutive steps are independent ingestion jobs, so the all-reduce of step i is put behind
    # the pair expansion of step i+1 (two matrices take turns, a few SMs are left to NCCL).  Every step still zeroes,
    # expands and all-reduces its own matrix, and all K all-reduces end inside the timed region.
    ov = None
    if overlap:
        h2 = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W, device=local_rank)
        h2.set_ingest_kernel(args.kernel)
        h2.counts_buffer()
        # "auto": the same NCCL integer all-reduce over counts packed two to a word when one job's counts leave room
        # (largest count on any rank x world x 2 <= 65535; decided once, on a first complete job)
        packed_ok = False
        if args.exchange == "auto" and world >= 4:          # (2 GPUs: the plain all-reduce is short enough; measured slower packed)
            h.reset_counts()
            h.ingest_device(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R)
            packed_ok = gdist.OverlappedAllreduce.packing_is_safe(h)
        ov = gdist.OverlappedAllreduce([h, h2], free_sms=args.comm_sms, packed=packed_ok)
        stream = ov.main

    def ov_ingest(hh):
        hh.reset_counts()
        hh.ingest_device(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R)

    for _ in range(max(args.warmup, 3)):
        if ov is not None:
            ov.step(ov_ingest)
        else:
            step()
    if ov is not None:
        ov.drain()
    barrier()
    totals = h.ingest_totals()
    n_obs_global = totals[1]               # crumbs of ALL ranks (totals are all-reduced too)
    kernel_ms = []
    launches0 = h.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.region(True)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    if ov is not None:
        launches0 += h2.launch_count()
        with torch.cuda.stream(stream):
            ev[0][0].record(stream)
            for i in range(args.steps):
                ov.step(ov_ingest)
            ov.drain()
            ev[0][1].record(stream)
        barrier()
        wall_s = time.perf_counter() - t_wall0
        sampler.region(False)
        launches = h.launch_count() + h2.launch_count() - launches0
        total_ms = float(ev[0][0].elapsed_time(ev[0][1]))
        # parity of the overlapped path itself: the matrix of the last job against the independent per-row recount
        last = ov.hs[(ov.i - 1) & 1]
        o_exp = torch.zeros(N + 2, dtype=torch.int64, device=dev)
        o_got = torch.zeros(N + 2, dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        last.probe_expected_rows(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R, o_exp.data_ptr())
        last.counts_row_sums(o_got.data_ptr())
        last.sync()
        dist.all_reduce(o_exp, op=dist.ReduceOp.SUM)
        o_ok = torch.tensor([int(torch.equal(o_exp, o_got))], device=dev)
        dist.all_reduce(o_ok, op=dist.ReduceOp.MIN)
        overlap_probe_ok = bool(o_ok.item())
        # the same K steps one after the other (the all-reduce fully exposed), for comparison
        barrier()
        with torch.cuda.stream(stream):
            ev[1 % len(ev)][0].record(stream)
            for i in range(args.steps):
                step()
            ev[1 % len(ev)][1].record(stream)
        barrier()
        serial_ms = float(ev[1 % len(ev)][0].elapsed_time(ev[1 % len(ev)][1]))
    else:
        with torch.cuda.stream(stream):
            for i in range(args.steps):
                ev[i][0].record(stream)
                step()
                ev[i][1].record(stream)
        barrier()
        wall_s = time.perf_counter() - t_wall0
        sampler.region(False)
        launches = h.launch_count() - launches0
        step_ms = [a.elapsed_time(b) for a, b in ev]
        total_ms = float(sum(step_ms))
        serial_ms = None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, h, N, W)
    # kernel-only duration (events inside the library, on the launching stream) for the roofline
    for _ in range(3):
        h.reset_counts()
        h.ingest_device(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R)
        h.ingest_totals()
        kernel_ms.append(h.kernel_ms("ingest"))
    if world > 1:
        tt = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms = float(tt.item())
    value = n_obs_global * args.steps / (total_ms * 1e-3)
    if serial_ms is not None and world > 1:
        tt = torch.tensor([serial_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        serial_ms = float(tt.item())

    # ---- parity probe: one more complete step (ingestion + exchange), then an independent recount of what
    # every band row must hold (hx_probe_expected_rows, summed over ranks) against the row sums of the
    # counters the step left behind, and the grand total against n_crumbs + sentinel increments.
    step()
    barrier()
    rows_exp = torch.zeros(N + 2, dtype=torch.int64, device=dev)
    rows_got = torch.zeros(N + 2, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    h.probe_expected_rows(t_rank.data_ptr(), t_off.data_ptr(), t_codes.data_ptr(), R, rows_exp.data_ptr())
    h.counts_row_sums(rows_got.data_ptr())
    h.sync()
    if world > 1:
        dist.all_reduce(rows_exp, op=dist.ReduceOp.SUM)
    pt = h.ingest_totals()
    holder = rank == 0 or (args.exchange != "reduce" and seam is None)   # "reduce" / the seam exchange leave the sums on rank 0
    rows_ok = bool(torch.equal(rows_exp, rows_got)) if holder else True
    sum_ok = int(rows_got.sum().item()) == int(pt[1]) + int(pt[3]) if holder else True
    pok = torch.tensor([int(rows_ok and sum_ok)], device=dev)
    if world > 1:
        dist.all_reduce(pok, op=dist.ReduceOp.MIN)
    if ov is not None:
        pok = torch.tensor([int(bool(pok.item()) and overlap_probe_ok)], device=dev)
    parity_probe = {"ok": bool(pok.item()), "rows_equal": rows_ok, "sum_equals_crumbs_plus_sentinels": sum_ok,
                    "rows": N + 2, "band_sum": int(rows_got.sum().item()), "n_crumbs": int(pt[1]),
                    "sentinel_increments": int(pt[3]), "ranks_checked": world if (args.exchange != "reduce" and seam is None) else 1,
                    "how": "hx_probe_expected_rows (one thread per read, independent of the ingestion kernels) "
                           "summed over ranks vs hx_counts_row_sums of the exchanged counts"}

    if fused is not None:
        fused.close()

    # ---- e2e through the public API with host buffers
    host_threads = max(1, (os.cpu_count() or 1) // max(1, world))
    os.environ.setdefault("HX_HOST_THREADS", str(host_threads))

    def e2e_step(fmt):
        hh = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W, device=local_rank)
        hh.set_ingest_kernel(args.kernel)
        if fmt == "auto":                  # the north_star boundary: packed arrays in, the library does the rest
            hh.ingest_packed(p_rank.numpy(), p_off.numpy(), p_codes.numpy())
        elif fmt in ("encoded", "wide", "packed"):   # force the host-side dense encoder / one plain copy / 4 plain chunks
            os.environ["HX_HOST_PIPELINE"] = {"encoded": "dense", "wide": "off", "packed": "packed"}[fmt]
            try:
                hh.ingest_packed(p_rank.numpy(), p_off.numpy(), p_codes.numpy())
            finally:
                del os.environ["HX_HOST_PIPELINE"]
        elif fmt == "dense":
            for c in dense_chunks:
                hh.ingest_packed_dense(c, wait=False)
        else:
            hh.ingest_packed_compact(p_rank.numpy(), p_klen.numpy(), p_codes4.numpy(), n_codes)
        if seam is not None:
            gdist.seam_exchange_counts(hh, None, plan=seam)
        elif world > 1:
            (gdist.allreduce_counts_packed if args.exchange == "packed" else gdist.allreduce_counts)(hh)
        hh.finalize()                      # enqueue the fold into the float matrix, then one wait for everything
        s, c, v, _ = hh.ingest_totals()
        util.set_totals(hh, s, c, v)
        return hh

    def time_e2e(fmt, steps):
        for _ in range(6):                    # untimed: thread pool, pinned staging and parked handles warm (fresh box)
            e2e_step(fmt).close()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            hh = e2e_step(fmt)
            crumbs = hh.n_crumbs
            hh.close()
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        return crumbs * steps / dt, dt / steps

    e2e_steps = args.steps
    # (the 1 kHz NVML sampling thread stays off here: its driver calls delay the ~100 CUDA API calls of a step; the
    # clocks line describes the device-timed region above)
    e2e_value, e2e_step_s = time_e2e(args.e2e_format, e2e_steps)
    e2e_pre = None
    if args.e2e_format == "auto" and dense_chunks:
        v2, s2 = time_e2e("dense", e2e_steps)
        v3, s3 = time_e2e("encoded", e2e_steps)
        v4, s4 = time_e2e("packed", e2e_steps)
        e2e_pre = {"packed_arrays": {"value": v4, "unit": UNIT, "ms_per_step": 1e3 * s4, "h2d_bytes_per_step": int(packed_h2d),
                                     "what": "HX_HOST_PIPELINE=packed: rank int32, off int64 and the allele bytes copied as "
                                             "they are in 4 chunks (round 2's first honest e2e path)"},
                   "preencoded_dense": {"value": v2, "unit": UNIT, "ms_per_step": 1e3 * s2, "h2d_bytes_per_step": int(dense_h2d),
                                        "what": "dense chunks encoded BEFORE the clock (device-side limit of the pipeline; not "
                                                "the headline)"},
                   "host_encoded_dense": {"value": v3, "unit": UNIT, "ms_per_step": 1e3 * s3, "h2d_bytes_per_step": int(dense_h2d),
                                          "what": "HX_HOST_PIPELINE=dense: the same packed host arrays re-encoded by the host "
                                                  "threads inside the clock, pipelined with copies and expansion"}}
    clocks = sampler.stop() if rank == 0 else None

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (this rank's launch)
    k_mean = float(k.mean())
    local_obs = n_obs_global / world
    kms = float(np.mean(kernel_ms))
    peak, peak_src = measured_peak_gbs()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            key = "%s:%d:k%d" % (args.workload, R, args.kernel)
            traffic = tj.get(key, tj.get(args.workload))
        except Exception:
            traffic = None
    # The bound that binds: HBM on the COMPULSORY bytes of one launch - the packed reads once (int32 rank + int64
    # offset per read, one byte per allele) plus one read-modify-write of every band counter the reads touch.
    # Counting happens on chip (tensor-core MMAs into TMEM / AND+POPC in registers), so SURVEY 8(d)'s model of one
    # uint32 read-modify-write in HBM per observation does not describe the kernel; its figure is kept beside it.
    touched = float(np.unique(d["rank"]).size) * max(W, 1) * 16 * 4 if R else 0.0
    compulsory = float(R) * 12.0 + float(k.sum()) + 2.0 * touched
    achieved = compulsory / (kms * 1e-3) / 1e9
    s8d_bytes = local_obs * b_obs(k_mean)
    s8d_achieved = s8d_bytes / (kms * 1e-3) / 1e9
    umma = args.kernel in (0, 6) and d["max_k"] <= 32 and R >= 64 * (N + 1)
    lumma = args.kernel == 7 or (args.kernel == 0 and d["max_k"] > 52)
    groups = float(np.ceil(np.bincount(d["rank"]) / 32.0).sum()) if R else 0.0
    roofline = {"bound": "hbm", "kernel": "ingestion (pair expansion): " + ("k1_umma (int8 tcgen05.mma)" if umma else "k_l2_tiles (int8 tcgen05.mma over one-hot slabs, long reads)" if lumma else "k1_bitsliced / tiles"),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "kernel_ms": kms,
                "algorithmic_bytes_per_launch": compulsory,
                "algorithmic_bytes_model": "compulsory traffic: 12 B per read (rank, offset) + 1 B per allele + one 4 B "
                                           "read-modify-write of each of the 16 ACGTxACGT counters of every band cell "
                                           "under the covered ranks",
                "obs_per_launch": local_obs,
                "dram_frac": (traffic / (kms * 1e-3) / 1e9 / peak) if traffic else None,
                "survey_8d": {"bytes_per_obs": b_obs(k_mean), "achieved": s8d_achieved, "frac": s8d_achieved / peak,
                              "note": "SURVEY 8(d) charges one uint32 RMW in HBM per observation; on-chip counting makes "
                                      "this exceed 1 - reported for continuity, not as a bound"},
                "tensor_floor": ({"mma_per_launch": groups, "cycles_per_mma": 64, "floor_ms": groups * 64 / 148 / 1.965e6,
                                  "frac": (groups * 64 / 148 / 1.965e6) / kms,
                                  "note": "one M=128,N<=128,K=32 int8 MMA per 32 reads at the 8192 MAC/clk/SM peak"} if umma
                                 else lumma_floor(d["rank"], d["off"], kms) if lumma else None),
                "pipe_floor": (popc_floor(d["rank"], d["off"], kms) if (d["max_k"] <= 52 and not umma) else None)}

    # which of the floors is the tightest (the largest fraction = the resource closest to binding)
    cands = [("hbm (compulsory traffic)", roofline["frac"])]
    if roofline["tensor_floor"]:
        cands.append(("tensor (MMA count at the 64-cycle int8 peak)", roofline["tensor_floor"]["frac"]))
    if roofline["pipe_floor"]:
        cands.append(("xu pipe (POPC count)", roofline["pipe_floor"]["frac"]))
    best = max(cands, key=lambda c: c[1])
    roofline["tightest_bound"] = {"name": best[0], "frac": best[1],
                                  "note": "none of the floors binds: the short-read kernel is limited by instruction issue and the "
                                          "per-run hand-over between its expander and readout warps, the long-read kernel by "
                                          "shared-memory bandwidth under the MMAs (DESIGN.md section 4, profiles/r2_ingest_*.md)"}

    # ---- CPU baseline: the reference's per-pair Python loop on a bounded sample, all cores
    if args.no_cpu_baseline:
        args.recovery_cpu_baseline = False
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import py_baseline as pb
        cores = os.cpu_count() or 1
        sample_reads = int(min(R, 1_000_000, max(2000, 15_000 * cores)))
        lo = (R - sample_reads) // 2
        sr, so = d["rank"][lo:lo + sample_reads], d["off"][lo:lo + sample_reads + 1]
        c_cr, c_t = pb.timed_ingest(sr, so - so[0], d["codes"][so[0]:so[-1]], N, W, n_procs=cores)
        cpu = {"value": c_cr / c_t, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d consecutive reads (%d observations) from the middle of rank 0's shard, %d forked "
                         "workers, oracle/py_baseline.py (per-pair Python calls as gretel/util.py:242-286)" % (
                             sample_reads, c_cr, cores)}
        try:                                   # BASELINE.md B1: the same loop in one process, on 1/cores of the sample
            one = max(2000, sample_reads // cores)
            s1, o1 = d["rank"][lo:lo + one], d["off"][lo:lo + one + 1]
            c1, t1 = pb.timed_ingest(s1, o1 - o1[0], d["codes"][o1[0]:o1[-1]], N, W, n_procs=1)
            cpu["one_core"] = {"value": c1 / t1, "unit": UNIT, "cores": 1, "sample": "%d reads" % one}
        except Exception as e:                 # never let the secondary figure break the bench line
            cpu["one_core"] = {"error": str(e)}

    # ---- secondary metric: haplotype recovery seconds on this matrix (rank 0, one GPU)
    recovery = None
    if args.recover_paths > 0:
        s, c, v, _ = h.ingest_totals()
        h.finalize()
        util.set_totals(h, s, c, v)
        orig = h.copy()
        t0 = time.perf_counter()
        paths, stats = h.recover_codes(orig, args.recover_paths, 0.01)
        rec_s = time.perf_counter() - t0
        recovery = {"haplotypes": int(len(paths)), "seconds": rec_s, "L": h.L, "n_snps": N,
                    "us_per_site": (1e6 * rec_s / max(1, len(paths)) / N) if len(paths) else None}
        if args.recovery_sweep:
            # BASELINE.json configs[4]: up to 50 ranked haplotypes at lookback L = 1..8 on the 10k-SNP matrix
            sweep = []
            for L in range(1, 9):
                hc = orig.copy()
                hc.L = L
                t0 = time.perf_counter()
                pp, _ = hc.recover_codes(orig, 50, 0.01)
                sweep.append({"L": L, "haplotypes": int(len(pp)), "seconds": time.perf_counter() - t0})
                hc.close()
            recovery["sweep_L1_8_50_haplotypes"] = sweep
        if args.recovery_cpu_baseline:
            recovery["cpu_port"] = recovery_cpu_baseline(local_rank)
            # BASELINE.md B3 at N = 10k: one haplotype per L in {1, 4, 8} by the C restatement (one host core) next
            # to the same haplotype on the GPU
            try:
                from oracle import c_oracle
                band0 = orig.band()
                b3 = []
                for L in (1, 4, 8):
                    cur = band0.copy()
                    t0 = time.perf_counter()
                    pc, res = c_oracle.generate_path(cur, band0, N, W, L)
                    t_gen = time.perf_counter() - t0
                    t0 = time.perf_counter()
                    if pc is not None:
                        c_oracle.reweight_path(cur, N, W, pc, max(res[2], 0.01))
                    t_rw = time.perf_counter() - t0
                    hc = orig.copy()
                    hc.L = L
                    t0 = time.perf_counter()
                    g = hc.generate_path_codes(orig)
                    if g[0] is not None:
                        hc.reweight_path_codes(g[0], max(g[3], 0.01))
                    t_gpu = time.perf_counter() - t0
                    b3.append({"L": L, "c_oracle_generate_s": t_gen, "c_oracle_reweight_s": t_rw, "gpu_s": t_gpu,
                               "same_haplotype": bool(pc is not None and g[0] is not None and np.array_equal(pc, g[0]))})
                    hc.close()
                recovery["cpu_c_oracle_n10k"] = {"cores": 1, "kind": "port (C restatement, oracle/hansel_oracle.c)", "per_L": b3}
            except Exception as e:                 # a secondary figure must not break the bench line
                recovery["cpu_c_oracle_n10k"] = {"error": repr(e)}

    # ---- e2e_bam: BAM file -> load_from_bam -> matrix (the reference's real entry point, gretel/util.py:33)
    e2e_bam = None
    if args.bam_reads > 0 and not synth.WORKLOADS[args.workload].long_reads:
        import tempfile
        from gretel_b200 import bamio
        wb = synth.scaled(synth.WORKLOADS[args.workload], args.bam_reads)
        db = synth.generate(wb)
        tmpd = tempfile.mkdtemp(prefix="hx_bam_")
        bpath = os.path.join(tmpd, "synthetic.bam")
        t0 = time.perf_counter()
        vh, keep = synth.write_bam(bpath, db, wb, threads=os.cpu_count() or 1)
        write_s = time.perf_counter() - t0
        cores = os.cpu_count() or 1
        best = None
        for _ in range(3):
            st = {}
            t0 = time.perf_counter()
            hb = util.load_from_bam(bpath, "ctg", 1, wb.genome_len, vh, n_threads=cores, device=local_rank, stages=st)
            dt = time.perf_counter() - t0
            crumbs_b, reads_b = hb.n_crumbs, st["reads"]
            hb.close()
            if best is None or dt < best[0]:
                best = (dt, st)
        dt, st = best
        # the same reads from the packed arrays ('-' is written as 'N' in the fixed-length records)
        cb = db["codes"].copy()
        cb[cb == 5] = 4
        kb_ = np.diff(db["off"])
        sel = np.repeat(keep, kb_)
        offb = np.concatenate([[0], np.cumsum(kb_[keep])]).astype(np.int64)
        href = util.load_from_packed(db["rank"][keep], offb, cb[sel], wb.n_snps, band_w=None, device=local_rank)
        same = bool(href.n_crumbs == crumbs_b and href.n_slices == reads_b)
        href.close()
        e2e_bam = {"reads_per_s": reads_b / dt, "obs_per_s": crumbs_b / dt, "seconds": dt, "reads": int(reads_b),
                   "records": int(st.get("records", 0)), "bam_mbytes": os.path.getsize(bpath) / 1e6, "threads": cores,
                   "max_depth": int(bamio.PYSAM_MAX_DEPTH),
                   "stage_seconds": {k_: round(float(st[k_]), 5) for k_ in ("read", "inflate", "scan", "depth", "walk", "gather",
                                                                          "pack_total", "gpu_ingest")},
                   "gpu_share": st["gpu_ingest"] / dt, "same_totals_as_packed_arrays": same,
                   "synthetic_bam_write_s": write_s,
                   "what": "util.load_from_bam on a synthetic coordinate-sorted BAM of %d of the workload's reads (150M "
                           "CIGARs, random base qualities), best of 3" % args.bam_reads}
        try:
            os.remove(bpath)
            os.rmdir(tmpd)
        except OSError:
            pass

    # ---- the other ingestion configs of BASELINE.json (configs[1] HIV-like, configs[3] ONT-like) in the same line, so
    # that the driver's default run carries a device-timed, parity-probed figure for each of them (N = 1 only)
    other_configs = None
    if world == 1 and args.other_configs and args.workload == "metagenome" and not args.reads:
        other_configs = {}
        for name in ("hiv", "ont"):
            try:
                other_configs[name] = measure_other_config(name, args, local_rank)
            except Exception as e:             # a secondary figure must not break the bench line
                other_configs[name] = {"error": repr(e)}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": dict(workload_config(args, k_mean, R), **({"reads_total": int(args.reads or w.n_reads),
                                                                 "reads_per_gpu": "one read set cut into %d contiguous chunks balanced by pair count" % world} if strong else {})),
            "step_overlap": ({"on": True, "comm_sms": args.comm_sms, "packed_uint16_lanes": bool(ov.packed),
                              "parity_probe_ok": overlap_probe_ok,
                              "what": "the all-reduce of step i runs on a second stream beside the pair expansion of step i+1 "
                                      "(two matrices take turns; the ingestion kernel leaves comm_sms SMs to NCCL)",
                              "value_without_overlap": n_obs_global * args.steps / (serial_ms * 1e-3),
                              "ms_per_step_without_overlap": serial_ms / args.steps} if ov is not None else None),
            "exchange_detail": ({"kind": "seam" if not seam.fallback else "allreduce (seam fallback)",
                                 "bytes_on_wire": seam.bytes_on_wire(), "own_rows": [seam.own_lo, seam.own_hi]} if seam is not None else None),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": 32 + 4, "steps": e2e_steps, "ms_per_step": 1e3 * e2e_step_s,
                    "wire_format": args.e2e_format, "host_threads": int(os.environ.get("HX_HOST_THREADS", "0")),
                    "host_bytes_read_per_step": int(p_rank.numel() * 4 + p_off.numel() * 8 + p_codes.numel()),
                    "api": {"auto": "Hansel.init_matrix + Hansel.ingest_packed(rank, off, codes in pinned host memory) -> "
                                    "hx_ingest_host: 6 chunks; per chunk the allele bytes are copied straight from the "
                                    "caller's memory while host threads turn its ranks and offsets into uint8 rank deltas "
                                    "and SNP counts (inside the clock), the device rebuilds rank / offsets with a scan and "
                                    "expands the chunk while the next is in flight [+ all-reduce] + finalize + totals, a "
                                    "new matrix every step",
                            "encoded": "the same with HX_HOST_PIPELINE=dense (host threads re-encode inside the clock)",
                            "dense": "pre-encoded dense chunks (encoding outside the clock) + finalize + totals",
                            "compact": "ingest_packed_compact", "wide": "hx_ingest_host, one plain copy"}[args.e2e_format],
                    "other_paths": e2e_pre},
            "e2e_bam": e2e_bam,
            "gpu_launches": int(launches), "parity_probe": parity_probe, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "observations_per_step": int(n_obs_global), "wall_s_timed_region": wall_s,
            "recovery": recovery, "other_configs": other_configs, "synth_seconds": gen_s, "band_w": W, "allreduce_segments": args.segments if world > 1 else 0, "exchange": args.exchange if world > 1 else None,
            "ingest_kernel": args.kernel}
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="metagenome", choices=sorted(synth.WORKLOADS))
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU (default: the workload's full size)")
    ap.add_argument("--kernel", type=int, default=0, help="ingestion kernel: 0 auto, 1 generic, 2 bit-sliced, 3 long-read bit-plane tiles, 6 tensor-core (short reads), 7 tensor-core (long reads)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N>1: weak = every GPU ingests its own full-size read set of the same region (default, what the "
                         "driver's scaling run uses); strong = ONE read set cut into contiguous chunks, seam-only exchange")
    ap.add_argument("--exchange", default="auto", choices=["auto", "allreduce", "packed", "reduce", "fused", "seam"],
                    help="N>1: NCCL all-reduce of the partial matrices (default, as north_star names it); the same "
                         "all-reduce over counts packed into uint16 lanes (half the bytes); reduce onto "
                         "rank 0 only (recovery runs there); or counts added straight into the owning GPU over "
                         "NVLink peer memory + all-gather of the owned rows")
    ap.add_argument("--overlap-steps", action="store_true", default=True,
                    help="N>1, weak scaling: put the all-reduce of step i behind the pair expansion of step i+1 (default)")
    ap.add_argument("--no-overlap-steps", dest="overlap_steps", action="store_false")
    ap.add_argument("--comm-sms", type=int, default=16, help="SMs left to NCCL when steps overlap")
    ap.add_argument("--segments", type=int, default=1,
                    help="N>1: ingest in this many launches, all-reducing finished band rows behind the next one")
    ap.add_argument("--e2e-format", default="auto", choices=["auto", "encoded", "dense", "compact", "wide"],
                    help="e2e leg: auto = packed (rank, off, codes) host arrays through hx_ingest_host (the headline); "
                         "encoded = the same with the host-side dense encoder forced; dense = chunks pre-encoded before "
                         "the clock; compact = int32 ranks + uint16 counts + nibble codes; wide = one plain copy")
    ap.add_argument("--e2e-chunks", type=int, default=4,
                    help="dense format: chunks per step (copy of chunk i+1 overlaps the expansion of chunk i)")
    ap.add_argument("--bam-reads", type=int, default=1_000_000,
                    help="reads of the synthetic BAM of the e2e_bam leg (0 = skip)")
    ap.add_argument("--recover-paths", type=int, default=5)
    ap.add_argument("--recovery-sweep", action="store_true", default=True,
                    help="also time configs[4]: 50 haplotypes at L=1..8 (a few seconds)")
    ap.add_argument("--no-recovery-sweep", dest="recovery_sweep", action="store_false")
    ap.add_argument("--recovery-cpu-baseline", action="store_true", default=True,
                    help="also recover one ~1k-SNP haplotype with the literal Python restatement (~10-20 s of CPU)")
    ap.add_argument("--no-recovery-cpu-baseline", dest="recovery_cpu_baseline", action="store_false")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", dest="other_configs", action="store_false", default=True,
                    help="skip the device-timed figures of configs[1] (HIV-like) and configs[3] (ONT-like) in the default line")
    ap.add_argument("--ref-sample", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the last step's totals and counts as .npy files into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm keeps no outputs")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
