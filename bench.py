#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 tree-likelihood path (driver contract, task ④).

One "step" = one full lnL + branch-gradient evaluation (protocol of the reference's
examples/benchmarking.c:498-503: every node dirty, new branch lengths in, transition matrices
rebuilt, post-order + pre-order passes, lnL and grad[N] back on the host).

Headline workload: BASELINE.json configs[1] -- GTR+Γ4 nucleotide, synthetic 1000 taxa × 100k site
patterns per GPU (weak scaling over ranks: one process per GPU, patterns sharded, ONE ncclAllReduce of
[lnL, grad[N], inf flag] per step issued by the C library on the evaluation's stream).
The same JSON line carries a `configs` object with one sub-record per remaining BASELINE config
(c1 fluA JC69 time tree, c2_1m = the north-star 1000 × 1M, c3 HKY+Γ4 × 128 samples, c4 LG+Γ4 200 × 200k,
c5 GY94 100 × 1M); at N > 1 those are STRONG splits of the named sizes (1M / N, 200k / N, 1M / N
patterns per GPU; c3 splits its samples).  Every record is gated on parity with the unmodified
reference (oracle/_ref) evaluated on a bounded sample of the same workload.

    python bench.py --gpus 1 --steps 20 --warmup 3
    torchrun --nproc-per-node N bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own CPU path (oracle/_ref) on host cores
"""
from __future__ import annotations

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
# the benchmark may run from a read-only tree and leaves it as it found it: no __pycache__ here or in worker processes
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

from physher_b200 import models, synthetic as syn  # noqa: E402

CONFIGS = {
    # name: (taxa, patterns per GPU, states, categories, model)
    "c2": dict(taxa=1000, patterns=100_000, states=4, cats=4, model="GTR+G4", mu=0.04),
    "c2_1m": dict(taxa=1000, patterns=1_000_000, states=4, cats=4, model="GTR+G4", mu=0.04),
    "c3": dict(taxa=500, patterns=50_000, states=4, cats=4, model="HKY+G4", mu=0.04, batch=128),
    "c4": dict(taxa=200, patterns=200_000, states=20, cats=4, model="LG+G4", mu=0.08),
    "c5": dict(taxa=100, patterns=1_000_000, states=61, cats=1, model="GY94", mu=0.1),
}
# FP64 tensor-core throughput measured on this pool's B200 with tools/dmma_peak.cu (profiles/r1_c_dmma_peak.md); nominal 40
DMMA_PEAK_TFLOPS_FILE = os.path.join(ROOT, "profiles", "dmma_peak.json")
CODON_BASES = "TCAG"
CODON_AA = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
METRIC = "lnL+gradient throughput (site patterns x tree nodes per second)"
UNIT = "pattern*node/s"


def make_inputs(cfg: dict, rank: int, seed: int = 20261017):
    """Seeded synthetic inputs (SURVEY.md §8d). Topology, model and branch lengths are identical on
    every rank; each rank draws its own pattern shard."""
    T, P, S, C = cfg["taxa"], cfg["patterns"], cfg["states"], cfg["cats"]
    topo = syn.random_topology(T, seed)
    bl = syn.random_branch_lengths(topo, seed + 1)
    if S == 4 and cfg["model"].startswith("HKY"):
        m = models.hky(3.0, [0.1, 0.2, 0.3, 0.4])
    elif S == 4:
        m = models.gtr([0.05, 0.3, 0.1, 0.15, 0.3, 0.1], [0.1, 0.2, 0.3, 0.4])
    elif S == 61:
        m = models.gy94(2.5, 0.3)
    elif S == 20:
        m = lg_model()
    else:
        m = models.random_reversible(S, seed + 2)
    rates, props = models.discrete_gamma(0.5, C)
    # data evolved down the same tree at 0.35x the evaluation branch lengths: all columns unique, per-pattern lnL
    # around -240 (min > -400), so neither arm ever switches rescaling on (SURVEY.md 8c caveat 2)
    patterns = syn.simulate_patterns(topo, bl * 0.35, P, S, seed + 100 + rank)
    weights = np.ones(P)
    return topo, bl, m, rates, props, patterns, weights


def inputs_sha256(topo, bl, m, rates, props, patterns=None, weights=None):
    """SHA-256 of the workload as both arms see it (SURVEY.md 8d: recorded next to every result).  `tree_model` covers topology,
    branch lengths, eigen system, frequencies and the site model -- identical in both arms and on every rank; `patterns` covers the
    pattern shard of rank 0 (our arm; the reference arm times bounded shards of the same generator, see cpu_baseline.sample)."""
    import hashlib

    h = hashlib.sha256()
    for a in (topo.left, topo.right, [topo.root], bl, m.evec, m.eval, m.ivec, m.freqs, rates, props):
        h.update(np.ascontiguousarray(a, dtype=np.float64).tobytes())
    out = {"tree_model": h.hexdigest()}
    if patterns is not None:
        g = hashlib.sha256()
        g.update(np.ascontiguousarray(patterns, dtype=np.uint8).tobytes())
        g.update(np.ascontiguousarray(weights, dtype=np.float64).tobytes())
        out["patterns_rank0"] = g.hexdigest()
    return out


def lg_model():
    """LG eigen system as the reference's host code produced it (lg.c + eigen.c), stored in the committed golden fixture."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "synth_lg_g4_tipstates.npz"))
    return models.SubstitutionModel("LG", 20, z["freqs"], z["evec"], z["eval"], z["ivec"])


def algorithmic_flops(cfg: dict) -> float:
    """SURVEY.md §8d: 8 S^2 (T-2) flop per pattern per category (one S x S mat-vec per internal operand)."""
    T, P, S, C = cfg["taxa"], cfg["patterns"], cfg["states"], cfg["cats"]
    return 8.0 * S * S * (T - 2) * C * P


def dmma_peak():
    try:
        d = json.load(open(DMMA_PEAK_TFLOPS_FILE))
        return float(d["dmma_tflops"]), f"measured (tools/dmma_peak.cu, {d.get('shape', 'm8n8k4')}, profiles/dmma_peak.json)"
    except Exception:
        return 40.0, "nominal B200 FP64 tensor (no measured file)"


def algorithmic_bytes(cfg: dict) -> float:
    """Streaming-model bytes per evaluation (SURVEY.md §8d): P * [(5T-9) * C*S*8 + 10T]."""
    T, P, S, C = cfg["taxa"], cfg["patterns"], cfg["states"], cfg["cats"]
    return P * ((5 * T - 9) * C * S * 8.0 + 10 * T)


class ClockSampler:
    """SM clock / throttle-reason sampling DURING the timed region (B200_PROFILING.md clocks line): NVML polled from a
    thread every few ms (the timed region of a short run is shorter than one `nvidia-smi -lms` period), with the
    nvidia-smi loop as the fallback when the NVML binding is missing."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int, period_s: float = 0.004):
        self.index, self.period = index, period_s
        self.proc, self.lines, self.samples, self.stop = None, [], [], threading.Event()
        self.nvml = None

    def _nvml_sample(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        self.samples.append((float(sm), float(self._mx), [k for k, b in self._bits.items() if r & b]))

    def _nvml_loop(self):
        while not self.stop.is_set():
            try:
                self._nvml_sample()
            except Exception:
                pass
            self.stop.wait(self.period)

    def __enter__(self):
        try:
            import pynvml

            # initialisation, the handle and a first query happen HERE, before the timed region starts: the first NVML calls of a
            # process take tens of milliseconds, longer than a short timed region (a run once came back with no sample at all)
            n = pynvml
            n.nvmlInit()
            self.nvml = n
            self._h = n.nvmlDeviceGetHandleByIndex(self.index)
            self._bits = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                          "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
            self._mx = n.nvmlDeviceGetMaxClockInfo(self._h, n.NVML_CLOCK_SM)
            n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)  # warm the query path; not a sample (the region has not started)
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        self.stop.set()
        if self.nvml is not None:
            self.thread.join(timeout=2)
            if not self.samples:  # the region ended inside the first polling period: one sample at its very end
                try:
                    self._nvml_sample()
                except Exception:
                    pass
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        for s_, m_, r_ in self.samples:
            sm.append(s_)
            mx.append(m_)
            reasons.update(r_)
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(self.NAMES, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvml" if self.samples else "nvidia-smi"}


def measured_traffic(config_name, kernels, patterns, lib_version):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed ncu --set full
    capture of this workload (profiles/traffic.json, written by tools/ncu_traffic.py).  A capture only counts for the kernel
    revision and pattern count it was taken on: None when the library reports another revision (phb_version()) or the launch
    covers another number of patterns -- a stale constant is worse than no number."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[f"{config_name}:{kernels}"]
        if int(d.get("patterns", -1)) != int(patterns) or d.get("kernel_rev") not in lib_version:
            return None
        return float(d["dram_bytes_per_launch"])
    except Exception:
        return None


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# -------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference (oracle/_ref) on host cores
# -------------------------------------------------------------------------------------------------

def _reference_worker(args):
    """One process = one single-threaded reference tree likelihood on a pattern shard."""
    cfg, shard_patterns, shard_index, iters, warm = args[:5]
    want_values = len(args) > 5 and args[5]
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    os.dup2(devnull, 1)  # the reference prints alignment statistics to stdout
    try:
        from oracle import oracle as O

        sub = dict(cfg, patterns=shard_patterns)
        topo, bl, m, rates, props, patterns, weights = make_inputs(sub, rank=1000 + shard_index)
        names = [f"t{i}" for i in range(sub["taxa"])]
        S = sub["states"]
        if S == 4:
            seqs = dict(zip(names, syn.sequences_from_patterns(patterns, syn.NUCLEOTIDES)))
            if sub["model"].startswith("HKY") and sub.get("ref_model") == "gtr_as_hky":
                # HKY(kappa) written as the GTR it is -- exchangeabilities (AC, AG, AT, CG, CT, GT) = (1, k, 1, 1, k, 1) -- so that the
                # reference takes its eigen-decomposition path (substmodel.c:518-557), the form the device path implements
                k = 3.0
                mspec = O.nucleotide_model_spec("gtr", [0.1, 0.2, 0.3, 0.4], list(np.array([1, k, 1, 1, k, 1]) / (4 + 2 * k)))
            elif sub["model"].startswith("HKY"):
                mspec = O.nucleotide_model_spec("hky", [0.1, 0.2, 0.3, 0.4], kappa=3.0)
            else:
                mspec = O.nucleotide_model_spec("gtr", [0.1, 0.2, 0.3, 0.4], [0.05, 0.3, 0.1, 0.15, 0.3, 0.1])
            spec = O.treelikelihood_spec(syn.to_newick(topo, bl, names), seqs, mspec, categories=sub["cats"], alpha=0.5, tipstates=False)
            ref = O.Reference(spec)
        elif S == 20:
            seqs = dict(zip(names, syn.sequences_from_patterns(patterns, syn.AMINO_ACIDS)))
            lg = {"id": "sm", "type": "substitutionmodel", "model": "lg", "datatype": "aa",
                  "frequencies": {"id": "freqs", "type": "Simplex", "values": [float(x) for x in m.freqs]}}
            spec = O.treelikelihood_spec(syn.to_newick(topo, bl, names), seqs, lg, categories=sub["cats"], alpha=0.5, tipstates=False,
                                         datatype="aa")
            ref = O.Reference(spec)
        elif S == 61:
            codons = [a + b + c for a in CODON_BASES for b in CODON_BASES for c in CODON_BASES]
            sense = [c for c, a in zip(codons, CODON_AA) if a != "*"]
            seqs = {n: "".join(sense[s_] for s_ in row) for n, row in zip(names, patterns)}
            ref = O.Reference(codon=dict(newick=syn.to_newick(topo, bl, names), sequences=seqs, kappa=2.5, omega=0.3))
        else:
            raise NotImplementedError(f"reference arm has no model for {S} states")
        # gradient request as in BASELINE.md §4.3: tree model flag, include_root_freqs = false
        ref.time_gradient(warm, O.FLAG_TREE_MODEL, 0)
        sec = ref.time_gradient(iters, O.FLAG_TREE_MODEL, 0)
        npat = ref.P
        nodes = ref.N
        values = None
        if want_values:  # the parity gate of our arm: lnL and branch gradients of this shard from the reference itself
            # ... on the inputs as the REFERENCE holds them after its own parsing (it clamps a zero branch length to its lower
            # bound 1e-8 and moves it to the sibling; its eigen system and Gamma quantiles come from its own eigen.c / gamma.c)
            pb = ref.problem()
            values = dict(lnl=ref.logP(), grad=ref.gradient(O.FLAG_TREE_MODEL, 0)[:nodes].copy(), rescaled=bool(ref.rescaling()),
                          left=pb.left, right=pb.right, root=int(pb.root), tip_states=pb.tip_states, weights=pb.weights, freqs=pb.freqs,
                          rates=pb.rates, props=pb.props, bl=pb.bl, evec=pb.evec, eval=pb.eval, ivec=pb.ivec)
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    return sec, npat, nodes, values


def run_reference(cfg: dict, cores: int, sample_patterns: int, iters: int, warm: int = 1, want_values: bool = False):
    """Throughput of the reference's SSE path: `cores` independent single-threaded processes (the path has no
    intra-likelihood threading, SURVEY.md §2.2) on disjoint pattern shards of a bounded sample."""
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor

    per = max(64, sample_patterns // cores)
    t0 = time.perf_counter()
    # an executor, not mp.Pool: a worker the reference takes down (it exits or crashes on what it dislikes) raises here instead of hanging
    with ProcessPoolExecutor(cores, mp_context=mp.get_context("spawn")) as pool:
        res = list(pool.map(_reference_worker, [(cfg, per, i, iters, warm, want_values and i == 0) for i in range(cores)]))
    wall = time.perf_counter() - t0
    # aggregate: every process evaluates its shard at its own rate
    pn_per_s = sum(npat * nodes / sec for sec, npat, nodes, _ in res)
    return dict(value=pn_per_s, sec_per_eval=[r[0] for r in res], patterns=[r[1] for r in res], nodes=res[0][2], wall=wall, per=per,
                values=res[0][3])


def reference_main(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as O

    if not O.reference_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_harness.so missing (built where /root/reference exists)"}))
        return 0
    cores = os.cpu_count() or 1
    cores = min(cores, 32)
    sample = sample_per_core(cfg) * cores
    iters = max(1, min(args.steps, 10))
    topo_, bl_, m_, rates_, props_, _, _ = make_inputs(dict(cfg, patterns=64), 0)
    t0 = time.perf_counter()
    r = run_reference(cfg, cores, sample, iters, warm=min(args.warmup, 1) or 1)
    total_patterns = sum(r["patterns"])
    ms = 1e3 * float(np.mean(r["sec_per_eval"]))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": iters, "warmup": 1,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(cfg), "taxa": cfg["taxa"], "patterns_per_gpu": cfg["patterns"], "states": cfg["states"],
                   "categories": cfg["cats"], "model": cfg["model"], "inputs_sha256": inputs_sha256(topo_, bl_, m_, rates_, props_)},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "reference",
                         "sample": f"{cores} single-threaded processes x {r['per']} patterns each ({total_patterns} unique patterns total) of the same "
                                   f"{cfg['taxa']}-taxon workload, {iters} lnL+gradient evaluations each, protocol examples/benchmarking.c:498-503"},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "evals_per_s_at_workload": r["value"] / (cfg["patterns"] * r["nodes"]),
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))
    return 0


def sample_per_core(cfg) -> int:
    """Patterns per reference process: ~1 s of CPU work per evaluation and process at each state count, i.e. 10-30 core-seconds
    per core over the warm-up + timed evaluations (the reference allocates every node's partials: ~1.3 GB per process at C2)."""
    return {4: 5000, 20: 2400, 61: 800}.get(cfg["states"], 200)


def workload_name(cfg):
    batch = f" x {cfg['batch']} branch-length samples per step" if cfg.get("batch", 1) > 1 else ""
    return f"{cfg['model']} {cfg['taxa']} taxa x {cfg['patterns']} patterns per GPU{batch}, lnL + branch gradients"


# -------------------------------------------------------------------------------------------------
# our arm
# -------------------------------------------------------------------------------------------------

SUB_CONFIGS = ["c1", "c2_1m", "c3", "c4", "c5"]  # every other BASELINE config, as sub-records of the one JSON line
PARITY_PATTERNS = {4: 256, 20: 128, 61: 64}      # sample the reference evaluates for a sub-record's parity gate (one process)
PARITY_RTOL = 1e-10                              # north_star: lnL and every branch gradient within 1e-10 relative


class Run:
    """What every config of one bench invocation shares: ranks, the torch plumbing, the library and its NCCL communicator."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        import physher_b200 as phb

        self.torch, self.dist, self.phb = torch, dist, phb
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the tree-likelihood path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.comm = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            # the collective of the hot path belongs to the C library (csrc/phb_nccl.c): torch.distributed only carries the
            # 128-byte NCCL id to the other ranks and the max-over-ranks of the timings after the timed regions
            box = [phb.Comm.unique_id() if self.rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            self.comm = phb.Comm(self.world, self.rank, box[0], self.local_rank)

    def reduce(self, values, op="max"):
        if self.world == 1:
            return [float(v) for v in values]
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return [float(v) for v in t.cpu()]

    def sync(self, tlk=None):
        if tlk is not None:
            tlk.synchronize()
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def close(self):
        if self.comm is not None:
            self.comm.close()
        if self.world > 1:
            self.dist.destroy_process_group()


GRAD_FLOOR = 1e-4  # see grad_err


def grad_err(g, ref, floor=GRAD_FLOOR):
    """max_i |g_i - ref_i| / max(|ref_i|, floor * |ref|_inf).  BASELINE.md 4.5 uses floor = 1e-6, which the small parity cases of
    tests/ keep.  At the sizes of this benchmark a branch gradient is a sum over thousands of patterns of terms of both signs, and
    the reference itself forms the per-pattern weights as w_k / exp(pattern_lk[k]) (treelikelihood.c:3207-3210): |lnL_k| ulps of
    noise per term (3e-14 at lnL_k = -250).  A branch whose gradient nearly cancels carries that as more than 1e-10 of its own value
    (two pattern orders of the CPU oracle differ by up to 8e-11 there), so entries below 1e-4 of the largest are compared relative
    to that floor; the strict-floor figure is reported next to it."""
    scale = np.maximum(np.abs(ref), np.abs(ref).max() * floor)
    return float(np.max(np.abs(g - ref) / np.where(scale == 0, 1.0, scale)))


def build_tlk(run, cfg, topo, m, rates, props, patterns, weights, kernels="auto"):
    phb = run.phb
    from physher_b200.treelikelihood import OPT_KERNELS

    tlk = phb.SingleTreeLikelihood(topo.left, topo.right, topo.root, cfg["states"], cfg["cats"], patterns.shape[1], use_tip_states=True,
                                   device=run.local_rank)
    tlk.set_tip_states(patterns)
    tlk.set_pattern_weights(weights)
    tlk.set_eigen(m.evec, m.eval, m.ivec)
    tlk.set_frequencies(m.freqs)
    tlk.set_site_model(rates, props)
    tlk.set_option(OPT_KERNELS, {"auto": phb.KERNELS_AUTO, "generic": phb.KERNELS_GENERIC, "fused": phb.KERNELS_FUSED}[kernels])
    tlk.initialize_gradient(phb.FLAG_TREE_MODEL)
    return tlk


def parity_gate(run, cfg, kernels, cores, sample_patterns, iters):
    """cpu_baseline leg + parity gate (rank 0): the unmodified reference (oracle/_ref) evaluates a bounded sample of this workload on
    the host cores -- timed, and its lnL / branch gradients of the first shard are the answers the device path must reproduce on
    the same patterns before any of its timings is reported."""
    from oracle import oracle as O

    if not O.reference_available():
        return ({"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref not built"},
                {"ok": None, "note": "no reference on this box: parity is covered by tests/ only"})
    T = cfg["taxa"]
    via = None
    if cfg["model"].startswith("HKY"):
        # The reference evaluates HKY through closed-form p_t / dp_dt (hky.c:230-400); the device path (and the oracle) build P(t) from
        # the eigen system like the reference's GTR.  Both are correct to an ulp of the LARGE entries of P, i.e. 1e-14 relative on the
        # small ones, and a branch whose gradient is a near-cancelling sum (|g| ~ 1e-5 of the largest entry) carries that as up to
        # 1e-9 of ITS value (measured on this workload: 8e-10 on one branch of 999 at 256 patterns, 7e-11 at 4096; every other branch
        # < 1e-10).  The gate therefore runs the reference on the same model written as a GTR -- its own eigen path.
        cfg = dict(cfg, ref_model="gtr_as_hky")
        via = "the reference's GTR eigen path with HKY's exchangeabilities (its closed-form HKY differs from ANY eigen form by up to 1e-9 on near-zero branch gradients)"
    r = run_reference(cfg, cores, sample_patterns, iters=iters, want_values=True)
    base = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "reference",
            "sample": f"{cores} single-threaded reference process(es) x {r['per']} patterns each, {iters} lnL+gradient evaluations each "
                      f"({cfg['model']}, {T} taxa, tip partials, SSE on), {r['wall']:.1f} s wall",
            "one_core_value": float(np.mean([p * r['nodes'] / s for s, p in zip(r['sec_per_eval'], r['patterns'])]))}
    v = r["values"]
    ref_lnl, ref_grad, ref_scaled = v["lnl"], v["grad"], v["rescaled"]
    phb = run.phb
    from physher_b200.treelikelihood import OPT_KERNELS

    S, C = cfg["states"], cfg["cats"]
    patterns = np.ascontiguousarray(v["tip_states"], dtype=np.uint8)
    root, right = v["root"], v["right"]
    tlk = phb.SingleTreeLikelihood(v["left"], v["right"], root, S, C, patterns.shape[1], use_tip_states=True, device=run.local_rank)
    tlk.set_tip_states(patterns)
    tlk.set_pattern_weights(v["weights"])
    tlk.set_eigen(v["evec"], v["eval"], v["ivec"])
    tlk.set_frequencies(v["freqs"])
    tlk.set_site_model(v["rates"], v["props"])
    tlk.set_option(OPT_KERNELS, {"auto": phb.KERNELS_AUTO, "generic": phb.KERNELS_GENERIC, "fused": phb.KERNELS_FUSED}[kernels])
    bl = np.asarray(v["bl"], dtype=np.float64)
    tlk.set_branch_lengths(bl)
    B = int(cfg.get("batch", 1))
    if B > 1:  # the batched entry point: sample 0 carries the reference's branch lengths
        bls = np.stack([bl, bl * 1.1])
        lnls, grads = tlk.gradient_batch(bls)
        lnl, g = float(lnls[0]), grads[0]
    else:
        g = tlk.gradient()
        lnl = tlk.calculate()
    family = {1: "generic", 2: "fused 4-state walk", 3: "FP64 tensor cores"}.get(tlk.last_kernels(), "?")
    tlk.close()
    g = g.copy()
    ref_grad = ref_grad.copy()
    ref_grad[root] = ref_grad[right[root]] = 0.0
    le = abs(lnl - ref_lnl) / abs(ref_lnl)
    ge = grad_err(g, ref_grad)
    par = {"ok": bool(le < PARITY_RTOL and ge < PARITY_RTOL), "lnl_rel_err": le, "grad_err": ge, "rtol": PARITY_RTOL, "patterns": int(patterns.shape[1]),
           "grad_metric": f"max_i |g_i - ref_i| / max(|ref_i|, {GRAD_FLOOR:g} |ref|_inf)", "grad_err_floor_1e-6": grad_err(g, ref_grad, 1e-6),
           "against": "unmodified reference (oracle/_ref), TREE_MODEL gradient, include_root_freqs = false, on the inputs as the reference holds them",
           "reference_rescaled": ref_scaled, "kernels": family}
    if via:
        par["reference_model"] = via
    return base, par


def roofline_record(name, cfg, P, B, kms, kernels, lib_version, cherries=0):
    T, S, C = cfg["taxa"], cfg["states"], cfg["cats"]
    sized = dict(cfg, patterns=P)
    peak, peak_src = measured_peak_gbs()
    alg = algorithmic_bytes(sized) * B  # one launch processes the whole batch
    achieved = alg / (kms * 1e-3) / 1e9 if kms > 0 else None
    fused = kernels != "generic" and S == 4
    tensor = kernels != "generic" and S in (20, 61)
    traffic = measured_traffic(name, kernels, P, lib_version)
    hbm = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
           "traffic": traffic, "peak_source": peak_src, "kernel_ms": kms, "algorithmic_bytes_per_launch": alg}
    if traffic and kms > 0:
        hbm["traffic_GBs"] = traffic / (kms * 1e-3) / 1e9
        hbm["traffic_frac"] = hbm["traffic_GBs"] / peak
    if fused:
        fused_bytes = float(P) * B * (2 * (T - 1) * C * S * 8 + 2 * T)  # what the fused walk must move: lower rows out and back, tip codes twice
        hbm.update(kernel="k_nuc4_walk<C=%d,scale=0,grad=1>" % C, fused_min_bytes_per_launch=fused_bytes,
                   fused_min_frac=(fused_bytes / (kms * 1e-3) / 1e9 / peak) if kms > 0 else None,
                   note="achieved = SURVEY.md 8d streaming-model bytes / kernel time; the fused walk keeps upper partials on chip, so it moves "
                        f"~{fused_bytes/1e9:.1f} GB per launch and frac can exceed 1; fused_min_frac (what the kernel must move / time / peak) and "
                        "traffic_frac (ncu dram bytes, when a capture of this kernel revision is committed) are the real DRAM utilisation")
        return hbm
    if tensor:
        flops = algorithmic_flops(sized)
        tpeak, tsrc = dmma_peak()
        tf = flops / (kms * 1e-3) / 1e12 if kms > 0 else None
        rec = {"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": (tf / tpeak) if tf else None, "traffic": traffic,
               "peak_source": tsrc, "kernel": "k_dmma_* (FP64 mma.sync m8n8k4, message form, branch gradients in adjoint form), all launches of one evaluation",
               "kernel_ms": kms, "algorithmic_flops_per_launch": flops, "hbm": hbm,
               "note": "launch = the kernel sequence of one evaluation; S=20 sits at the FP64 ridge so the HBM view is given too"}
        if S == 20:  # whole-tree walk (phb_dwalk.cu): every message row crosses HBM once each way, upper partials stay in shared memory
            walk_bytes = float(P) * B * ((2 * T - 3) * C * S * 8 + 2 * T)
            rec["kernel"] = "k_dwalk_post + k_dwalk_pre (whole-tree walk on the FP64 tensor cores, mma.sync m8n8k4, TMA bulk copies), both launches of one evaluation"
            hbm.update(fused_min_bytes_per_launch=walk_bytes, fused_min_frac=(walk_bytes / (kms * 1e-3) / 1e9 / peak) if kms > 0 else None)
            rec["note"] = ("launch = the two walk launches (+ root integration) of one evaluation; the walk moves ~%.1f GB where the streaming model "
                           "(hbm.algorithmic_bytes_per_launch) counts %.1f GB, so the path is bound by the FP64 pipe, which DMMA and the element-wise "
                           "products share" % (walk_bytes / 1e9, alg / 1e9))
        elif P >= 4 * (S + 1) ** 2 and T > 2:
            # message form: 3 dense products per non-root internal node and pattern (P_n L_n, P_n U_n, U_n (f o dP_n)), padded to 64 states;
            # cherries are evaluated once per PAIR of tip states and looked up per pattern (k_dmma_cherry_*), their products are not executed
            executed = 2.0 * 64 * 64 * 3 * (T - 2 - cherries) * C * P
            rec.update(executed_tensor_flops_per_launch=executed, executed_frac=(executed / (kms * 1e-3) / 1e12 / tpeak) if kms > 0 else None,
                       cherries=int(cherries))
            rec["note"] = ("launch = the kernel sequence of one evaluation.  frac is on the ALGORITHMIC flops (SURVEY.md 8d: four S x S mat-vecs per internal "
                           "operand); the message form executes three products per internal node, and the %d cherries of this tree are evaluated once per "
                           "pair of tip states ((S+1)^2 = %d pairs against %d patterns) instead of per pattern: executed_frac is what the tensor pipe "
                           "really issues (padded to 64 states) over the measured DMMA peak" % (cherries, (S + 1) ** 2, P))
        return rec
    hbm.update(kernel="generic node-at-a-time kernels, all levels of one evaluation")
    return hbm


def run_config(run, name, cfg, K, W, kernels="auto", strong=False, full_cpu_baseline=False, gate=True, outputs=None):
    """One BASELINE config on this invocation's GPUs: device-resident throughput, end-to-end throughput through the C ABI with host
    buffers, the live kernel time for the roofline, clocks, and the parity gate against the reference on a bounded sample.
    outputs[name] receives the arrays the last timed end-to-end step returned to its caller."""
    torch = run.torch
    from physher_b200.treelikelihood import OPT_TIMING

    world, rank = run.world, run.rank
    T, S, C = cfg["taxa"], cfg["states"], cfg["cats"]
    N = 2 * T - 1
    B_total = int(cfg.get("batch", 1))
    P_total = cfg["patterns"] * (1 if strong or B_total > 1 else world)
    if B_total > 1:  # batched samples: shard the SAMPLES across ranks (SURVEY.md 8e), no collective on the data path
        B = (B_total * (rank + 1)) // world - (B_total * rank) // world
        P = cfg["patterns"]
        sharding = f"{B_total} samples over {world} GPUs ({B} on rank 0), patterns replicated" if world > 1 else "single GPU"
    elif strong:
        P = (cfg["patterns"] * (rank + 1)) // world - (cfg["patterns"] * rank) // world
        B = 1
        sharding = f"{cfg['patterns']} patterns split over {world} GPUs (strong scaling)" if world > 1 else "single GPU"
    else:
        P, B = cfg["patterns"], 1
        sharding = f"{P} patterns per GPU x {world} (weak scaling)" if world > 1 else "single GPU"
    rec = {"workload": workload_name(dict(cfg, patterns=P_total)).replace(" per GPU", " in total"), "taxa": T, "patterns_total": int(P_total),
           "patterns_per_gpu": int(P), "states": S, "categories": C, "model": cfg["model"], "samples_per_step": B_total, "sharding": sharding,
           "scaling": "strong" if (strong or B_total > 1) else "weak", "n_gpus": world}

    cpu, par = None, None
    if rank == 0 and gate:
        try:
            cores = min(os.cpu_count() or 1, 32) if full_cpu_baseline else 1
            sample = sample_per_core(cfg) * cores if full_cpu_baseline else PARITY_PATTERNS.get(S, 64)
            cpu, par = parity_gate(run, cfg, kernels, cores, sample, iters=3 if full_cpu_baseline else 1)
        except Exception as exc:  # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {exc!r}"}
            par = {"ok": None, "note": f"gate did not run: {exc!r}"}
    ok = run.reduce([0.0 if (par is not None and par.get("ok") is False) else 1.0], "max" if world == 1 else "sum")[0]
    if world > 1:
        ok = 1.0 if ok >= world else 0.0
    if cpu is not None:
        rec["cpu_baseline"], rec["parity"] = cpu, par
    if not ok:
        rec["error"] = "parity gate failed: the device path does not reproduce the reference on the sample; no timing reported"
        return rec

    topo, bl, m, rates, props, patterns, weights = make_inputs(dict(cfg, patterns=P), 0 if B_total > 1 else rank)
    rec["inputs_sha256"] = inputs_sha256(topo, bl, m, rates, props, patterns, weights) if rank == 0 else None
    tlk = build_tlk(run, cfg, topo, m, rates, props, patterns, weights, kernels)
    ext = torch.cuda.ExternalStream(tlk.stream(), device=torch.device("cuda", run.local_rank))
    rng = np.random.default_rng(7)
    last = {}

    def new_bl():
        # every step sees new branch lengths (host buffer), like an optimiser / VI iteration would produce; the same on every rank
        b = bl * rng.uniform(0.98, 1.02, size=bl.shape)
        b[topo.root] = 0.0
        b[topo.right[topo.root]] = 0.0
        return b

    def step_batch():
        """BASELINE config 3: B branch-length samples (base x LogNormal(0, 0.1)) per step through phb_tlk_gradient_batch --
        host buffers in ([B][N] doubles) and out (lnl[B], grad[B][N]); one fused launch for the whole batch."""
        bls = bl[None, :] * rng.lognormal(0.0, 0.1, size=(B, N))
        bls[:, topo.root] = 0.0
        bls[:, topo.right[topo.root]] = 0.0
        lnls, grads = tlk.gradient_batch(bls)
        last.update(lnl=lnls, grad=grads)
        return float(lnls[-1]), grads[-1]

    def step_e2e():
        """The call a user makes, host in / host out: H2D of the branch lengths, the evaluation, (N > 1: the library's NCCL all-reduce
        on the same stream,) D2H of lnL + gradient."""
        if B_total > 1:
            return step_batch()
        tlk.set_branch_lengths(new_bl())
        if world == 1:
            g = tlk.gradient()
            lnl = tlk.calculate()
        else:
            lnl, g = tlk.gradient_allreduce(run.comm)
        last.update(lnl=lnl, grad=g)
        return lnl, g

    def step_device():
        """Device-resident step: inputs already in HBM, the (reduced) result left on the device; nothing waits on the host."""
        if B_total > 1:  # the batched entry point takes host buffers (2 x B x N doubles per step, ~1 MB each way at C3)
            step_batch()
        else:
            tlk.gradient_allreduce_device(run.comm)

    tlk.set_branch_lengths(bl)
    lnl = float("nan")
    for _ in range(W):
        lnl, g = step_e2e()
    if not np.isfinite(lnl):
        tlk.close()
        rec["error"] = f"non-finite lnL {lnl}"
        return rec
    for _ in range(W):
        step_device()
    run.sync(tlk)

    # ---- timed region 1: device-resident throughput ("value"), CUDA events on the launching stream
    tlk.set_option(OPT_TIMING, 1)
    launches0 = tlk.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(run.local_rank) as clocks:
        run.sync(tlk)
        e0.record(ext)
        for _ in range(K):
            step_device()
        e1.record(ext)
        run.sync(tlk)
        dev_ms = e0.elapsed_time(e1)
        launches = tlk.launch_count() - launches0
        kern_ms, kern_n = tlk.kernel_time()
        tlk.set_option(OPT_TIMING, 0)
        # ---- timed region 2: end to end through the public API with host buffers
        run.sync(tlk)
        t0 = time.perf_counter()
        for _ in range(K):
            lnl, g = step_e2e()
        run.sync(tlk)
        e2e_ms = (time.perf_counter() - t0) * 1e3 / K
    kms = kern_ms / max(kern_n, 1)
    step_ms, e2e_ms, kms_max = run.reduce([dev_ms / K, e2e_ms, kms], "max")
    total_pn = run.reduce([float(P) * N * B], "sum")[0]
    rec.update({
        "value": total_pn / (step_ms * 1e-3), "unit": UNIT, "steps": K, "warmup": W, "ms_per_step": step_ms,
        "evals_per_s": B_total * 1e3 / step_ms, "lnl": lnl,
        "e2e": {"value": total_pn / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": 8 * N * B, "d2h_bytes_per_step": 8 * (N + 1) * B,
                "evals_per_s": B_total * 1e3 / e2e_ms},
        "gpu_launches": int(launches), "launches_per_step": launches / K,
        "collective": (f"one ncclAllReduce(sum, double, {N + 2}) per step issued by libphysher_b200 on the evaluation's stream" if (world > 1 and B_total == 1)
                       else "none"),
        "clocks": clocks.summary(),
        "roofline": roofline_record(name, cfg, P, B, kms_max, kernels, run.phb.load_library().phb_version().decode(),
                                    cherries=int(np.sum((topo.left[T:] < T) & (topo.right[T:] < T)))),
        "l2": "per-evaluation working set exceeds the 126 MB L2; no explicit flush",
    })
    tlk.close()
    if outputs is not None:
        outputs[name] = last
    return rec


def run_c1(run, K, W, outputs=None):
    """BASELINE config 1 (examples/fluA JC69 strict-clock time tree: 69 taxa x 238 patterns, one rate category): a LATENCY workload.
    (a) single lnL + gradient evaluations through the C ABI with host buffers (what the glue does per model->logP / dlogP);
    (b) the ELBO shape of examples/fluA/JC69-time-ELBO.json: 100 reparameterised tree samples per step through
        phb_tlk_gradient_batch_time (heights, branch lengths, one fused launch, ratio / root-height / clock gradients).
    The reference's own known answers (tests/test_tree_likelihood.c:28-116, tests/golden/c1_kat.json) gate the record.
    outputs["c1"] receives what the last timed call of (a) and of (b) returned."""
    phb = run.phb
    gold = os.path.join(ROOT, "tests", "golden")
    z = dict(np.load(os.path.join(gold, "c1_jc69_fluA_tipstates.npz")))
    tt = dict(np.load(os.path.join(gold, "c1_time_tree.npz")))
    kat = json.load(open(os.path.join(gold, "c1_kat.json")))
    T, P = z["tip_states"].shape
    N = 2 * T - 1
    rec = {"workload": f"JC69 strict clock, fluA {T} taxa x {P} patterns (tests/data/jc69-time.json = the likelihood of examples/fluA/JC69-time-ELBO.json)",
           "taxa": int(T), "patterns_total": int(P), "states": 4, "categories": 1, "model": "JC69", "n_gpus": 1, "sharding": "rank 0 only (latency-bound, does not shard)"}
    tlk = phb.SingleTreeLikelihood(z["left"], z["right"], int(z["root"]), 4, 1, P, use_tip_states=True, device=run.local_rank)
    tlk.set_tip_states(z["tip_states"])
    tlk.set_pattern_weights(z["weights"])
    # JC69 as an eigen system: Q = (J - 4 I) / 3 is diagonalised by the 4 x 4 Hadamard matrix (entries +-1/2, exact in binary)
    vec = 0.5 * np.array([[1, 1, 1, 1], [1, 1, -1, -1], [1, -1, 1, -1], [1, -1, -1, 1]], dtype=np.float64)
    tlk.set_eigen(vec, np.array([0.0, -4.0 / 3.0, -4.0 / 3.0, -4.0 / 3.0]), vec)
    tlk.set_frequencies(z["freqs"])
    tlk.set_site_model(z["rates"], z["props"])
    tlk.set_option(phb.treelikelihood.OPT_UNROOTED, 0)
    tlk.initialize_gradient(phb.FLAG_TREE_MODEL)
    tlk.set_time_tree(tt["tip_heights"])
    bl = z["bl"].astype(np.float64)
    # gate: the reference's known answers
    tlk.set_branch_lengths(bl)
    lnl = tlk.calculate()
    l1, lj, gr, gc = tlk.gradient_batch_time(tt["ratios"][:1], tt["rates"][:1, None], include_jacobian=False)
    want = np.array(kat["ratio_grad"] + [kat["root_height_grad"]])
    le = abs(lnl - kat["logP"]) / abs(kat["logP"])
    ge = max(grad_err(gr[0], want), abs(gc[0, 0] - kat["rate_grad"]) / abs(kat["rate_grad"]), abs(l1[0] - kat["logP"]) / abs(kat["logP"]))
    rec["parity"] = {"ok": bool(le < PARITY_RTOL and ge < PARITY_RTOL), "lnl_rel_err": le, "grad_err": ge, "rtol": PARITY_RTOL,
                     "against": "known answers of the reference's tests/test_tree_likelihood.c:28-84 (lnL, clock-rate gradient, 67 ratio gradients, root height)"}
    if not rec["parity"]["ok"]:
        rec["error"] = "parity gate failed; no timing reported"
        tlk.close()
        return rec
    rng = np.random.default_rng(5)
    n_single = max(200, 10 * K)
    launches0 = tlk.launch_count()

    def single():
        tlk.set_branch_lengths(bl * rng.uniform(0.98, 1.02, size=N))
        g = tlk.gradient()
        return tlk.calculate(), g

    for _ in range(max(W, 10)):
        single()
    tlk.synchronize()
    with ClockSampler(run.local_rank) as clocks:
        t0 = time.perf_counter()
        for _ in range(n_single):
            l0, g0 = single()
        tlk.synchronize()
        single_ms = (time.perf_counter() - t0) * 1e3 / n_single
        launches = (tlk.launch_count() - launches0) / (n_single + max(W, 10))
        # (b) the ELBO batch
        Bs = 100
        ratios = np.clip(tt["ratios"][0][None, :] + rng.normal(0.0, 0.01, size=(Bs, T - 1)), 1e-3, 1 - 1e-3)
        ratios[:, -1] = tt["ratios"][0][-1] * rng.lognormal(0.0, 0.01, size=Bs)  # root height
        rates = tt["rates"][0] * rng.lognormal(0.0, 0.05, size=(Bs, 1))
        for _ in range(W):
            tlk.gradient_batch_time(ratios, rates, include_jacobian=True)
        t0 = time.perf_counter()
        for _ in range(K):
            lb, ljb, grb, gcb = tlk.gradient_batch_time(ratios, rates, include_jacobian=True)
        batch_ms = (time.perf_counter() - t0) * 1e3 / K
    pn = float(P) * N
    rec.update({
        "value": pn * 1e3 / single_ms, "unit": UNIT, "ms_per_step": single_ms, "evals_per_s": 1e3 / single_ms, "steps": n_single, "lnl": lnl,
        "timing": "wall clock around set_branch_lengths + gradient + calculate with host buffers (a latency workload: the host round trip IS the step)",
        "e2e": {"value": pn * 1e3 / single_ms, "unit": UNIT, "ms_per_step": single_ms, "evals_per_s": 1e3 / single_ms, "h2d_bytes_per_step": 8 * N, "d2h_bytes_per_step": 8 * (N + 1)},
        "launches_per_step": launches,
        "elbo_batch": {"samples_per_step": Bs, "ms_per_step": batch_ms, "sample_evals_per_s": Bs * 1e3 / batch_ms, "steps": K,
                       "call": "phb_tlk_gradient_batch_time (ratios, root height, clock rate in; lnL, log Jacobian, ratio / root-height / clock gradients out)",
                       "h2d_bytes_per_step": 8 * Bs * T, "d2h_bytes_per_step": 8 * Bs * (T + 2), "lnl_finite": bool(np.isfinite(lb).all())},
        "clocks": clocks.summary(),
        "roofline": {"bound": "latency", "note": "23 kB of tip codes and 137 nodes: launch + copy latency bound, no bandwidth roofline applies"},
    })
    tlk.close()
    if outputs is not None:
        outputs["c1"] = dict(lnl=l0, grad=g0, elbo_lnl=lb, elbo_log_jacobian=ljb, elbo_grad_ratios=grb, elbo_grad_rates=gcb)
    try:  # cpu_baseline leg: the reference's own evaluation of the same fixture on one host core
        from oracle import oracle as O

        if O.reference_available():
            devnull, saved = os.open(os.devnull, os.O_WRONLY), os.dup(1)
            os.dup2(devnull, 1)
            try:
                spec = json.load(open(os.path.join(gold, "c1_jc69_time.json")))["model"]
                ref = O.Reference(spec)
                ref.time_gradient(20, O.FLAG_TREE_MODEL | O.FLAG_BRANCH_MODEL, -1)
                sec = ref.time_gradient(200, O.FLAG_TREE_MODEL | O.FLAG_BRANCH_MODEL, -1)
                ref.close()
            finally:
                os.dup2(saved, 1)
                os.close(devnull)
            rec["cpu_baseline"] = {"value": pn / sec, "unit": UNIT, "evals_per_s": 1.0 / sec, "cores": 1, "kind": "reference",
                                   "sample": "200 lnL+gradient evaluations (tree + clock flags) of tests/data/jc69-time.json, tipstates as the fixture sets them, one core"}
            rec["elbo_batch"]["cpu_sequential_sample_evals_per_s"] = 1.0 / sec
    except Exception as exc:
        rec["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {exc!r}"}
    return rec


def dump_outputs(path, outputs):
    """outputs {config: {array: values}} -> path/<config>_<array>.npy in float64.  Inputs are seeded, so two builds run with the same
    arguments can be compared output for output.  Everything is per node or per sample (1.1 MB in all for the default records)."""
    os.makedirs(path, exist_ok=True)
    for config, arrays in outputs.items():
        for key, a in arrays.items():
            np.save(os.path.join(path, f"{config}_{key}.npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="headline workload (default: BASELINE configs[1])")
    ap.add_argument("--sub", default=None, help="comma list of further configs reported as sub-records under `configs` "
                                                "(default: all of c1,c2_1m,c3,c4,c5 for the default headline; 'none' to skip)")
    ap.add_argument("--sub-steps", type=int, default=None, help="timed steps of each sub-record (default: --steps)")
    ap.add_argument("--patterns", type=int, default=0, help="override patterns per GPU of the headline workload")
    ap.add_argument("--kernels", default="auto", choices=["auto", "generic", "fused"])
    ap.add_argument("--strong", action="store_true", help="headline: split --config's patterns over the GPUs instead of weak scaling")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of every record returned (lnL, gradients) as DIR/<config>_<array>.npy, float64")
    args = ap.parse_args()
    if args.sub_steps is None:
        args.sub_steps = args.steps
    if args.steps < 1 or args.sub_steps < 1:
        ap.error("--steps and --sub-steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    if args.patterns:
        cfg["patterns"] = args.patterns
    if args.impl == "reference":
        return reference_main(args, cfg)

    run = Run()
    W, K = max(args.warmup, 3), args.steps
    outputs = {}
    head = run_config(run, args.config, cfg, K, W, kernels=args.kernels, strong=args.strong, full_cpu_baseline=(run.world == 1),
                      gate=not args.no_cpu_baseline, outputs=outputs)
    if args.sub is None:
        subs = SUB_CONFIGS if (args.config == "c2" and not args.patterns and args.kernels == "auto") else []
    else:
        subs = [] if args.sub in ("none", "") else [s.strip() for s in args.sub.split(",")]
    records = {}
    for name in subs:
        t0 = time.perf_counter()
        try:
            if name == "c1":
                if run.rank == 0:
                    records[name] = run_c1(run, args.sub_steps, W, outputs=outputs)
                run.sync()
            else:
                records[name] = run_config(run, name, dict(CONFIGS[name]), args.sub_steps, W, strong=True, gate=not args.no_cpu_baseline,
                                           outputs=outputs)
        except Exception as exc:  # a sub-record must not take the headline down
            records[name] = {"error": repr(exc)}
            if run.world > 1:
                raise
        if name in records:
            records[name]["wall_s"] = time.perf_counter() - t0
    if args.dump_outputs and run.rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    if "error" in head:
        if run.rank == 0:
            print(json.dumps({"metric": METRIC, "value": None, "unit": UNIT, "n_gpus": run.world, "error": head["error"], "parity": head.get("parity")}))
        run.close()
        return 1
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": run.world, "steps": K, "warmup": W, "ms_per_step": head["ms_per_step"],
        "higher_is_better": True, "scaling": head["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(cfg), "taxa": cfg["taxa"], "patterns_per_gpu": head["patterns_per_gpu"], "states": cfg["states"],
                   "categories": cfg["cats"], "model": cfg["model"], "kernels": args.kernels, "l2": head["l2"], "sharding": head["sharding"],
                   "samples_per_step": head["samples_per_step"], "inputs_sha256": head["inputs_sha256"]},
        "evals_per_s": head["evals_per_s"], "lnl": head["lnl"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
        "collective": head["collective"], "clocks": head["clocks"], "roofline": head["roofline"],
    }
    if "cpu_baseline" in head:
        line["cpu_baseline"], line["parity"] = head["cpu_baseline"], head["parity"]
    if records:
        line["configs"] = records
    if run.rank == 0:
        print(json.dumps(line))
    run.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
