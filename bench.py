#!/usr/bin/env python
"""bench.py -- site-pattern conditional-likelihood updates per second (BASELINE.json's metric).

Default workload (N=1): BASELINE.json configs[1] AS WRITTEN -- ONE analysis of primates.nex, 4-state
GTR+G4, nruns=2 x nchains=4, all 8 chains on one B200: every generation one proposal per chain, the 8
chains evaluated in ONE chain-batched engine call = one fused kernel launch (P(t) rebuild for the dirty
branches, pruning over the dirty nodes with the rescaler fused, root integration, lnL reduction), the
accept step, and the Metropolis-coupling swap attempt (MC^3 shard coordinator, include/mb200_mc3.h).
A *step* is G generations (--generations-per-step, default 512) so that the timed region is >= 100 ms
whatever --steps is.  Site patterns, pattern weights and the GTR eigensystem are the reference's own
(tests/golden: MrBayes' compressed matrix of primates.nex, 413 patterns / 898 sites); proposals are
synthetic but MCMC-shaped (a branch move dirties one P(t) and the path to the root, 15 % of the moves
dirty the whole tree, 30 % are accepted, rejects undo the index flips on the host).

Under torchrun (N > 1) the SAME analysis grows to nruns = 2N: the reference's chain -> process map
(contiguous blocks, src/mcmc.c:18331) then gives every GPU two whole runs, all swap pairs are
co-resident, and the only collective is the end-of-run reduce (weak scaling, one process per GPU).
--workload codon20k / cynmix shard ONE run's heated chains over the GPUs (BASELINE configs[3] / [4]):
there the swap exchange crosses GPUs every generation (ncclAllGather of {lnL, lnPrior, chainId},
overlapped with the next generation's likelihood launches).

Legs (timed regions run in C, mrbayes_b200/host/mb200_host_loop.c, a plain client of the C-ABI):
  value     job descriptors resident in HBM (mb200_replay_begin/_end), results polled from pinned host
            memory, accept + swap logic on the host: per-step device time from CUDA events, L2 flushed
            between steps (256 MB memset), MAX over ranks
  e2e       the reference-facing C-ABI with HOST structs (mb200_evaluate_begin/_end: pack, launch with the
            job in the kernel parameter block, 16-byte result records written into pinned host memory)
  roofline  algorithmic bytes per launch of the fused pruning kernel / its event-timed duration
  cpu_baseline  the unmodified reference (oracle/_ref, FMA build) on the same workload, one process
            (the reference has no threads; MPI is not installed), bounded sample

--impl reference times the reference's own CPU path on this arm's config (one serial process per
analysis: N processes under torchrun, rank 0 runs them all).

--dump-outputs DIR writes what the value and e2e legs computed in their last timed step (every chain's lnL
in every generation, the chains' state after it, the coordinator's heats and swap counters) as
DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output (see dump_outputs).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "site-pattern CL updates/sec (node*pattern*rate)"
UNIT = "CL updates/s"
GOLD = ROOT / "tests" / "golden" / "primates_gtr_g4_fma.gold.gz"
GOLD_CYNMIX = ROOT / "tests" / "golden" / "cynmix_full_fma.gold.gz"
REF_BIN = ROOT / "oracle" / "_ref" / "mb_b200"
REF_DATA = ROOT / "oracle" / "_ref" / "data"


def bytes_per_update(S: int, K: int) -> float:
    """SURVEY 8d: fp32, two child vectors read + one written (12 S bytes) + scalers (12 / K bytes)."""
    return 12.0 * S + 12.0 / K


# ------------------------------------------------------------------------------ workloads
def primates_partition(n_chains: int, trees):
    """primates.nex as MrBayes compressed it, GTR+G4 eigensystem of the reference's own run."""
    from mrbayes_b200 import abi, records, workloads
    divs, events = records.load(GOLD)
    d = divs[0]
    eig = next(e for e in events if e.kind == "eigen")
    first = next(e for e in events if e.kind == "eval").spec
    masks = np.stack([d.tips[t] for t in range(d.cfg["tip_count"])])
    pr = workloads.Problem(4, 4, d.cfg["pattern_count"], n_chains, trees, masks, d.weights[0], first.freqs,
                           eig.V, eig.Vinv, eig.lam, first.rates, 0.0, flags=abi.FLAG_NUC4_PINVAR_QUIRK)
    pr.allocate()
    return pr


def cynmix_partitions(n_chains: int, trees):
    """cynmix.nex, the file's own 5-partition model: morphology Mk+G4 (variable-state kernels) + four
    GTR+I+G4 DNA partitions; data, pattern tables and eigensystems from the reference's own run."""
    from mrbayes_b200 import abi, records, workloads
    divs, events = records.load(GOLD_CYNMIX)
    parts = []
    for di in sorted(divs):
        d = divs[di]
        first = next(e.spec for e in events if e.kind == "eval" and e.division == di)
        masks = np.stack([d.tips[t] for t in range(d.cfg["tip_count"])])
        if d.pattern_states is not None:
            ps = d.pattern_states
            S = d.cfg["state_count"]
            pr = workloads.StdProblem(S, d.cfg["category_count"], d.cfg["pattern_count"], n_chains, trees, masks, d.weights[0],
                                      first.freqs, np.zeros((S, S)), np.zeros((S, S)), np.zeros(S), first.rates, 0.0, flags=0,
                                      state_counts=ps["state_counts"], matrix_offsets=ps["matrix_offsets"],
                                      freq_offsets=ps["freq_offsets"], matrix_length=ps["matrix_length"],
                                      dummy=ps["dummy_patterns"], uncompressed=ps["uncompressed_sites"])
        else:
            eig = next(e for e in events if e.kind == "eigen" and e.division == di)
            p_inv = 0.1
            pr = workloads.Problem(4, 4, d.cfg["pattern_count"], n_chains, trees, masks, d.weights[0], first.freqs,
                                   eig.V, eig.Vinv, eig.lam, first.rates * (1.0 - first.p_invar), p_inv,
                                   flags=abi.FLAG_NUC4_PINVAR_QUIRK)
        pr.allocate()
        parts.append(pr)
    return parts


def synthetic_partition(name: str, n_chains: int, trees, seed: int):
    from mrbayes_b200 import abi, workloads
    S, K, C, tips = SYNTH[name]
    rng = np.random.default_rng(seed)
    pi, V, Vinv, lam = workloads.reversible_model(S, rng)
    rates = workloads.discrete_gamma_rates(0.5, K)
    masks = workloads.random_masks(tips, C, S, rng, 0.02, 0.0)
    weights = np.ones(C, np.float32)
    flags = abi.FLAG_NUC4_PINVAR_QUIRK if S == 4 else abi.FLAG_TIP_SHORTCUTS
    pr = workloads.Problem(S, K, C, n_chains, trees, masks, weights, pi, V, Vinv, lam, rates, 0.0, flags=flags)
    pr.allocate()
    return pr


SYNTH = {"nuc200k": (4, 4, 200_000, 32), "aa50k": (20, 4, 50_000, 64), "codon20k": (61, 1, 20_000, 32)}

# name -> (runs at N GPUs, chains per run at N GPUs, swaps per run and generation, generations per step,
#          taxa, scaling, description)
WORKLOADS = {
    "primates": dict(runs=lambda n: 2 * n, chains=lambda n: 4, swaps=1, gens=512, tips=12, scaling="weak",
                     text="primates.nex 4-state GTR+G4, nruns=2 nchains=4: all 8 chains on one GPU, one chain-batched launch per "
                          "generation (BASELINE configs[1]); N GPUs: nruns=2N, two whole runs per GPU"),
    "aa50k": dict(runs=lambda n: n, chains=lambda n: 4, swaps=1, gens=4, tips=64, scaling="weak",
                  text="synthetic 20-state WAG-like+G4 amino-acid alignment, 50k unique patterns, 64 taxa, nruns=1 nchains=4 per GPU "
                       "(BASELINE configs[2]: tensor-core CL path)"),
    "codon20k": dict(runs=lambda n: 1, chains=lambda n: 16, swaps=4, gens=16, tips=32, scaling="strong",
                     text="synthetic 61-state M0 codon alignment, 20k unique patterns, 32 taxa, nruns=1 nchains=16, the run's heated "
                          "chains sharded over the GPUs with the per-generation NCCL swap exchange (BASELINE configs[3])"),
    "cynmix": dict(runs=lambda n: 1, chains=lambda n: 32, swaps=8, gens=256, tips=32, scaling="strong",
                   text="cynmix.nex, 5 partitions (morphology Mk+G4 + 4 x GTR+I+G4), nruns=1 nchains=32, partitions x chains "
                        "sharded over the GPUs with the per-generation NCCL swap exchange (BASELINE configs[4])"),
    "nuc200k": dict(runs=lambda n: n, chains=lambda n: 2, swaps=1, gens=32, tips=32, scaling="weak",
                    text="synthetic 4-state GTR+G4 alignment, 200k unique patterns, 32 taxa, nruns=1 nchains=2 per GPU (streaming regime)"),
    # development / test workload: ONE run of primates whose 8 heated chains are dealt out over the processes
    "primates-sharded": dict(runs=lambda n: 1, chains=lambda n: 8, swaps=2, gens=256, tips=12, scaling="strong",
                             text="primates.nex 4-state GTR+G4, nruns=1 nchains=8, the run's heated chains sharded over the GPUs "
                                  "(development workload for the swap exchange)"),
}


class Job:
    """One analysis' share on this process: partitions (Problems with the local chains), engine instances,
    the pre-generated proposal cycle, the coordinator."""

    def __init__(self, name, rank, world, lib, device, cycle_len, seed=20260924, flags=0):
        from mrbayes_b200 import mc3, workloads
        w = WORKLOADS[name]
        self.name, self.rank, self.world, self.w = name, rank, world, w
        self.runs, self.chains = w["runs"](world), w["chains"](world)
        n_global = self.runs * self.chains
        if n_global % world != 0 or world > n_global:
            raise SystemExit(f"bench.py: {n_global} chains do not divide over {world} processes (src/mcmc.c:18338)")
        self.n_local = n_global // world
        self.first = rank * self.n_local
        self.globals = list(range(self.first, self.first + self.n_local))
        # one tree per GLOBAL chain, seeded by the chain, so that a chain's trajectory does not depend on
        # which process owns it; the partitions of a chain share its tree (linked branch lengths)
        # the chains of a run start from the run's common tree (like a real run after burn-in they sit at
        # comparable likelihoods, so that heat swaps are actually accepted) and then go their own way
        import copy
        # weak-scaling workloads (whole runs per GPU): every GPU gets the SAME two runs' trees and proposals (seeded by the
        # chain's index within its process), so that the work per GPU is exactly equal and value(N) / (N value(1)) measures
        # the machine, not the luck of the proposal draw; sharded workloads seed by the global chain (a chain's trajectory
        # must not depend on which process owns it)
        self.seed_ids = [(g - self.first) if w["scaling"] == "weak" else g for g in self.globals]
        trees = [copy.deepcopy(workloads.random_tree(w["tips"], np.random.default_rng([seed, s // self.chains]), mean_len=0.08))
                 for s in self.seed_ids]
        if name.startswith("primates"):
            self.parts = [primates_partition(self.n_local, trees)]
        elif name == "cynmix":
            self.parts = cynmix_partitions(self.n_local, trees)
        else:
            self.parts = [synthetic_partition(name, self.n_local, trees, seed)]
        self.insts = [p.create(lib, device=device, max_evaluations=self.n_local, flags=flags) for p in self.parts]
        self.cycle_len = cycle_len
        self.seed = seed
        self.mc = None
        self._build_cycle()

    # -- proposal cycle ---------------------------------------------------------------------
    def _lnprior(self, ch):
        return float(-10.0 * self.parts[0].tree[ch].length.sum())      # brlenspr = unconstrained:exp(10)

    def _build_cycle(self, p_full=0.15, p_accept=0.3):
        from mrbayes_b200 import workloads
        nl, parts = self.n_local, self.parts
        # initial full evaluation of every local chain on every partition
        lnl0 = np.zeros(nl)
        for pr, inst in zip(parts, self.insts):
            lnl, st = inst.evaluate([pr.full_evaluation(ch) for ch in range(nl)])
            assert not st.any() and np.isfinite(lnl).all()
            lnl0 += lnl
        self.lnl0 = lnl0
        self.lnpr0 = np.array([self._lnprior(ch) for ch in range(nl)])
        snaps = [workloads.snapshot(pr) for pr in parts]
        rngs = [np.random.default_rng([self.seed, 1, s]) for s in self.seed_ids]
        steps = [[None] * self.cycle_len for _ in parts]        # [part][step] -> list of specs (local chains)
        accept = np.zeros((self.cycle_len, nl), np.uint8)
        lnprior = np.zeros((self.cycle_len, nl))
        for i in range(self.cycle_len - 1):
            specs = [[] for _ in parts]
            for ch in range(nl):
                rng = rngs[ch]
                tr = parts[0].tree[ch]
                old = tr.length.copy()
                full = rng.random() < p_full
                node, new_len = None, None
                if not full:
                    node = int(rng.integers(0, tr.n_nodes))
                    while node == tr.root:
                        node = int(rng.integers(0, tr.n_nodes))
                    new_len = float(tr.length[node] * np.exp(0.5 * (rng.random() - 0.5)))
                ok = rng.random() < p_accept
                sps = []
                for pi, pr in enumerate(parts):
                    sp = pr.full_evaluation(ch) if full else pr.branch_update(ch, node, new_len)
                    specs[pi].append(sp); sps.append(sp)
                lnprior[i, ch] = self._lnprior(ch)
                accept[i, ch] = 1 if ok else 0
                if not ok:
                    for pr, sp in zip(parts, sps):
                        pr.reject(ch, sp, old)
            for pi in range(len(parts)):
                steps[pi][i] = specs[pi]
        # closing step: a whole-tree move, accepted, that lands every chain on the post-initialisation state
        for pi, pr in enumerate(parts):
            steps[pi][self.cycle_len - 1] = [workloads.reset_evaluation(pr, ch, snaps[pi]) for ch in range(nl)]
        accept[self.cycle_len - 1, :] = 1
        lnprior[self.cycle_len - 1, :] = self.lnpr0
        self.steps, self.accept, self.lnprior = steps, accept, lnprior
        C0, K0 = parts[0].C, parts[0].K
        self.updates_per_step = np.array([sum(len(sp.ops) * pr.C * pr.K for pr, st in zip(parts, steps) for sp in st[i])
                                          for i in range(self.cycle_len)], np.float64)
        self.bytes_per_step = np.array([sum(len(sp.ops) * pr.C * pr.K * bytes_per_update(pr.S, pr.K)
                                            for pr, st in zip(parts, steps) for sp in st[i]) for i in range(self.cycle_len)])
        self.nodes_per_eval = float(np.mean([len(sp.ops) for st in steps for s in st for sp in s]))
        del C0, K0

    # -- engine-side tables -----------------------------------------------------------------
    def prepare(self, mc):
        from mrbayes_b200 import abi
        self.mc = mc
        nP = len(self.parts)
        self.batches = [[inst.pack(self.steps[pi][i]) for i in range(self.cycle_len)] for pi, inst in enumerate(self.insts)]
        self.host_arrays = [[abi.make_eval_array(self.steps[pi][i]) for i in range(self.cycle_len)] for pi in range(nP)]
        self.c_parts = (C.c_int * nP)(*[i.handle for i in self.insts])
        self.c_batches = (C.c_int * (nP * self.cycle_len))(*[b for br in self.batches for b in br])
        self.c_steps = (C.c_void_p * (nP * self.cycle_len))(*[C.cast(a, C.c_void_p) for hr in self.host_arrays for a in hr])
        self.c_accept = np.ascontiguousarray(self.accept)
        self.c_lnprior = np.ascontiguousarray(self.lnprior)
        self.cur_lnl = self.lnl0.copy()
        self.cur_lnpr = self.lnpr0.copy()

    def run(self, hl, mode, order, swap_freq=1, trace=None):
        """-> (wall seconds, device ms, swaps accepted) for the generations in `order`; `trace`, if given, a float64
        array [len(order)][n_local] that receives every chain's lnL in every generation."""
        arr = (C.c_int * len(order))(*order)
        sums = (C.c_double * 2)()
        nacc = C.c_longlong(0)
        rc = hl.mb200_host_mc3_loop(self.mc.handle, self.c_parts, len(self.parts), self.n_local, mode,
                                    self.c_steps, self.c_batches, self.cycle_len,
                                    self.c_accept.ctypes.data_as(C.POINTER(C.c_ubyte)),
                                    self.c_lnprior.ctypes.data_as(C.POINTER(C.c_double)), arr, len(order), swap_freq,
                                    self.cur_lnl.ctypes.data_as(C.POINTER(C.c_double)),
                                    self.cur_lnpr.ctypes.data_as(C.POINTER(C.c_double)), sums, C.byref(nacc),
                                    None if trace is None else trace.ctypes.data_as(C.POINTER(C.c_double)))
        if rc != 0:
            raise RuntimeError(f"mb200_host_mc3_loop failed with code {rc}")
        return sums[0], sums[1], nacc.value

    def close(self):
        for i in self.insts:
            i.close()


def python_mc3_loop(job, mc, n_generations, gather=None):
    """The generation loop of mb200_host_mc3_loop restated in Python for the CPU tests (oracle instances,
    LOOPBACK coordinator; `gather(rows) -> table` is the transport, e.g. a gloo all_gather).
    -> final current lnL of the local chains."""
    cur_lnl, cur_lnpr = job.lnl0.copy(), job.lnpr0.copy()
    for g in range(n_generations):
        i = g % job.cycle_len
        lnl = np.zeros(job.n_local)
        for pi, inst in enumerate(job.insts):
            l, st = inst.evaluate(job.steps[pi][i])
            assert not st.any()
            lnl += l
        acc = job.accept[i].astype(bool)
        cur_lnl = np.where(acc, lnl, cur_lnl)
        cur_lnpr = np.where(acc, job.lnprior[i], cur_lnpr)
        mc.exchange_begin(cur_lnl, cur_lnpr)
        if gather is not None:
            mc.table()[:] = gather(mc.table()[mc.first:mc.first + mc.n_local].copy())
        mc.exchange_end()
        mc.attempt_swaps()
    return cur_lnl


def load_host_loop():
    from mrbayes_b200 import abi, mc3
    mc3.library()                                        # NCCL first (one copy per process)
    hl = C.CDLL(str(abi.ENGINE_LIB.parent / "libmb200_hostloop.so"))
    hl.mb200_host_mc3_loop.restype = C.c_int
    hl.mb200_host_mc3_loop.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p),
                                       C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_ubyte), C.POINTER(C.c_double),
                                       C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                       C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_double)]
    hl.mb200_host_generation_loop.restype = C.c_double
    hl.mb200_host_replay_loop.restype = C.c_double
    return hl


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-3:]]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        try:
            sm = sorted(float(r[1]) for r in rows)
            reasons = set()
            for r in rows:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                    "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}
        except (ValueError, IndexError):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": len(rows)}


# ------------------------------------------------------------------------------ reference arm
def usable_cores() -> int:
    """Host cores this process may actually use: the smaller of the CPU count, the scheduler affinity
    mask and the cgroup CPU quota (a container often sees every core of the machine but is capped)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError, IndexError):
        pass
    try:
        q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
        per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
        if q > 0 and per > 0:
            n = min(n, max(1, int(q / per + 0.5)))
    except (OSError, ValueError):
        pass
    return max(1, n)


AA = "ARNDCQEGHILKMFPSTWYV"
SENSE = [a + b + c for a in "TCAG" for b in "TCAG" for c in "TCAG" if a + b + c not in ("TAA", "TAG", "TGA")]


# the reference's pattern compression is quadratic in the number of columns (200 000 columns: 7 minutes before the first
# likelihood call): its CPU baseline for nuc200k runs on the first 20 000 columns (CL updates per second do not depend on it)
REF_COLUMNS = {"nuc200k": 20_000}


def write_synthetic_nexus(name: str, path: Path, seed: int = 7):
    """A NEXUS alignment of the synthetic workload's size for the reference binary: random residues
    (every column a distinct pattern with overwhelming probability; the reference compresses it itself)."""
    S, K, Cpat, tips = SYNTH[name]
    Cpat = REF_COLUMNS.get(name, Cpat)
    rng = np.random.default_rng(seed)
    with open(path, "w") as f:
        if S == 20:
            f.write(f"#NEXUS\nbegin data;\ndimensions ntax={tips} nchar={Cpat};\nformat datatype=protein gap=- missing=?;\nmatrix\n")
            lut = np.frombuffer(AA.encode(), np.uint8)
            for t in range(tips):
                f.write(f"t{t} " + lut[rng.integers(0, 20, Cpat)].tobytes().decode() + "\n")
        elif S == 61:
            f.write(f"#NEXUS\nbegin data;\ndimensions ntax={tips} nchar={3 * Cpat};\nformat datatype=dna gap=- missing=?;\nmatrix\n")
            cod = np.array(SENSE)
            for t in range(tips):
                f.write(f"t{t} " + "".join(cod[rng.integers(0, 61, Cpat)]) + "\n")
        else:
            f.write(f"#NEXUS\nbegin data;\ndimensions ntax={tips} nchar={Cpat};\nformat datatype=dna gap=- missing=?;\nmatrix\n")
            lut = np.frombuffer(b"ACGT", np.uint8)
            for t in range(tips):
                seq = lut[rng.integers(0, 4, Cpat)].tobytes().decode()
                # the reference's parser takes tokens of at most 99 990 characters (blanks inside a sequence are allowed)
                f.write(f"t{t} " + " ".join(seq[i:i + 50_000] for i in range(0, Cpat, 50_000)) + "\n")
        f.write(";\nend;\n")


def reference_commands(name: str, data: Path, nruns: int, nchains: int, ngen: int, seed: int, out: Path) -> str:
    head = f"set autoclose=yes nowarn=yes seed={seed} swapseed={seed};\nexecute {data};\n"
    tail = (f"mcmc nruns={nruns} nchains={nchains} ngen={ngen} printfreq=1000000 samplefreq=1000000 diagnfreq=1000000 "
            f"filename={out};\nquit;\n")
    if name.startswith("primates"):
        return head + "lset nst=6 rates=gamma ngammacat=4;\n" + tail
    if name == "cynmix":
        return head + ("set partition=favored;\nlset app=(1) rates=gamma;\nlset app=(2,3,4,5) rates=invgamma nst=6;\n"
                       "unlink revmat=(all) pinvar=(all) shape=(all) statefreq=(all);\nprset applyto=(all) ratepr=variable;\n") + tail
    if name == "aa50k":
        return head + "prset aamodelpr=fixed(wag);\nlset rates=gamma ngammacat=4;\n" + tail
    if name == "codon20k":
        return head + "lset nucmodel=codon;\n" + tail
    return head + "lset nst=6 rates=gamma ngammacat=4;\n" + tail


# reference sample sizes: (nruns, nchains, generations) bounded to roughly 10-30 s of one core
REF_SAMPLE = {"primates": (2, 4, 4000), "primates-sharded": (1, 8, 4000), "cynmix": (1, 4, 600), "aa50k": (1, 2, 4), "codon20k": (1, 4, 3), "nuc200k": (1, 2, 60)}


def reference_sample(name: str, n_procs: int, seed0: int, ngen_scale: float = 1.0):
    """n_procs concurrent serial reference processes on the workload; -> (sum of per-process kernel-only
    CL-updates/s, total CL updates, wall seconds, mean in-kernel seconds, description)."""
    nruns, nchains, ngen = REF_SAMPLE[name]
    ngen = max(1, int(ngen * ngen_scale))
    with tempfile.TemporaryDirectory() as td:
        tmp = Path(td)
        # the processes run in the temporary directory and see short relative names only: MrBayes refuses file names
        # longer than 99 characters
        data = tmp / f"{name}.nex"
        if name in SYNTH:
            write_synthetic_nexus(name, data)
        else:
            data.symlink_to(REF_DATA / ("primates.nex" if name.startswith("primates") else f"{name}.nex"))
        procs = []
        t0 = time.perf_counter()
        for i in range(n_procs):
            nex = tmp / f"p{i}.nex"
            nex.write_text(reference_commands(name, Path(data.name), nruns, nchains, ngen, seed0 + i, Path(f"p{i}")))
            env = dict(os.environ, MB200_MODE="cpu", MB200_REPORT=str(tmp / f"p{i}.json"))
            procs.append(subprocess.Popen([str(REF_BIN), nex.name], cwd=tmp, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
        for p in procs:
            p.wait()
        wall = time.perf_counter() - t0
        tot_rate, tot_upd, secs = 0.0, 0, []
        for i in range(n_procs):
            rep = json.loads((tmp / f"p{i}.json").read_text().strip().splitlines()[-1])
            tot_rate += rep["cl_updates"] / rep["sec_cpu"]
            tot_upd += rep["cl_updates"]
            secs.append(rep["sec_cpu"])
    cols = f" ({REF_COLUMNS[name]} of its columns)" if name in REF_COLUMNS else ""
    desc = (f"unmodified reference (gcc -O3 -mavx -mfma), {name}{cols}: nruns={nruns} nchains={nchains}, {ngen} generations, "
            f"{n_procs} process(es): {tot_upd} CL updates, {float(np.mean(secs)):.2f} s inside LaunchLogLikeForDivision per process "
            f"({wall:.1f} s wall incl. reading and compressing the alignment)")
    return tot_rate, tot_upd, wall, float(np.mean(secs)), desc


def port_baseline(seconds: float):
    """Fallback CPU baseline when oracle/_ref did not travel: the oracle port replaying bench-shaped steps."""
    from mrbayes_b200 import abi
    lib = abi.oracle_library()
    job = Job("primates", 0, 1, lib, 0, 64)
    t0 = time.perf_counter(); upd = 0; n = 0
    for inst in job.insts:
        inst.set_arith(1)
    while time.perf_counter() - t0 < seconds:
        i = n % job.cycle_len
        job.insts[0].evaluate(job.steps[0][i]); upd += job.updates_per_step[i]; n += 1
    dt = time.perf_counter() - t0
    job.close()
    return upd / dt, f"oracle port, {n} generations x 8 chains in {dt:.1f} s"


def cpu_baseline(name: str):
    if REF_BIN.exists() and (name in SYNTH or (REF_DATA / "primates.nex").exists()):
        rate, upd, wall, sec, desc = reference_sample(name, 1, 12345)
        return {"value": rate, "unit": UNIT, "cores": 1, "kind": "reference", "sample": desc}
    val, sample = port_baseline(3.0)
    return {"value": val, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample}


def bench_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    w = WORKLOADS[name]
    world = max(1, args.gpus)
    base = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "higher_is_better": True,
            "scaling": w["scaling"], "vs_baseline": None, "dtype": "f32"}
    if not REF_BIN.exists():
        val, sample = port_baseline(2.0)
        line = dict(base, value=val, steps=args.steps, warmup=args.warmup, ms_per_step=None,
                    data="primates.nex patterns, synthetic proposals", config={"workload": w["text"] + " [oracle port: oracle/_ref missing]"},
                    cpu_baseline={"value": val, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
                    e2e={"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        print(json.dumps(line), flush=True)
        return
    # the same config as the engine arm: one serial process per analysis (the reference has no threads and MPI is
    # not installed here): weak-scaled workloads run `world` analyses, sharded ones a single one
    procs = world if w["scaling"] == "weak" else 1
    procs = max(1, procs)
    for _ in range(min(args.warmup, 1)):
        reference_sample(name, procs, 900, 0.1)
    steps = max(1, min(args.steps, 3))
    rates, walls, desc = [], [], ""
    for s in range(steps):
        r, u, wall, sec, desc = reference_sample(name, procs, 1000 + 100 * s, 1.0)
        rates.append(r); walls.append(wall)
    val = float(np.mean(rates))
    line = dict(base, value=val, steps=steps, warmup=min(args.warmup, 1), ms_per_step=1e3 * float(np.mean(walls)),
                data="the reference's own input and MCMC proposals" if name not in SYNTH else "synthetic alignment (random residues), the reference's own MCMC proposals",
                config={"workload": w["text"], "reference_build": "unmodified sources, gcc -O3 -std=c99 -mavx -mfma (FMA kernels)",
                        "processes": procs, "usable_host_cores": usable_cores(),
                        "timing": "time inside LaunchLogLikeForDivision (ld --wrap), summed rate over concurrent processes",
                        "note": "one serial process per analysis: the reference cannot use more than one core per analysis without MPI"},
                cpu_baseline={"value": val, "unit": UNIT, "cores": procs, "kind": "reference", "sample": desc},
                e2e={"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ engine arm
def measured_peaks():
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        return dict(json.loads(pk.read_text()), which="measured (MEASURED_PEAKS.json)")
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1650.0, "which": "fallback (B200_PROFILING.md)"}


def kernel_roofline(torch, job, flush, peaks, device, max_launches=1024):
    """Event-timed launches of the fused pruning kernel of partition 0 (L2 flushed before each), resident
    descriptors; -> roofline dict."""
    pi = int(np.argmax([p.C * p.K * p.S for p in job.parts]))          # the partition that dominates the step
    inst, pr = job.insts[pi], job.parts[pi]
    inst.set_kernel_timing(True)
    stream = torch.cuda.ExternalStream(inst.stream(), device=device)
    n = min(max_launches, job.cycle_len * max(1, max_launches // job.cycle_len))
    n = max(job.cycle_len, n - n % job.cycle_len)
    tot_bytes = 0.0
    with torch.cuda.stream(stream):
        for g in range(n):
            i = g % job.cycle_len
            flush.zero_()
            inst.replay(job.batches[pi][i])
            tot_bytes += sum(len(sp.ops) for sp in job.steps[pi][i]) * pr.C * pr.K * bytes_per_update(pr.S, pr.K)
    ms, cnt = inst.kernel_time()
    inst.set_kernel_timing(False)
    inst.synchronize()
    avg_s = ms * 1e-3 / max(cnt, 1)
    ach = (tot_bytes / max(cnt, 1)) / avg_s / 1e9
    kind = "eval_nuc4_kernel<K=4,NT=256,FUSE> (4-state shuffle kernel)" if pr.S == 4 else \
           f"eval_tcp_kernel<{pr.S}> (tcgen05, warp-specialised pipeline)" if pr.S in (20, 61) else "eval_gen_kernel"
    if len(job.parts) > 1:
        kind += f" of partition {pi + 1} of {len(job.parts)} (the largest)"
    return {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
            "traffic": None, "traffic_note": "per-launch DRAM bytes: see the ncu captures under profiles/ (the working set of a "
                                             "primates analysis, 2.7 MB, lives in L2; a constant here would not belong to this run)",
            "kernel": kind, "avg_kernel_us": avg_s * 1e6, "launches_timed": cnt,
            "algorithmic_bytes_per_launch": tot_bytes / max(cnt, 1), "bytes_per_update": bytes_per_update(pr.S, pr.K),
            "peak_source": peaks["which"]}


def full_tree_workload(torch, lib, name, peaks, device, with_cpu=True):
    """Large synthetic configs (working set >> L2): full-tree evaluations of one chain, whole evaluation
    (P(t) kernels + pruning) event-timed, device-resident and through the host-struct C-ABI call."""
    from mrbayes_b200 import workloads
    S, K, Cn, tips = SYNTH[name]
    pr = workloads.make_problem(S, K, Cn, tips, 1, seed=2026)
    with pr.create(lib, device=device) as inst:
        stream = torch.cuda.ExternalStream(inst.stream(), device=device)
        sp = pr.full_evaluation(0)
        inst.evaluate(sp)
        batch = inst.pack([pr.full_evaluation(0)])
        inst.set_kernel_timing(True)
        for _ in range(3):
            inst.replay(batch)
        inst.kernel_time()
        reps = 10
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            inst.replay(batch)
        b.record(stream)
        inst.synchronize()
        ms = a.elapsed_time(b) / reps
        kms, kn = inst.kernel_time()
        inst.set_kernel_timing(False)
        # end to end: host structs in, lnL out (pack + H2D of the job + launch + result)
        sp2 = pr.full_evaluation(0)
        inst.evaluate(sp2)
        t0 = time.perf_counter()
        for _ in range(reps):
            inst.evaluate(sp2)
        sec = (time.perf_counter() - t0) / reps
        upd = pr.n_int * pr.C * pr.K
        bpu = bytes_per_update(pr.S, pr.K)
        flops = upd * (4 * pr.S * pr.S + pr.S)
        ach = upd * bpu / (ms * 1e-3) / 1e9
        out = {"workload": f"{name}: S={pr.S} K={pr.K} C={pr.C} taxa={pr.n_tips}, full-tree evaluation (62/30 nodes), 1 chain, working set >> L2",
               "value": upd / (ms * 1e-3), "unit": UNIT, "ms_per_evaluation": ms,
               "e2e": {"value": upd / sec, "unit": UNIT, "ms_per_evaluation": sec * 1e3,
                       "api": "mb200_evaluate (host structs in, lnL out)"},
               "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                            "basis": "whole evaluation (P(t) kernels + pruning kernel), CUDA events on the instance's stream",
                            "pruning_kernel_ms": kms / max(kn, 1), "traffic": None,
                            "algorithmic_tflops": flops / (ms * 1e-3) / 1e12,
                            "tensor_frac_3xtf32": (3.0 * flops / (ms * 1e-3) / 1e12) / (0.5 * peaks.get("bf16_tflops", 1650.0)) if S in (20, 61) else None}}
    if with_cpu and REF_BIN.exists():
        try:
            rate, upd_c, wall, sec_c, desc = reference_sample(name, 1, 4321)
            out["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": 1, "kind": "reference", "sample": desc}
        except Exception as ex:                                             # noqa: BLE001
            out["cpu_baseline"] = {"error": repr(ex)}
    return out


def many_analyses(torch, lib, hl, device, flush, R=32, gens=1024):
    """Throughput regime (informational): R independent 8-chain primates analyses in flight on one GPU,
    one instance / stream / launch per analysis and generation."""
    from mrbayes_b200 import abi
    # MB200_CONFIG_THROUGHPUT (one CTA per evaluation walks its pattern tiles, P(t) built once) was measured here: 86 us per
    # generation against 75 us for one CTA per tile -- 256 CTAs leave half the SMs' warp slots empty; MB200_BENCH_THROUGHPUT=1 for the A/B
    tflag = abi.CONFIG_THROUGHPUT if os.environ.get("MB200_BENCH_THROUGHPUT") else 0
    jobs = [Job("primates", 0, 1, lib, device, 128, seed=20260924 + 1000 * (r + 1), flags=tflag) for r in range(R)]
    for j in jobs:
        j.batches = [[j.insts[0].pack(j.steps[0][i]) for i in range(j.cycle_len)]]
        j.host_arrays = [[abi.make_eval_array(j.steps[0][i]) for i in range(j.cycle_len)]]
    ids = (C.c_int * R)(*[j.insts[0].handle for j in jobs])
    bids = (C.c_int * (R * 128))(*[b for j in jobs for b in j.batches[0]])
    sptr = (C.c_void_p * (R * 128))(*[C.cast(a, C.c_void_p) for j in jobs for a in j.host_arrays[0]])
    order = [i % 128 for i in range(gens)]
    arr = (C.c_int * gens)(*order)
    warm = (C.c_int * 128)(*range(128))
    hl.mb200_host_replay_loop(ids, C.c_int(R), bids, C.c_int(128), warm, C.c_int(128), C.c_void_p(None), C.c_size_t(0))
    ms = hl.mb200_host_replay_loop(ids, C.c_int(R), bids, C.c_int(128), arr, C.c_int(gens), C.c_void_p(flush.data_ptr()), C.c_size_t(flush.numel()))
    lnl = np.zeros(8 * R); st = np.zeros(8 * R, np.int32)
    HT = max(1, min(8, R, usable_cores()))
    hl.mb200_host_generation_loop(ids, C.c_int(R), sptr, C.c_int(128), C.c_int(8), warm, C.c_int(128),
                                  lnl.ctypes.data_as(C.POINTER(C.c_double)), st.ctypes.data_as(C.POINTER(C.c_int)), C.c_int(HT))
    sec = hl.mb200_host_generation_loop(ids, C.c_int(R), sptr, C.c_int(128), C.c_int(8), arr, C.c_int(gens),
                                        lnl.ctypes.data_as(C.POINTER(C.c_double)), st.ctypes.data_as(C.POINTER(C.c_int)), C.c_int(HT))
    upd = sum(float(j.updates_per_step[i]) for j in jobs for i in order)
    for j in jobs:
        j.close()
    return {"analyses_in_flight": R, "chains": 8 * R, "value": upd / (ms * 1e-3), "ms_per_generation": ms / gens,
            "e2e": upd / sec, "e2e_ms_per_generation": sec * 1e3 / gens, "host_threads": HT, "unit": UNIT,
            "roofline_frac": upd * bytes_per_update(4, 4) / (ms * 1e-3) / 1e9 / measured_peaks()["hbm_gbs"],
            "note": f"{R} independent nruns=2 x nchains=4 analyses of primates.nex sharing one GPU (device-resident replay with the L2 "
                    f"flushed between generations; e2e: mb200_evaluate_begin/_end from {HT} host threads); the reference needs one host core per analysis"}


def bench_engine(args):
    import torch
    from mrbayes_b200 import abi, mc3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    peaks = measured_peaks()
    lib = abi.engine_library()
    if lib.fn("device_count")() < 1:
        raise SystemExit("bench.py: no sm_100 device; the engine has no CPU fallback")
    hl = load_host_loop()

    name = args.workload
    w = WORKLOADS[name]
    G = args.generations_per_step if args.generations_per_step > 0 else w["gens"]
    K, W = args.steps, max(args.warmup, 3)
    cycle_len = 128 if name in ("primates", "cynmix") else 16
    job = Job(name, rank, world, lib, local, cycle_len, flags=(abi.CONFIG_THROUGHPUT if os.environ.get("MB200_BENCH_THROUGHPUT") else 0))

    # ---- coordinator: its own NCCL communicator, id shipped through the launcher's process group ----
    nccl_id = None
    if world > 1:
        buf = torch.zeros(mc3.ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            buf.copy_(torch.frombuffer(bytearray(mc3.unique_id()), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        nccl_id = bytes(buf.cpu().numpy().tobytes())
    mc = mc3.Coordinator(rank=rank, world=world, device=local, num_runs=job.runs, chains_per_run=job.chains,
                         num_swaps=w["swaps"], chain_temp=0.1, swap_seed=12345, nccl_id=nccl_id)
    job.prepare(mc)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        for i in job.insts:
            i.synchronize()
        torch.cuda.synchronize()

    def run_steps(mode, n_steps, timed, record=None):
        """n_steps steps of G generations each, L2 flushed before every step; -> (device ms, wall s, updates, swaps).
        `record`, if given, a dict that receives what the last step computed: every chain's lnL in every generation
        and the chains' current lnL / log prior after it."""
        ms_tot = wall_tot = upd = 0.0
        nacc = 0
        g0 = 0
        for s in range(n_steps):
            order = [(g0 + g) % cycle_len for g in range(G)]
            g0 = (g0 + G) % cycle_len
            if timed:
                flush.zero_()
                torch.cuda.synchronize()
            trace = np.zeros((G, job.n_local)) if record is not None and s == n_steps - 1 else None
            wall, ms, acc = job.run(hl, mode, order, trace=trace)
            if trace is not None:
                record.update(lnl=trace, current_lnl=job.cur_lnl.copy(), current_lnprior=job.cur_lnpr.copy())
            ms_tot += ms; wall_tot += wall; nacc += acc
            upd += float(sum(job.updates_per_step[i] for i in order))
        # return to the cycle start so that the next leg replays the same generations
        if g0 != 0:
            job.run(hl, mode, [(g0 + g) % cycle_len for g in range(cycle_len - g0)])
        return ms_tot, wall_tot, upd, nacc

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- warm-up (untimed): W steps through both paths ----
    run_steps(1, min(W, 4), False)
    run_steps(0, 1, False)

    # ---- value: resident descriptors ----
    launches0 = sum(i.launch_count() for i in job.insts)
    coll0 = mc.collectives()
    barrier()
    t_clock0 = time.perf_counter()
    out_value, out_e2e = {}, {}
    ms_value, wall_value, updates, swaps_acc = run_steps(1, K, True, out_value if args.dump_outputs else None)
    barrier()
    launches = sum(i.launch_count() for i in job.insts) - launches0
    collectives = mc.collectives() - coll0
    # end of run: one double per run summed over the processes (marginal-likelihood reduce, src/mcmc.c:17246)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    run_sums = np.zeros(job.runs)
    for c, g in enumerate(job.globals):
        run_sums[g // job.chains] += job.cur_lnl[c]
    a.record()
    red = mc.reduce_sum(run_sums, 0)
    b.record(); torch.cuda.synchronize()
    ms_reduce = a.elapsed_time(b)
    ms_value += ms_reduce

    # ---- e2e: host structs through the C-ABI ----
    barrier()
    mc3_state = {"chain_id": np.array([mc.chain_id(g) for g in range(job.runs * job.chains)], np.float64),
                 "swap_info": mc.swap_info().astype(np.float64)} if args.dump_outputs else {}
    ms_e2e_dev, wall_e2e, updates_e2e, _ = run_steps(0, K, True, out_e2e if args.dump_outputs else None)
    barrier()
    t_clock1 = time.perf_counter()
    if rank == 0:
        sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank if world > 1 else None,
                     {**{f"value_{k}": v for k, v in out_value.items()}, **{f"e2e_{k}": v for k, v in out_e2e.items()},
                      **{f"mc3_{k}": v for k, v in mc3_state.items()}})

    # ---- reduce over ranks: MAX time, SUM work ----
    vals = torch.tensor([ms_value, wall_value * 1e3, wall_e2e * 1e3], dtype=torch.float64, device=dev)
    # accepted swaps: every process of a sharded run takes every decision (global count on each rank); whole runs per GPU count their own
    sums = torch.tensor([updates, float(launches), updates_e2e, float(swaps_acc) if w["scaling"] == "weak" else 0.0], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    ms_value, ms_wall_value, ms_e2e = (float(x) for x in vals.tolist())
    all_updates, all_launches, all_updates_e2e, swaps_sum = (float(x) for x in sums.tolist())
    if w["scaling"] == "weak":
        swaps_acc = swaps_sum
    decision_hash = mc.decision_hash()

    roof = kernel_roofline(torch, job, flush, peaks, local) if rank == 0 else None

    if rank == 0:
        clocks = sampler.summary(t_clock0, t_clock1)
        gens_total = K * G
        h2d = float(np.mean([sum(pack_bytes(job.steps[pi][i]).bytes for pi in range(len(job.parts))) for i in range(cycle_len)])) * G
        d2h = float(len(job.parts) * job.n_local * 16 * G)
        step_bytes = float(np.mean(job.bytes_per_step)) * G
        line = {
            "metric": METRIC, "value": all_updates / (ms_value * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_value / K, "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "f32",
            "data": ("primates.nex site patterns / weights / GTR eigensystem from the reference's own run (tests/golden); synthetic MCMC-shaped proposals"
                     if name.startswith("primates") else
                     "cynmix.nex patterns / state tables / eigensystems from the reference's own run (tests/golden); synthetic MCMC-shaped proposals"
                     if name == "cynmix" else "synthetic alignment and model of the named shape; synthetic MCMC-shaped proposals"),
            "config": {"workload": w["text"], "generations_per_step": G, "nruns": job.runs, "nchains": job.chains,
                       "chains_per_gpu": job.n_local, "partitions": len(job.parts),
                       "patterns": [p.C for p in job.parts], "rate_categories": [p.K for p in job.parts], "states": [p.S for p in job.parts],
                       "taxa": w["tips"], "mean_dirty_nodes_per_evaluation": job.nodes_per_eval, "cycle_generations": cycle_len,
                       "swaps_per_run_and_generation": w["swaps"],
                       "l2": "flushed before every timed step (256 MB memset); within a step the working set stays where a real run keeps it",
                       "sharding": ("whole runs per GPU (reference chain->process map): swap pairs co-resident, no data-path collective; "
                                    "end-of-run ncclReduce of per-run lnL sums in the timed region; every GPU's runs replay the same "
                                    "proposal cycle, so the work per GPU is exactly equal" if w["scaling"] == "weak" else
                                    "one run's heated chains dealt out over the GPUs in contiguous blocks; per swap generation one ncclAllGather of "
                                    "{lnL, lnPrior, chainId} per chain (24 B), overlapped with the next generation's launches; end-of-run ncclReduce")},
            "timed_region_ms": ms_value, "wall_ms_of_value_leg": ms_wall_value,
            "e2e": {"value": all_updates_e2e / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / K, "us_per_generation": ms_e2e * 1e3 / gens_total,
                    "api": "mb200_evaluate_begin / _end per partition and generation (C-ABI, host structs in, one lnL per chain out), "
                           "accept step and mb200_mc3 swap attempt on the host, C generation loop (mrbayes_b200/host/mb200_host_loop.c)"},
            "gpu_launches": int(all_launches),
            "mc3": {"swap_attempts": int(gens_total * job.runs * w["swaps"]), "swaps_accepted_value_leg": int(swaps_acc),
                    "allgathers_in_value_leg": int(collectives), "end_of_run_reduce_ms": ms_reduce,
                    "decision_hash": f"{decision_hash:016x}", "run0_cold_sum": float(red[0])},
            "us_per_generation": ms_value * 1e3 / gens_total,
            "roofline": dict(roof, step_achieved_gbs_per_gpu=step_bytes * K / (ms_value * 1e-3) / 1e9,
                             step_frac_per_gpu=step_bytes * K / (ms_value * 1e-3) / 1e9 / peaks["hbm_gbs"]),
            "clocks": clocks,
        }
        if clocks.get("samples", 0) < 3:
            clocks["note"] = "timed region shorter than three 100 ms samples; nearest samples used"
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(name)
        if world == 1 and not args.no_extras and name == "primates":
            try:
                line["many_analyses"] = many_analyses(torch, lib, hl, local, flush)
            except Exception as ex:                                          # noqa: BLE001
                line["many_analyses"] = {"error": repr(ex)}
            line["other_workloads"] = []
            for n in [x for x in args.other.split(",") if x]:
                try:
                    line["other_workloads"].append(full_tree_workload(torch, lib, n, peaks, local, with_cpu=not args.no_cpu_baseline))
                except Exception as ex:                                      # noqa: BLE001
                    line["other_workloads"].append({"workload": n, "error": repr(ex)})
        print(json.dumps(line), flush=True)
    job.close()
    mc.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir, rank, arrays, limit=64 << 20):
    """Writes what the timed legs computed in their last step as out_dir/<name>.npy (float64; `rank` prefixes the
    names of a multi-process run), so that two builds can be compared output for output on identical inputs:
      value_lnl / e2e_lnl                 [G][chains]: lnL of every local chain's proposal in every generation of the
                                          last timed step (resident descriptors / host structs through the C-ABI)
      value_current_lnl, _current_lnprior [chains]: each chain's state after that step (likewise e2e_*)
      mc3_chain_id, mc3_swap_info         the coordinator's heat assignment and swap counters after the value leg"""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > limit:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {limit})")
    for k, a in arrays.items():
        np.save(d / (k if rank is None else f"rank{rank}_{k}"), a)


class pack_bytes:
    """Size of the packed job a generation ships host->device (header + DevEval + rates/frequencies + branch
    list + node records).  Small jobs ride in the kernel parameter block, i.e. inside the launch."""

    def __init__(self, specs):
        a16 = lambda x: (x + 15) & ~15
        n_mat = sum(len(s.mats) for s in specs)
        n_op = sum(len(s.ops) for s in specs)
        n_dbl = sum(len(s.rates) + len(s.cat_weights) + len(s.freqs) for s in specs)
        self.bytes = a16(a16(a16(a16(16) + 96 * len(specs)) + 8 * n_dbl) + 16 * n_mat) + 48 * n_op


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="primates", choices=sorted(WORKLOADS))
    ap.add_argument("--generations-per-step", type=int, default=0,
                    help="MCMC generations per timed step (0 = the workload's default: 512 for primates)")
    ap.add_argument("--other", default="nuc200k,aa50k,codon20k",
                    help="N=1 default workload only: large synthetic configs reported under other_workloads ('' = none)")
    ap.add_argument("--no-extras", action="store_true", help="skip many_analyses / other_workloads")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed legs computed in their last step to DIR/<name>.npy (engine arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the engine arm's outputs")
    if args.impl == "reference":
        bench_reference(args)
    else:
        bench_engine(args)


if __name__ == "__main__":
    main()
