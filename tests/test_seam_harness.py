"""The seam (mrbayes_b200/seam/mb200_seam.c) inside the reference's own `mb` program.

oracle/_ref/mb_b200 = the UNMODIFIED reference objects + the seam + oracle/ref_harness.c (ld --wrap on
the single call site of the hot path).  Two kinds of tests:

* CPU (no GPU): in `dump` mode the seam's engine calls are recorded, not executed.  The records written
  through the node-granular function-pointer forms (TiProbs_B200 ... Likelihood_B200 installed in
  ModelInfo, driven by the reference's own LaunchLogLikeForDivision loop) must be byte-identical to the
  ones written through the seam's own loop -- and to the committed golden files, which pins the flip
  order, the operation lists, the rate assembly and the scaler bookkeeping of both paths.
* GPU: `shadow` mode -- the reference's CPU kernels drive a real MCMC run while every evaluation also
  runs on the engine; |lnL_gpu - lnL_cpu| / |lnL_cpu| is checked per evaluation (bar: 1e-6, the
  north-star tolerance; observed ~1e-8).  `gpu` mode: the engine alone drives the chain, through the
  seam's loop and through the function-pointer forms: identical lnL streams.
"""
from __future__ import annotations

import gzip
import json
import os
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "oracle" / "_ref" / "mb_b200"
BIN_BATCHED = ROOT / "oracle" / "_ref" / "mb_b200_batched"     # the same objects with the patched RunChain (oracle/patch_runchain.py)
CMD = ROOT / "tests" / "golden" / "cmd"

needs_harness = pytest.mark.skipif(not BIN.exists(), reason="oracle/_ref/mb_b200 not built (needs the reference sources at build time)")


def run_mb(binary: Path, nex: Path, env, timeout=900):
    """Runs a harness binary on `nex` from the directory `nex` is in.  MrBayes refuses file names longer than 99 characters,
    so the program sees short names relative to that directory only: the command files' output prefixes are bare names, and
    `oracle` there links to the repository's oracle/ for their `execute oracle/_ref/data/...` lines."""
    link = nex.parent / "oracle"
    if not link.is_symlink():
        link.symlink_to(ROOT / "oracle", target_is_directory=True)
    return subprocess.run([str(binary), nex.name], cwd=nex.parent, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                          text=True, timeout=timeout)


def run_harness(tmp_path: Path, stem: str, ngen: int, mode: str, via: str = "seam", extra_env=None, timeout=900, binary: Path = BIN, tag: str = ""):
    key = f"{stem}.{mode}.{via}" if not tag else "r" + tag.replace(".", "_")     # MrBayes limits file name lengths to 100 characters
    nex = tmp_path / f"{key}.nex"
    prefix = tmp_path / (f"out_{stem}_{mode}_{via}" if not tag else "o" + tag.replace(".", "_"))
    text = (CMD / f"{stem}.nex").read_text().replace("NGEN", str(ngen)).replace("OUTPREFIX", prefix.name)
    nex.write_text(text)
    report = tmp_path / f"{key}.json"
    env = dict(os.environ, MB200_MODE=mode, MB200_REPORT=str(report), MB200_VIA=via)
    env.update(extra_env or {})
    p = run_mb(binary, nex, env, timeout)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    assert report.exists(), p.stdout[-2000:] + p.stderr[-2000:]
    rep = json.loads(report.read_text().strip().splitlines()[-1])
    rep["stderr"] = p.stderr[-2000:]
    # what the run sampled (parameter and tree files), minus the random [ID: ...] stamp MrBayes puts in each file
    rep["samples"] = {f.name.replace(prefix.name, ""): "\n".join(l for l in f.read_text().splitlines() if "ID:" not in l)
                      for f in sorted(tmp_path.glob(prefix.name + "*")) if f.suffix in (".p", ".t")}
    return rep


# (command stem, generations, max evaluations recorded, committed golden written from the same command or None)
RECORD_CASES = [
    ("primates_gtr_g4", 60, 400, "primates_gtr_g4_fma"),
    ("primates_hky_g4", 100, 200, "primates_hky_g4_fma"),
    ("primates_f81_i", 100, 150, "primates_f81_i_fma"),
    ("cynmix_full", 40, 200, "cynmix_full_fma"),
    ("replicase_ny98", 60, 40, "replicase_ny98_sse"),
]


@needs_harness
@pytest.mark.parametrize("stem,ngen,max_evals,golden", RECORD_CASES)
def test_function_pointer_forms_record_the_same_evaluations(tmp_path, stem, ngen, max_evals, golden):
    files = {}
    for via in ("seam", "fnptr"):
        out = tmp_path / f"{stem}.{via}.gold"
        rep = run_harness(tmp_path, stem, ngen, "dump", via, {"MB200_DUMP_FILE": str(out), "MB200_DUMP_MAX": str(max_evals)})
        assert rep["dumped"] > 0 and rep["via"] == via
        files[via] = out.read_bytes()
    assert files["seam"] == files["fnptr"], "function-pointer forms and the seam's own loop disagree on the evaluation records"
    if golden is not None:
        committed = gzip.open(ROOT / "tests" / "golden" / f"{golden}.gold.gz").read()
        assert files["seam"] == committed, f"seam no longer reproduces tests/golden/{golden}.gold.gz"


# Chain-batched generations (SURVEY 8f1).  oracle/patch_runchain.py cuts RunChain's chain loop in two around LogLike; the
# seam queues every local chain's evaluation and sends one call per division and generation.  Here the seam's
# backend is the CPU oracle (harness mode "oracle"), which is bit-exact on the FMA build -- so the batched run must
# sample exactly what the unmodified reference samples: same accept / reject decisions, same trees, same lnL, every
# generation.  (The reference's seed, proposals and acceptance draws are untouched: the acceptance variate is drawn
# at the same position of the random stream.)
needs_batched = pytest.mark.skipif(not BIN_BATCHED.exists(), reason="oracle/_ref/mb_b200_batched not built (needs /root/reference at build time)")


@needs_harness
@needs_batched
@pytest.mark.parametrize("stem,ngen", [("primates_gtr_g4", 400), ("primates_hky_g4", 200), ("primates_gtr_ig4", 200), ("cynmix_full", 60),
                                       ("cynmix_ordered", 60)])      # ordered characters: P(t) from the reference's TiProbs_Std on the host
def test_chain_batched_generations_reproduce_the_serial_reference(tmp_path, stem, ngen):
    ref = run_harness(tmp_path, stem, ngen, "cpu", tag=".ref")                                  # the unmodified reference
    ser = run_harness(tmp_path, stem, ngen, "cpu", binary=BIN_BATCHED, tag=".patched")          # patched loop, serial path
    bat = run_harness(tmp_path, stem, ngen, "oracle", binary=BIN_BATCHED, tag=".batched")      # one call per generation
    assert ref["samples"] and ref["samples"] == ser["samples"], "the patched RunChain changed the serial trajectory"
    assert bat["batched_generations"] == ngen and bat["flushes"] == ngen and bat["unsupported_calls"] == 0, bat
    assert bat["calls"] == ref["calls"] and bat["aborts"] == ref["aborts"]
    assert bat["samples"] == ref["samples"], "chain-batched generations sample differently from the serial reference"


# The same identity over the model space: two runs x three chains, every sampled tree and parameter of the chain-batched loop
# (seam + bit-exact CPU oracle) equal to the unmodified reference's -- model jumping, rooted clock trees with relaxed-clock
# rates, amino-acid model jumping, codon models with one and three omega categories (host eigensystems), two partitions.
BATCHED_SWEEP = [
    ("primates.nex", "lset nst=mixed rates=gamma;", 200),
    ("primates.nex", "lset nst=6 rates=invgamma; prset brlenspr=clock:birthdeath clockvarpr=igr;", 200),
    ("avian_ovomucoids.nex", "prset aamodelpr=mixed; lset rates=gamma;", 60),
    ("replicase.nex", "lset nucmodel=codon omegavar=m3;", 100),
    ("primates.nex", "charset a=1-400; charset b=401-898; partition p=2:a,b; set partition=p; lset applyto=(1) nst=2 rates=gamma; "
                     "lset applyto=(2) nst=6 rates=propinv; unlink shape=(all) revmat=(all); prset applyto=(all) ratepr=variable;", 200),
    ("finch.nex", "lset nst=2 rates=gamma;", 200),          # 30 unlinked gene trees under a species tree
    ("hymfossil_nomcmc.nex", "lset applyto=(1) coding=variable rates=gamma; lset applyto=(2) nst=6 rates=invgamma; unlink shape=(all); "
                             "prset applyto=(all) ratepr=variable; prset brlenspr=clock:uniform clockvarpr=igr;", 40),
]


def _run_inline(tmp_path, binary, mode, data, cmds, ngen, tag, env=None):
    d = tmp_path / tag
    d.mkdir()
    nex = d / "r.nex"
    nex.write_text(f"set autoclose=yes nowarn=yes seed=99 swapseed=99;\nexecute oracle/_ref/data/{data};\n{cmds}\n"
                   f"mcmc nruns=2 nchains=3 ngen={ngen} printfreq=100000 samplefreq=25 diagnfreq=100000 filename=o;\nquit;\n")
    report = d / "r.json"
    e = dict(os.environ, MB200_MODE=mode, MB200_BATCH="1", MB200_REPORT=str(report))
    e.update(env or {})
    p = run_mb(binary, nex, e)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    rep = json.loads(report.read_text().strip().splitlines()[-1])
    rep["samples"] = {f.name: "\n".join(l for l in f.read_text().splitlines() if "ID:" not in l)
                      for f in sorted(d.glob("o*")) if f.suffix in (".p", ".t")}
    return rep


@needs_harness
@needs_batched
@pytest.mark.parametrize("data,cmds,ngen", BATCHED_SWEEP)
def test_chain_batched_generations_over_the_model_space(tmp_path, data, cmds, ngen):
    ref = _run_inline(tmp_path, BIN, "cpu", data, cmds, ngen, "ref")
    bat = _run_inline(tmp_path, BIN_BATCHED, "oracle", data, cmds, ngen, "bat")
    assert bat["batched_generations"] == ngen and bat["unsupported_calls"] == 0 and bat["calls"] == ref["calls"], bat
    assert len(ref["samples"]) >= 4 and bat["samples"] == ref["samples"]


@needs_harness
@needs_batched
@pytest.mark.parametrize("mc", ["nruns=2 nchains=8 ngen=100", "nruns=3 nchains=2 ngen=150 swapfreq=3 nswaps=2 temp=0.3"])
def test_chain_batched_generations_with_other_chain_layouts(tmp_path, mc):
    """16 local chains in one call per generation; three runs with two swap attempts every third generation at a hotter ladder."""
    def run(binary, mode, tag):
        d = tmp_path / tag
        d.mkdir()
        nex = d / "r.nex"
        nex.write_text(f"set autoclose=yes nowarn=yes seed=99 swapseed=99;\nexecute oracle/_ref/data/primates.nex;\nlset nst=6 rates=gamma;\n"
                       f"mcmc {mc} printfreq=100000 samplefreq=25 diagnfreq=100000 filename=o;\nquit;\n")
        report = d / "r.json"
        e = dict(os.environ, MB200_MODE=mode, MB200_BATCH="1", MB200_REPORT=str(report))
        p = run_mb(binary, nex, e)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        rep = json.loads(report.read_text().strip().splitlines()[-1])
        rep["samples"] = {f.name: "\n".join(l for l in f.read_text().splitlines() if "ID:" not in l)
                          for f in sorted(d.glob("o*")) if f.suffix in (".p", ".t")}
        return rep
    ref, bat = run(BIN, "cpu", "ref"), run(BIN_BATCHED, "oracle", "bat")
    assert bat["batched_generations"] > 0 and bat["unsupported_calls"] == 0 and bat["calls"] == ref["calls"]
    assert len(ref["samples"]) >= 4 and bat["samples"] == ref["samples"]


# Dynamic rescaling (SURVEY 8f2, opt-in MB200_RESCALE=dynamic): nodes are rescaled every few levels instead of at every
# node; an evaluation that trips the float-range guard is repeated at once with every node rescaled.  lnL then differs from
# the always-rescale arithmetic by rounding only -- a run follows the reference run's decisions and stays within the
# north-star tolerance of its lnL, generation by generation (CPU oracle as the seam's backend).
def _lnl_columns(rep_stdout):
    import re
    return [[float(x) for x in re.findall(r"-\d+\.\d+", l)] for l in rep_stdout.splitlines() if re.match(r"^\s+\d+ -- ", l)]


def _run_printing(tmp_path, stem, ngen, env, tag, mode="oracle"):
    nex = tmp_path / f"r{tag}.nex"
    text = (CMD / f"{stem}.nex").read_text().replace("NGEN", str(ngen)).replace("OUTPREFIX", f"o{tag}") \
                                          .replace("printfreq=100000", "printfreq=1")
    nex.write_text(text)
    report = tmp_path / f"r{tag}.json"
    e = dict(os.environ, MB200_MODE=mode, MB200_BATCH="1", MB200_REPORT=str(report))
    e.update(env)
    p = run_mb(BIN_BATCHED, nex, e)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    return json.loads(report.read_text().strip().splitlines()[-1]), _lnl_columns(p.stdout)


@needs_harness
@needs_batched
@pytest.mark.parametrize("env,min_retries", [
    ({"MB200_RESCALE": "dynamic", "MB200_RESCALE_RUN": "3", "MB200_RESCALE_MAXFREQ": "8"}, 0),           # sparse rescaling
    ({"MB200_RESCALE": "dynamic", "MB200_RESCALE_RUN": "4", "MB200_RESCALE_MAXFREQ": "1000"}, 1),        # ... until the guard trips
    ({"MB200_RESCALE": "dynamic", "MB200_RESCALE_RUN": "4", "MB200_RESCALE_MAXFREQ": "6", "MB200_RESCALE_FORCE_RETRY": "1"}, 500),
])
def test_dynamic_rescaling_follows_the_always_rescale_run(tmp_path, env, min_retries):
    ngen = 120
    base, a = _run_printing(tmp_path, "cynmix_part", ngen, {}, "a")
    dyn, b = _run_printing(tmp_path, "cynmix_part", ngen, env, "d")
    assert base["rescale_retries"] == 0 and dyn["rescale_retries"] >= min_retries, dyn
    assert dyn["aborts"] == base["aborts"] and dyn["calls"] == base["calls"] and dyn["batched_generations"] == ngen
    assert len(a) == len(b) and len(a) >= ngen
    worst = max(abs(u - v) / abs(u) for x, y in zip(a, b) for u, v in zip(sorted(x), sorted(y)))
    assert worst < 1e-6, worst          # printed lnL of every chain, every generation (3 decimals of ~3e4: resolves 3e-8)


# Host readers of conditional-likelihood buffers (SURVEY 8f4): ancestral states at a constrained node and site rates are
# computed by the reference's own CondLikeUp_* / PrintAncStates_* / PrintSiteRates_* on its host arrays at sample time; the
# seam wraps the three function pointers and copies the cold chain's buffers back first (MB200InstallReaders).  The
# reference's own numbers cannot serve as the yardstick here: with these reports on it switches to its scalar kernels
# (src/mcmc.c:17971-17992), which in this snapshot return lnL -1559.354 for two DIFFERENT starting trees of primates where
# its SIMD kernels, the oracle and the engine agree on -8019.475 / -7576.147 / -7942.846 for such states (shadow mode
# against the oracle shows it evaluation by evaluation; the covarion models use the same scalar path).  So: the run must be
# driven entirely by the engine side, batched and serial must sample the same, and what the readers print must be
# probabilities and rates.
@needs_harness
@needs_batched
def test_host_readers_of_cl_buffers_run_on_synced_buffers(tmp_path):
    ngen = 100
    ser = run_harness(tmp_path, "primates_readers", ngen, "oracle", binary=BIN_BATCHED, extra_env={"MB200_BATCH": "0"}, tag=".s")
    bat = run_harness(tmp_path, "primates_readers", ngen, "oracle", binary=BIN_BATCHED, extra_env={"MB200_BATCH": "1"}, tag=".b")
    assert ser["unsupported_calls"] == 0 and bat["unsupported_calls"] == 0 and bat["batched_generations"] == ngen
    assert ser["samples"] and ser["samples"] == bat["samples"]
    lines = [l for l in ser["samples"][".p"].splitlines() if l and not l.startswith("[")]
    head, rows = lines[0].split("\t"), [l.split("\t") for l in lines[1:]]
    anc = [i for i, h in enumerate(head) if h.startswith("p(")]
    rate = [i for i, h in enumerate(head) if h.startswith("r(") and h[2:-1].isdigit()]
    lnl = head.index("lnLike")
    assert len(anc) % 4 == 0 and len(anc) >= 4 * 800 and len(rate) >= 800 and len(rows) >= 5
    for r in rows:
        assert -9000.0 < float(r[lnl]) < -5000.0            # what primates allows; the reference's scalar path says -1559
        for i in range(0, len(anc), 4):
            p4 = [float(r[j]) for j in anc[i:i + 4]]
            assert all(0.0 <= x <= 1.0 for x in p4) and abs(sum(p4) - 1.0) < 1e-5
        assert all(0.0 < float(r[j]) < 100.0 for j in rate)


# The reference's SCALAR kernel family (CondLikeDown_Gen / _NUC4, Likelihood_Gen, ...) serves covarion and doublet divisions and
# every division whose conditional likelihoods are read on the host (report ancstates / siterates).  In an SSE-enabled build of
# the reference those kernels read SIMD-laid-out buffers: primates starts at lnL -1558.16 with covarion=yes and at the SAME
# -1559.354 for two different trees with ancstates=yes.  A build without any SIMD switch (oracle/Makefile: mb_ref_scalar,
# mb_b200_scalar) gives -9051.351 / -7576.147, -7942.846 -- the values of the seam + oracle and of the engine.  Parity of
# these paths is therefore pinned on the scalar build: every evaluation of a shadow run compared.
BIN_SCALAR = ROOT / "oracle" / "_ref" / "mb_b200_scalar"
needs_scalar = pytest.mark.skipif(not BIN_SCALAR.exists(), reason="oracle/_ref/mb_b200_scalar not built")
SCALAR_CASES = [("primates_covarion", 200, 400), ("primates_readers", 200, 400), ("kim_mixed", 60, 600), ("ovomucoids_covarion", 30, 60)]


@needs_scalar
@pytest.mark.parametrize("stem,ngen,min_calls", SCALAR_CASES)
def test_scalar_kernel_family_matches_the_no_simd_reference(tmp_path, stem, ngen, min_calls):
    rep = run_harness(tmp_path, stem, ngen, "shadow", binary=BIN_SCALAR, extra_env={"MB200_SHADOW_BACKEND": "oracle"}, tag=".sc")
    assert rep["calls"] >= min_calls and rep["unsupported_calls"] == 0, rep
    assert rep["failed"] == 0 and rep["compared"] == rep["calls"], rep
    assert rep["max_rel"] < 1e-6, rep


# A sweep over the model space the seam accepts, each as a shadow run in the no-SIMD build (every evaluation compared with the
# reference's own): substitution-model jumping (nst=mixed), closed-form models with readers, lognormal / k-mixture rate
# variation, JC, amino-acid model jumping and protein GTR, codon M3 (three omega categories) and codon GTR; autocorrelated gamma
# is outside the path and must be declined, not mis-evaluated; rooted clock trees with and without relaxed-clock branch rates,
# eight gamma categories, two differently modelled partitions of one alignment.
MODEL_SWEEP = [
    ("primates.nex", "lset nst=mixed rates=gamma;", True),
    ("primates.nex", "lset nst=2 rates=propinv; report ancstates=yes;", True),
    ("primates.nex", "lset nst=6 rates=lnorm;", True),
    ("primates.nex", "lset nst=6 rates=kmixture;", True),
    ("primates.nex", "lset nst=1 rates=equal;", True),
    ("avian_ovomucoids.nex", "prset aamodelpr=mixed; lset rates=gamma;", True),
    ("avian_ovomucoids.nex", "prset aamodelpr=fixed(gtr); lset rates=equal;", True),
    ("replicase.nex", "lset nucmodel=codon omegavar=m3;", True),
    ("replicase.nex", "lset nucmodel=codon nst=6 rates=equal;", True),
    # rooted (clock) trees, relaxed-clock branch rates (the effective branch length is length x rate, SeamBranchLength)
    ("primates.nex", "lset nst=6 rates=gamma; prset brlenspr=clock:uniform;", True),
    ("primates.nex", "lset nst=6 rates=invgamma; prset brlenspr=clock:birthdeath clockvarpr=igr;", True),
    ("primates.nex", "lset nst=6 rates=gamma; prset brlenspr=clock:uniform clockvarpr=tk02;", True),
    ("primates.nex", "lset nst=6 rates=gamma ngammacat=8;", True),
    ("primates.nex", "lset nst=6 rates=gamma ngammacat=10;", True),          # more than 8 categories: 4 states on the generic kernel
    ("primates.nex", "lset nst=6 rates=invgamma ngammacat=19;", True),       # the most MrBayes accepts
    ("primates.nex", "charset a=1-400; charset b=401-898; partition p=2:a,b; set partition=p; lset applyto=(1) nst=2 rates=gamma; "
                     "lset applyto=(2) nst=6 rates=propinv; unlink shape=(all) revmat=(all); prset applyto=(all) ratepr=variable;", True),
    # hymfossil.nex: 114 taxa (45 fossils: mostly missing data), 7-state morphology with ordered characters and coding=variable,
    # 2 765 DNA patterns, rooted clock tree with independent-gamma branch rates
    ("hymfossil_nomcmc.nex", "ctype ordered: 20 23 27 30 35 36 41 42 44 46 48 59 65 75 78 79 89 99 112 117 134 146 157; "
                             "lset applyto=(1) coding=variable rates=gamma; lset applyto=(2) nst=6 rates=invgamma; unlink shape=(all); "
                             "prset applyto=(all) ratepr=variable; prset brlenspr=clock:uniform clockvarpr=igr;", True),
    # finch.nex: 30 loci with UNLINKED topologies (gene trees under a species tree): every division has its own tree
    ("finch.nex", "lset nst=2 rates=gamma;", True),
    ("primates.nex", "lset nst=6 rates=adgamma;", False),
]


def _run_sweep_case(tmp_path, data, cmds, ngen, env):
    nex = tmp_path / "sweep.nex"
    nex.write_text(f"set autoclose=yes nowarn=yes seed=99 swapseed=99;\nexecute oracle/_ref/data/{data};\n{cmds}\n"
                   f"mcmc nruns=1 nchains=2 ngen={ngen} printfreq=100000 samplefreq=50 diagnfreq=100000 filename=o;\nquit;\n")
    report = tmp_path / "sweep.json"
    e = dict(os.environ, MB200_MODE="shadow", MB200_REPORT=str(report))
    e.update(env)
    p = run_mb(BIN_SCALAR, nex, e)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    return json.loads(report.read_text().strip().splitlines()[-1])


@needs_scalar
@pytest.mark.parametrize("data,cmds,supported", MODEL_SWEEP)
def test_model_sweep_against_the_no_simd_reference(tmp_path, data, cmds, supported):
    rep = _run_sweep_case(tmp_path, data, cmds, 100, {"MB200_SHADOW_BACKEND": "oracle"})
    assert rep["calls"] >= 150, rep
    if supported:
        assert rep["unsupported_calls"] == 0 and rep["compared"] == rep["calls"] and rep["failed"] == 0 and rep["max_rel"] < 1e-6, rep
    else:
        assert rep["unsupported_calls"] == rep["calls"] and rep["compared"] == 0, rep


def _run_session(tmp_path, binary, mode, tag, env=None):
    """Three mcmc commands in ONE session, the model changed in between: codon M0 (61 states) -> GTR + 6 gamma categories on the
    nucleotides (3 chains) -> codon NY98 (three eigensystems per slot).  Instances, scratch sets and work matrices must follow."""
    d = tmp_path / tag
    d.mkdir()
    nex = d / "r.nex"
    nex.write_text("set autoclose=yes nowarn=yes seed=99 swapseed=99;\nexecute oracle/_ref/data/replicase.nex;\nlset nucmodel=codon;\n"
                   "mcmc nruns=1 nchains=2 ngen=40 printfreq=100000 samplefreq=20 diagnfreq=100000 filename=a;\n"
                   "lset nucmodel=4by4 nst=6 rates=gamma ngammacat=6;\n"
                   "mcmc nruns=1 nchains=3 ngen=60 printfreq=100000 samplefreq=20 diagnfreq=100000 filename=b;\n"
                   "lset nucmodel=codon omegavar=ny98;\n"
                   "mcmc nruns=1 nchains=2 ngen=40 printfreq=100000 samplefreq=20 diagnfreq=100000 filename=c;\nquit;\n")
    report = d / "r.json"
    e = dict(os.environ, MB200_MODE=mode, MB200_BATCH="1", MB200_REPORT=str(report))
    e.update(env or {})
    p = run_mb(binary, nex, e)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    rep = json.loads(report.read_text().strip().splitlines()[-1])
    rep["samples"] = {f.name: "\n".join(l for l in f.read_text().splitlines() if "ID:" not in l)
                      for f in sorted(d.glob("[abc].*")) if f.suffix in (".p", ".t")}
    return rep


@needs_harness
@needs_batched
def test_model_changes_between_mcmc_commands(tmp_path):
    ref = _run_session(tmp_path, BIN, "cpu", "ref")
    bat = _run_session(tmp_path, BIN_BATCHED, "oracle", "bat")
    assert bat["unsupported_calls"] == 0 and bat["calls"] == ref["calls"] and bat["batched_generations"] == 140
    assert len(ref["samples"]) == 6 and bat["samples"] == ref["samples"]


BIN_SCALAR_BATCHED = ROOT / "oracle" / "_ref" / "mb_b200_scalar_batched"


@pytest.mark.skipif(not BIN_SCALAR_BATCHED.exists(), reason="oracle/_ref/mb_b200_scalar_batched not built")
@pytest.mark.parametrize("stem,ngen", [("primates_covarion", 200), ("primates_readers", 200), ("kim_mixed", 100), ("replicase_possel", 60)])
def test_chain_batched_scalar_family_follows_the_no_simd_reference(tmp_path, stem, ngen):
    """Chain-batched generations in the no-SIMD build (seam + CPU oracle) vs the reference driving itself: hidden-state models,
    host readers (ancestral states / site rates; selection probabilities / site omegas), kim.nex's seven partitions -- every sampled
    value agrees to the printed precision over the whole run, i.e. the two runs took the same decisions throughout."""
    ref = run_harness(tmp_path, stem, ngen, "cpu", binary=BIN_SCALAR, tag=".sbr")
    bat = run_harness(tmp_path, stem, ngen, "oracle", binary=BIN_SCALAR_BATCHED, extra_env={"MB200_BATCH": "1"}, tag=".sbb")
    assert bat["unsupported_calls"] == 0 and bat["calls"] == ref["calls"] and bat["batched_generations"] == ngen
    (ha, ra), (hb, rb) = _sample_rows(ref), _sample_rows(bat)
    assert ha == hb and len(ra) == len(rb) >= 4
    assert _rows_agree(ra, rb) == len(ra), (_rows_agree(ra, rb), len(ra))
    assert ref["samples"][".t"] == bat["samples"][".t"]            # the sampled trees: identical text


FNPTR_SWEEP = [
    ("primates.nex", "lset nst=6 rates=gamma covarion=yes;"),
    ("primates.nex", "lset nst=2 rates=propinv; report ancstates=yes;"),
    ("kim.nex", "set partition=by_gene_and_struct; lset applyto=(1) nucmodel=doublet nst=6; lset applyto=(2,3,4) nst=6 rates=invgamma; "
                "prset applyto=(5,6) aamodelpr=fixed(wag); lset applyto=(5,6) rates=gamma; lset applyto=(7) rates=gamma;"),
    ("hymfossil_nomcmc.nex", "ctype ordered: 20 23 27 30 35 36; lset applyto=(1) coding=variable rates=gamma; lset applyto=(2) nst=6 rates=invgamma; "
                             "prset brlenspr=clock:uniform clockvarpr=igr;"),
    ("finch.nex", "lset nst=2 rates=gamma;"),
]


@needs_scalar
@pytest.mark.parametrize("data,cmds", FNPTR_SWEEP)
def test_function_pointer_forms_drive_like_the_seam_loop_over_models(tmp_path, data, cmds):
    """The node-granular forms installed in ModelInfo (the reference's own LaunchLogLikeForDivision loop records the evaluation
    through them) and the seam's replacement loop sample the same trees and parameters: hidden-state models, host readers,
    seven mixed partitions, host-built ordered-character matrices, unlinked gene trees."""
    def run(via):
        d = tmp_path / via
        d.mkdir()
        nex = d / "r.nex"
        nex.write_text(f"set autoclose=yes nowarn=yes seed=99 swapseed=99;\nexecute oracle/_ref/data/{data};\n{cmds}\n"
                       f"mcmc nruns=1 nchains=2 ngen=100 printfreq=100000 samplefreq=25 diagnfreq=100000 filename=o;\nquit;\n")
        report = d / "r.json"
        e = dict(os.environ, MB200_MODE="oracle", MB200_VIA=via, MB200_MULTIPART="0", MB200_EIGEN="host", MB200_REPORT=str(report))
        p = run_mb(BIN_SCALAR, nex, e)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        rep = json.loads(report.read_text().strip().splitlines()[-1])
        rep["samples"] = {f.name: "\n".join(l for l in f.read_text().splitlines() if "ID:" not in l)
                          for f in sorted(d.glob("o*")) if f.suffix in (".p", ".t")}
        return rep
    a, b = run("seam"), run("fnptr")
    assert a["unsupported_calls"] == 0 and b["unsupported_calls"] == 0 and a["calls"] == b["calls"] > 0
    assert len(a["samples"]) >= 2 and a["samples"] == b["samples"]


def _sample_rows(rep):
    lines = [l for l in rep["samples"][".p"].splitlines() if l and not l.startswith("[")]
    return lines[0].split("\t"), [[float(x) for x in l.split("\t")] for l in lines[1:]]


def _rows_agree(ra, rb, rel=2e-6):
    """How many leading sample rows agree in every column (7 significant digits are printed)."""
    n = 0
    for x, y in zip(ra, rb):
        if len(x) != len(y) or any(abs(u - v) > rel * max(abs(u), abs(v)) + 1e-9 for u, v in zip(x, y)):
            break
        n += 1
    return n


@needs_scalar
@pytest.mark.parametrize("stem", ["primates_covarion", "primates_readers", "replicase_possel"])
def test_scalar_build_runs_sample_what_the_reference_samples(tmp_path, stem):
    """The no-SIMD reference driving itself vs the seam + CPU oracle driving the same binary: the sampled parameters -- for
    primates_readers including ~3 300 ancestral-state probabilities and ~900 site rates per sample, read by the reference's own
    CondLikeUp / PrintAncStates / PrintSiteRates from the buffers the seam synced -- agree to the printed precision."""
    ngen = 100 if stem == "replicase_possel" else 200      # (possel: ~240 selection probabilities + ~240 site omegas per sample)
    ref = run_harness(tmp_path, stem, ngen, "cpu", binary=BIN_SCALAR, tag=".scr")
    orc = run_harness(tmp_path, stem, ngen, "oracle", binary=BIN_SCALAR, tag=".sco")
    assert orc["unsupported_calls"] == 0 and orc["calls"] == ref["calls"]
    (ha, ra), (hb, rb) = _sample_rows(ref), _sample_rows(orc)
    assert ha == hb and len(ra) == len(rb) >= 10
    assert _rows_agree(ra, rb) == len(ra), (_rows_agree(ra, rb), len(ra))


@needs_harness
@needs_batched
def test_covarion_division_batched_equals_per_chain(tmp_path):
    ngen = 100
    off = run_harness(tmp_path, "primates_covarion", 20, "oracle", binary=BIN_BATCHED, extra_env={"MB200_NO_COVARION": "1"}, tag=".off")
    assert off["unsupported_calls"] == off["calls"] > 0                 # A/B switch: left to the reference
    ser = run_harness(tmp_path, "primates_covarion", ngen, "oracle", binary=BIN_BATCHED, extra_env={"MB200_BATCH": "0"}, tag=".s")
    bat = run_harness(tmp_path, "primates_covarion", ngen, "oracle", binary=BIN_BATCHED, extra_env={"MB200_BATCH": "1"}, tag=".b")
    assert ser["unsupported_calls"] == 0 and bat["unsupported_calls"] == 0 and bat["batched_generations"] == ngen
    assert ser["samples"] and ser["samples"] == bat["samples"]
    lines = [l for l in ser["samples"][".p"].splitlines() if l and not l.startswith("[")]
    lnl = lines[0].split("\t").index("lnLike")
    assert all(-9500.0 < float(l.split("\t")[lnl]) < -5000.0 for l in lines[1:])


# ---------------------------------------------------------------------------------------- GPU
@needs_harness
@needs_batched
@pytest.mark.gpu
@pytest.mark.parametrize("stem,ngen", [("primates_gtr_g4", 2000), ("cynmix_full", 200), ("primates_readers", 200), ("cynmix_ordered", 100)])
def test_chain_batched_generations_on_the_engine(tmp_path, engine_lib, stem, ngen):
    """The engine driving the chain: all local chains of a generation in ONE launch per division == one launch per chain
    (bit-identical lnL streams, hence identical samples), and both stay within the north-star tolerance of the
    reference's own trajectory for as long as the two runs make the same decisions."""
    one = run_harness(tmp_path, stem, ngen, "gpu", binary=BIN_BATCHED, extra_env={"MB200_BATCH": "0"}, tag=".serial")
    bat = run_harness(tmp_path, stem, ngen, "gpu", binary=BIN_BATCHED, extra_env={"MB200_BATCH": "1"}, tag=".batched")
    assert bat["batched_generations"] == ngen and bat["unsupported_calls"] == 0 and one["batched_generations"] == 0, (one, bat)
    assert bat["calls"] == one["calls"] and bat["aborts"] == one["aborts"]
    assert bat["samples"] and bat["samples"] == one["samples"], "chain-batched launches sample differently from per-chain launches"


@needs_scalar
@pytest.mark.gpu
@pytest.mark.parametrize("stem,ngen,min_calls", SCALAR_CASES)
def test_engine_matches_the_no_simd_reference_on_its_scalar_kernel_family(tmp_path, engine_lib, stem, ngen, min_calls):
    """Covarion (8 hidden-state model states), host readers, and kim.nex's seven partitions (doublet 16 states on the generic
    kernel, 4-state, 20-state tensor-core, morphology) against the reference built without SIMD switches: every evaluation."""
    rep = run_harness(tmp_path, stem, ngen, "shadow", binary=BIN_SCALAR, tag=".scg")
    assert rep["calls"] >= min_calls and rep["unsupported_calls"] == 0, rep
    assert rep["failed"] == 0 and rep["compared"] == rep["calls"], rep
    assert rep["max_rel"] < 1e-6, rep


@needs_scalar
@pytest.mark.gpu
@pytest.mark.parametrize("data,cmds,supported", [c for c in MODEL_SWEEP if c[2]])
def test_model_sweep_on_the_engine(tmp_path, engine_lib, data, cmds, supported):
    rep = _run_sweep_case(tmp_path, data, cmds, 150, {})
    assert rep["calls"] >= 250 and rep["unsupported_calls"] == 0, rep
    assert rep["compared"] == rep["calls"] and rep["failed"] == 0 and rep["max_rel"] < 1e-6, rep


@needs_scalar
@pytest.mark.gpu
@pytest.mark.parametrize("stem", ["primates_covarion", "primates_readers", "replicase_possel"])
def test_engine_driven_scalar_build_samples_like_the_reference(tmp_path, engine_lib, stem):
    """The engine drives the no-SIMD reference binary; its samples (incl. ancestral states / site rates through the wrapped host
    readers) follow the reference's own for as long as the two runs take the same decisions (at least the first five samples)."""
    ngen = 200
    ref = run_harness(tmp_path, stem, ngen, "cpu", binary=BIN_SCALAR, tag=".sgr")
    eng = run_harness(tmp_path, stem, ngen, "gpu", binary=BIN_SCALAR, tag=".sge")
    assert eng["unsupported_calls"] == 0
    (ha, ra), (hb, rb) = _sample_rows(ref), _sample_rows(eng)
    assert ha == hb and len(ra) >= 10
    assert _rows_agree(ra, rb, rel=1e-5) >= 5, _rows_agree(ra, rb, rel=1e-5)


@needs_harness
@needs_batched
@pytest.mark.gpu
def test_covarion_on_the_engine_follows_the_oracle_run(tmp_path, engine_lib):
    """Engine (generic-state kernel, 8 states, per-category eigensystems) vs the CPU oracle as the seam's backend on the
    same command: the two runs print the same lnL, generation by generation, within the north-star tolerance for as long
    as they make the same decisions (at least the first 30 generations)."""
    env = {}
    ro, lo = _run_printing(tmp_path, "primates_covarion", 60, env, ".co", mode="oracle")
    rg, lg = _run_printing(tmp_path, "primates_covarion", 60, env, ".cg", mode="gpu")
    assert rg["unsupported_calls"] == 0 and rg["batched_generations"] == 60 and ro["calls"] == rg["calls"]
    assert len(lo) >= 60 and len(lg) >= 60
    for g in range(30):
        for a, b in zip(lo[g], lg[g]):
            assert abs(a - b) <= 1e-6 * abs(a) + 2e-3, (g, lo[g], lg[g])      # 3 decimals are printed


@needs_harness
@needs_batched
@pytest.mark.gpu
@pytest.mark.parametrize("stem,ngen,min_eigens", [("replicase_m0", 150, 2), ("replicase_ny98", 100, 2), ("primates_gtr_g4", 150, 4),
                                                  ("ovomucoids_wag_g4", 40, 1)])
def test_device_eigensystems_follow_the_host_run(tmp_path, engine_lib, stem, ngen, min_eigens):
    """MB200_EIGEN=device (SURVEY 8 f3; the default for more than 32 states): the rate matrices go to the engine, which diagonalises them on its stream, instead of
    the host's GetEigens + CalcCijk and a block upload.  P(t) then agrees to the rounding of double sums, so the run prints
    the same lnL as the host-eigensystem run, generation by generation, within the north-star tolerance."""
    rh, lh = _run_printing(tmp_path, stem, ngen, {"MB200_EIGEN": "host"}, ".eh", mode="gpu")
    rd, ld = _run_printing(tmp_path, stem, ngen, {"MB200_EIGEN": "device"}, ".ed", mode="gpu")
    assert rh["device_eigens"] == 0 and rd["device_eigens"] >= min_eigens, (rh["device_eigens"], rd["device_eigens"])
    assert rd["unsupported_calls"] == 0 and rd["calls"] == rh["calls"] and rd["aborts"] == rh["aborts"]
    assert len(lh) >= ngen and len(ld) >= ngen
    for g in range(ngen):
        for a, b in zip(lh[g], ld[g]):
            assert abs(a - b) <= 1e-6 * abs(a) + 2e-3, (g, lh[g], ld[g])      # 3 decimals are printed


@needs_harness
@needs_batched
@pytest.mark.gpu
def test_model_changes_between_mcmc_commands_on_the_engine(tmp_path, engine_lib):
    """The same session on the engine (device eigensystems for the two codon runs: 1 and then 3 rate matrices per slot): batched
    launches == per-chain launches, nothing handed back to the reference."""
    one = _run_session(tmp_path, BIN_BATCHED, "gpu", "one", {"MB200_BATCH": "0"})
    bat = _run_session(tmp_path, BIN_BATCHED, "gpu", "bat", {"MB200_BATCH": "1"})
    assert one["unsupported_calls"] == 0 and bat["unsupported_calls"] == 0 and bat["batched_generations"] == 140
    assert bat["device_eigens"] > 0 and len(one["samples"]) == 6 and bat["samples"] == one["samples"]


ENGINE_BATCH_SWEEP = [
    ("replicase.nex", "lset nucmodel=codon omegavar=ny98;", "nruns=1 nchains=4 ngen=200", {}),                       # device eigensystems
    ("replicase.nex", "lset nucmodel=codon omegavar=ny98;", "nruns=1 nchains=4 ngen=200", {"MB200_EIGEN": "host"}),
    ("finch.nex", "lset nst=2 rates=gamma;", "nruns=2 nchains=3 ngen=300", {}),                                     # 30 unlinked gene trees
    ("hymfossil_nomcmc.nex", "lset applyto=(1) coding=variable rates=gamma; lset applyto=(2) nst=6 rates=invgamma; unlink shape=(all); "
                             "prset applyto=(all) ratepr=variable; prset brlenspr=clock:uniform clockvarpr=igr;", "nruns=1 nchains=4 ngen=300", {}),
    ("kim.nex", "set partition=by_gene_and_struct; lset applyto=(1) nucmodel=doublet nst=6; lset applyto=(2,3,4) nst=6 rates=invgamma; "
                "prset applyto=(5,6) aamodelpr=fixed(wag); lset applyto=(5,6) rates=gamma; lset applyto=(7) rates=gamma; "
                "unlink revmat=(all) pinvar=(all) shape=(all) statefreq=(all); prset applyto=(all) ratepr=variable;", "nruns=1 nchains=4 ngen=200", {}),
    ("primates.nex", "lset nst=6 rates=gamma covarion=yes;", "nruns=2 nchains=4 ngen=300", {}),
]


@needs_harness
@needs_batched
@pytest.mark.gpu
@pytest.mark.parametrize("data,cmds,mc,env", ENGINE_BATCH_SWEEP)
def test_chain_batched_launches_equal_per_chain_launches_over_data_sets(tmp_path, engine_lib, data, cmds, mc, env):
    """All local chains of a generation in one launch per division == one launch per chain: identical samples, whatever the
    kernel family (4-state, tensor-core 20 / 61 states, generic 8 / 16 states, morphology) and the tree layout."""
    def run(batch):
        d = tmp_path / ("b" + batch)
        d.mkdir()
        nex = d / "r.nex"
        nex.write_text(f"set autoclose=yes nowarn=yes seed=99 swapseed=99;\nexecute oracle/_ref/data/{data};\n{cmds}\n"
                       f"mcmc {mc} printfreq=100000 samplefreq=25 diagnfreq=100000 filename=o;\nquit;\n")
        report = d / "r.json"
        e = dict(os.environ, MB200_MODE="gpu", MB200_BATCH=batch, MB200_REPORT=str(report))
        e.update(env)
        p = run_mb(BIN_BATCHED, nex, e)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        rep = json.loads(report.read_text().strip().splitlines()[-1])
        rep["samples"] = {f.name: "\n".join(l for l in f.read_text().splitlines() if "ID:" not in l)
                          for f in sorted(d.glob("o*")) if f.suffix in (".p", ".t")}
        return rep
    one, bat = run("0"), run("1")
    assert one["unsupported_calls"] == 0 and bat["unsupported_calls"] == 0 and one["batched_generations"] == 0 and bat["batched_generations"] > 0
    assert bat["calls"] == one["calls"] and len(one["samples"]) >= 2 and bat["samples"] == one["samples"]


SHADOW_CASES = [
    # stem, generations, expected unsupported calls (None = any), min evaluations
    ("primates_gtr_g4", 2000, 0, 16000),
    ("primates_gtr_ig4", 500, 0, 1000),
    ("primates_hky_g4", 500, 0, 1000),
    ("primates_f81_i", 300, 0, 500),
    ("ovomucoids_wag_g4", 300, 0, 300),
    ("replicase_m0", 200, 0, 200),
    ("replicase_ny98", 100, 0, 100),
    ("cynmix_full", 300, 0, 1500),
    ("cynmix_ordered", 200, 0, 1000),     # ordered morphology: host-built matrices (set_transition_matrix), engine pruning
]


@needs_harness
@pytest.mark.gpu
@pytest.mark.parametrize("stem,ngen,unsupported,min_calls", SHADOW_CASES)
def test_shadow_run_matches_reference_per_evaluation(tmp_path, engine_lib, stem, ngen, unsupported, min_calls):
    rep = run_harness(tmp_path, stem, ngen, "shadow")
    assert rep["calls"] >= min_calls, rep
    assert rep["failed"] == 0, rep
    assert rep["compared"] == rep["calls"] - rep["unsupported_calls"], rep
    if unsupported is not None:
        assert rep["unsupported_calls"] == unsupported, rep
    assert rep["max_rel"] < 1e-6, rep          # north-star tolerance: 1e-6 relative per evaluation


@needs_harness
@pytest.mark.gpu
@pytest.mark.parametrize("stem,ngen", [("primates_gtr_g4", 1000), ("cynmix_full", 100), ("replicase_m0", 60)])
def test_engine_drives_the_chain_identically_through_both_entry_levels(tmp_path, engine_lib, stem, ngen):
    # eigensystems from the host in both runs: the function-pointer forms are driven by the reference's own loop, which calls
    # UpDateCijk itself, and "bit for bit" needs the same eigensystem on both sides (codon divisions default to the device solver)
    a = run_harness(tmp_path, stem, ngen, "gpu", "seam", {"MB200_MULTIPART": "0", "MB200_EIGEN": "host"})
    b = run_harness(tmp_path, stem, ngen, "gpu", "fnptr", {"MB200_EIGEN": "host"})
    assert a["calls"] == b["calls"] and a["calls"] > 0
    assert a["unsupported_calls"] == 0 and b["unsupported_calls"] == 0
    assert a["lnl_hash"] == b["lnl_hash"], (a, b)       # the same lnL, bit for bit, at every evaluation
    c = run_harness(tmp_path, stem, ngen, "gpu", "seam")    # partition-batched LogLike (MB200LogLike)
    assert c["unsupported_calls"] == 0 and c["aborts"] == a["aborts"]
