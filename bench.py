#!/usr/bin/env python
"""bench.py — mutants/sec of ESM-1v 650M masked-marginal scoring (BASELINE.json metric, config 2), plus bounded samples of
BASELINE configs 3-5 in the same JSON line.

A "step" is one pass of the hot path over one synthetic assay: WT of L=512 residues, 5000 single mutants
(SURVEY.md §8d config 2): 512 masked copies x 514 tokens through 33 layers, masked-row LM head, mutant scoring.

  python bench.py --gpus N --steps K --warmup W            # our arm  (one JSON line on rank 0)
  python bench.py ... --dump-outputs DIR                   # + DIR/scores.npy: the scores of the last timed step, to compare builds
  python bench.py --impl reference --gpus N ...            # reference arm: the reference's CPU loop (oracle port) on the host cores

`value`  : whole-job mutants/s with inputs already resident in HBM (device-timed with CUDA events, max over ranks; no profiling
           events inside this leg).
`e2e`    : same metric through the public API (EsmScorer.score_assay) with host buffers: tokenise/parse on host, pinned
           H2D of the int32 block, D2H of the scores, all inside the timed region.
`roofline`: tensor-pipe bound; a separate pass of the same K steps with per-kernel CUDA events: achieved = algorithmic GEMM
           FLOPs (2*M*N*K per launch; x1, never the split-operand work) / event time of the tcgen05 GEMM launches, vs
           MEASURED_PEAKS.json bf16 sustained. `issued_*` counts the tensor-pipe work really executed (x2 / x3 by precision mode,
           with the pruned last layer counted as pruned).
`other_workloads`: bounded samples of config 3 (ESM2-3B over the DMS_substitutions length distribution, LPT over the ranks),
           config 4 (Tranception-L on DMS_indels shapes) and config 5 (TranceptEVE fusion with synthetic priors).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

L_SEQ, N_MUT, N_ASSAYS = 512, 5000, 10
PASSES = {"f16x3": 3, "f16f8": 2, "f16": 1, "f16d": 1}  # tensor-pipe units per algorithmic FLOP of a linear layer
METRIC = "mutants/sec (ESM-1v 650M masked-marginal, L<=1024)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="f16d", choices=["f16d", "f16f8", "f16x3", "f16"],
                    help="f16d (headline: what `--precision auto` picks for this workload), f16f8 and f16x3 = parity modes (<=1e-3 abs vs the "
                         "fp32 reference); f16 = plain single-pass fast mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-workloads", action="store_true", help="skip the config 3/4/5 samples")
    ap.add_argument("--no-other-modes", action="store_true", help="skip the legs at the other precision modes")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--small", action="store_true", help="tiny model/assay (debugging only; not a valid bench)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the per-mutant scores of the last timed step (rank 0, headline precision) to DIR/scores.npy (float32); "
                         "inputs are seeded, so runs with the same arguments score the same assay")
    return ap.parse_args()


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["bf16_tflops_sustained"]), float(p["bf16_tflops"]), float(p["hbm_gbs"]), "measured"
    except Exception:
        return 1400.0, 1590.0, 6650.0, "fallback"


def algorithmic_flops(arch, T, P):
    """SURVEY.md §8d: F_fwd(T) = Lyr*[2*T*(4d^2+2df) + 4*T^2*d] + 2*T*(d^2+d*V), per assay P*F_fwd."""
    Lyr, d, f, V = arch.layers, arch.embed_dim, arch.ffn_dim, arch.vocab
    lin = Lyr * 2 * T * (4 * d * d + 2 * d * f)
    att = Lyr * 4 * T * T * d
    head = 2 * T * (d * d + d * V)
    return P * (lin + att + head), P * lin


def issued_linear_flops(arch, T, P, passes):
    """Tensor-pipe FLOPs the linear layers really execute per assay: all layers but the last in full, the last layer's QKV in
    full and its out_proj / fc1 / fc2 for the one emitted row per copy (exact pruning), times the operand-split multiplier."""
    Lyr, d, f = arch.layers, arch.embed_dim, arch.ffn_dim
    full = 2.0 * T * (4 * d * d + 2 * d * f)
    last = 2.0 * T * 3 * d * d + 2.0 * (d * d + 2 * d * f)
    return passes * P * ((Lyr - 1) * full + last)


def secondary(cats, arch, T, P, steps, precision, hbm):
    """Rooflines of the non-dominant kernels from the same event timings: LayerNorm against measured HBM bandwidth
    (algorithmic bytes: read 4d, write 2d per operand plane, per row), attention as algorithmic TFLOP/s (4*T^2*d per layer)."""
    out = {}
    npl = 1 if precision in ("f16", "f16d") else 2  # f16d: LayerNorm writes ONE fp16 plane of differences (the base row it reads is L2-resident)
    rows = P * T
    if "layernorm" in cats and cats["layernorm"]["ms"] > 0:
        byts = 2 * arch.layers * rows * (4 * arch.embed_dim + 2 * arch.embed_dim * npl) * steps
        gbs = byts / (cats["layernorm"]["ms"] / 1e3) / 1e9
        out["layernorm"] = {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm}
    if "attention" in cats and cats["attention"]["ms"] > 0:
        fl = arch.layers * P * 4.0 * T * T * arch.embed_dim * steps
        out["attention"] = {"bound": "tensor+mufu", "achieved": fl / (cats["attention"]["ms"] / 1e3) / 1e12, "unit": "TFLOP/s (algorithmic)"}
    return out


def make_assay(i, L, n_mut):
    from proteingym_b200 import synth
    seq = synth.random_protein(L, seed=i)
    return seq, synth.sample_mutants(seq, n_mut, seed=1000 + i)


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, dev):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(dev)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def window(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, pw, reasons = [], None, [], set()
        for ts, line in list(self.rows):
            if ts < t0 or ts > t1 + 0.3:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx = float(f[1]); pw.append(float(f[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w": statistics.median(pw) if pw else None}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------------------- CPU arm
_CPU_CACHE = {}


def _cpu_forward_fn(arch, state):
    """-> (kind, fn(tokens[1,T]) -> logits): the oracle port of the reference forward (oracle/esm_oracle.py), so the CPU arm
    runs from this repository alone."""
    if "fwd" in _CPU_CACHE:
        return _CPU_CACHE["fwd"]
    from oracle import esm_oracle as O
    kind = "esm2" if arch.kind == "esm2" else "esm1v"
    st = O.load_state(state, kind, torch.float32)
    fn = lambda toks: O.esm_forward(st, toks, kind, arch.layers, arch.heads, arch.token_dropout)
    _CPU_CACHE["fwd"] = ("port", fn)
    return _CPU_CACHE["fwd"]


def cpu_mutants_per_s(arch, state, seconds, threads, L, n_mut):
    """Time the reference's CPU loop body (one batch-1 masked forward + log_softmax row, compute_fitness.py:497-503) on a bounded
    sample of config 2 and extrapolate: mutants/s = N_MUT / ((L+2) * t_forward) — the reference runs L+2 forwards per
    checkpoint (:489) and forward time does not depend on which position is masked. Thread count: the fastest of 8/16/32/64
    (<= host cpus) on a probe at the SAME sequence length (batch-1 forwards regress when oversubscribed)."""
    from oracle import esm_oracle as O
    which, fwd = _cpu_forward_fn(arch, state)
    seq, _ = make_assay(0, L, 10)
    toks = O.tokenize(seq)[None]
    best = _CPU_CACHE.get("best", (None, float("inf")))
    for nt in ([] if best[0] else sorted({t for t in (8, 16, 32, 64) if t <= threads} or {threads})):
        torch.set_num_threads(nt)
        with torch.no_grad():
            fwd(toks)
            t0 = time.time()
            fwd(toks)
            dt = time.time() - t0
        if dt < best[1]:
            best = (nt, dt)
    _CPU_CACHE["best"] = best
    torch.set_num_threads(best[0])
    log(f"cpu arm ({which}): {best[0]} threads (probe at T={toks.shape[1]}: {best[1]:.3f} s)")
    times, t_start, i = [], time.time(), 0
    with torch.no_grad():
        while True:
            tb = toks.clone(); tb[0, 1 + i] = O.MASK_IDX
            t0 = time.time()
            torch.log_softmax(fwd(tb), -1)[:, 1 + i]
            times.append(time.time() - t0)
            i += 1
            if (i >= 3 and time.time() - t_start > seconds) or i >= min(64, L):
                break
    t_fwd = statistics.median(times[1:]) if len(times) > 1 else times[0]
    T = toks.shape[1]
    return n_mut / (T * t_fwd), {"forwards_timed": len(times), "t_forward_s": t_fwd, "T": T, "threads": best[0], "kind": which}


def cpu_sample_text(info):
    return (f"{info['forwards_timed']} batch-1 masked forwards of T={info['T']} (median {info['t_forward_s']:.3f} s each, "
            "oracle port of the reference forward) "
            f"extrapolated x{info['T']} = the reference's L+2 forwards per assay")


# ------------------------------------------------------------------------------------------------ other workloads
def other_workloads(a, rank, world, local_rank, dist, sustained, sampler):
    """Bounded samples of BASELINE configs 3, 4, 5 at the headline precision. Every rank scores its LPT share of a deterministic
    subset of assays; time = max over ranks of the device time between a barrier pair; mutants/s = all mutants of the subset /
    that time."""
    side_prec = "f16f8" if a.precision == "f16d" else a.precision  # f16d is built for the ESM-1b / ESM-1v masked-marginal pass only
    import pandas as pd
    from proteingym_b200 import checkpoint, sharding, synth, workloads
    from proteingym_b200.esm_engine import EsmScorer
    from proteingym_b200.tranception_engine import TranceptionScorer
    from proteingym_b200.trancepteve_engine import TranceptEVEScorer
    dev = torch.device("cuda", local_rank)
    shapes = workloads.load_shapes()
    out = []

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        barrier()
        t_host = time.time()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        per_rank = [ms.clone() for _ in range(world)]
        if dist is not None:
            dist.all_gather(per_rank, ms)
        barrier()
        return res, [float(x.item()) for x in per_rank], (t_host, time.time())

    def share(entries, costs, k, cap):
        picks, info = workloads.pick_subset(entries, costs, k, cap, replicas=world)
        assign = sharding.lpt_assign([costs[i] for i in picks], world)
        return picks, [picks[j] for j in assign[rank]], info

    def record(config, sample, picks, costs, n_mut_total, per_rank, tw, precision=None, extra=None):
        secs = max(per_rank) / 1e3
        tf = sum(costs[i] for i in picks) / 1e12
        out.append({"config": config, "sample": sample, "precision_mode": precision or side_prec, "n_gpus": world, "value": n_mut_total / secs,
                    "unit": "mutants/s", "seconds": secs, "per_rank_ms": per_rank, "algorithmic_tflops": tf / secs,
                    "frac_of_peak": tf / secs / (sustained * world), "clocks": sampler.window(*tw) if sampler else None, **(extra or {})})

    # ---- config 3: ESM2-3B masked-marginals over the DMS_substitutions length distribution ----
    log("config 3: ESM2-3B")
    arch = synth.ESM2_3B
    ents = shapes["substitutions"]
    costs = [workloads.esm_cost(e, arch) for e in ents]
    picks, mine, info = share(ents, costs, 3, 3.0e15)
    from proteingym_b200.esm_engine import choose_precision
    prec3 = choose_precision(checkpoint.config_from_synth(arch), None) if a.precision != "f16" else "f16"  # the CLI's auto rule: f16x3 at this width
    state = checkpoint.normalise_synth_state(arch, synth.make_esm_state(arch, seed=0, device=dev))
    sc = EsmScorer(checkpoint.config_from_synth(arch), state, precision=prec3, device=local_rank)
    del state
    torch.cuda.empty_cache()
    assays = {i: workloads.substitution_assay(ents[i], seed=i, max_mutants=20000) for i in mine}
    sc.score_assay(*workloads.substitution_assay(ents[picks[0]], seed=picks[0], max_mutants=200))  # warm-up
    _, per_rank, tw = timed(lambda: [sc.score_assay(*assays[i]) for i in mine])
    sc.close()
    record("config3: ESM2 3B (36x2560, 40 heads, ffn 10240, rotary) masked-marginals, synthetic assays with the lengths / mutant counts / "
           "multi-mutant shares of reference_files/DMS_substitutions.csv, LPT over the ranks",
           f"{len(picks)} of {len(ents)} assays ({info.get('classes')} size classes evenly spaced over the cost-sorted list x {world} neighbours per class), of the {info.get('eligible')} with cost <= "
           f"{info.get('cost_cap_tflop', 0):.0f} TFLOP ({info.get('dropped_over_cap')} dropped); L = {[ents[i]['L'] for i in picks]}; "
           "mutants capped at 20000 per assay; masked positions = unique mutated positions",
           picks, costs, sum(min(ents[i]["n_mutants"], 20000, 19 * ents[i]["L"]) for i in picks), per_rank, tw, precision=prec3)
    torch.cuda.empty_cache()

    # ---- config 4 / 5: Tranception-L ----
    log("config 4: Tranception-L indels")
    tarch = synth.TRANCEPTION_L
    tstate = {k[len("transformer."):]: v for k, v in synth.make_tranception_state(tarch, 0).items() if k.startswith("transformer.")}
    cfg = {"n_embd": tarch.embed_dim, "n_head": tarch.heads, "n_layer": tarch.layers, "n_ctx": tarch.n_ctx, "n_inner": tarch.ffn_dim,
           "vocab_size": 25}
    ents = shapes["indels"]
    nm = [min(e["n_mutants"], 2000) for e in ents]
    costs = [workloads.tranception_cost(e, tarch, n) for e, n in zip(ents, nm)]
    picks, mine, info = share(ents, costs, 3, 1.0e15)
    tsc = TranceptionScorer(cfg, tstate, precision=side_prec, device=local_rank)
    frames = []
    for i in mine:
        seq, var = workloads.indel_assay(ents[i], seed=i, max_mutants=2000)
        frames.append((seq, pd.DataFrame({"mutant": var, "mutated_sequence": var})))
    wseq = synth.random_protein(64, 1)
    wv = synth.random_indels(wseq, 20, 2)
    tsc.score_mutants(pd.DataFrame({"mutant": wv, "mutated_sequence": wv}), wseq, indel_mode=True)  # warm-up
    _, per_rank, tw = timed(lambda: [tsc.score_mutants(df, seq, indel_mode=True) for seq, df in frames])
    record("config4: Tranception-L (36x1280, 20 heads, n_ctx 1024) autoregressive scoring, both directions + WT, synthetic indel assays "
           "with the lengths / variant counts of reference_files/DMS_indels.csv, LPT over the ranks",
           f"{len(picks)} of {len(ents)} assays ({info.get('classes')} size classes evenly spaced over the cost-sorted list x {world} neighbours per class, {info.get('dropped_over_cap')} over the cap dropped); "
           f"L = {[ents[i]['L'] for i in picks]}; variants capped at 2000 per assay",
           picks, costs, sum(nm[i] for i in picks), per_rank, tw)
    tsc.close()

    log("config 5: TranceptEVE")
    ents = [e for e in shapes["substitutions"] if e["L"] <= 1022]
    nm = [min(e["n_mutants"], 500, 19 * e["L"]) for e in ents]
    costs = [workloads.tranception_cost(e, tarch, n) for e, n in zip(ents, nm)]
    picks, mine, info = share(ents, costs, 2, 1.0e15)
    esc = TranceptEVEScorer(cfg, tstate, full_target_seq="M", precision=side_prec, device=local_rank)
    jobs = []
    for i in mine:
        seq, muts = workloads.substitution_assay(ents[i], seed=i, max_mutants=500)
        jobs.append((seq, pd.DataFrame({"mutant": muts, "mutated_sequence": [synth.apply_mutant(seq, m) for m in muts]}),
                     torch.from_numpy(workloads.synthetic_log_prior(len(seq), 2 * i)),
                     torch.from_numpy(workloads.synthetic_log_prior(len(seq), 2 * i + 1))))

    def run5(js):
        res = []
        for seq, df, p1, p2 in js:  # what the constructor sets up from an MSA + EVE checkpoints, here from synthetic priors
            esc.full_target_seq, esc.full_protein_length = seq, len(seq)
            esc.inference_time_retrieval_type = "TranceptEVE"
            esc.MSA_log_prior, esc.EVE_log_prior, esc.MSA_start, esc.MSA_end = p1, p2, 0, len(seq)
            esc.retrieval_inference_MSA_weight, esc.retrieval_inference_EVE_weight = 0.3, 0.5
            esc.MSA_threshold_focus_cols_frac_gaps, esc.MSA_recalibrate_probas, esc.EVE_recalibrate_probas = 1.0, False, False
            res.append(esc.score_mutants(df, seq))
        return res
    wseq = synth.random_protein(80, 3)
    wm = synth.sample_mutants(wseq, 20, 4)
    run5([(wseq, pd.DataFrame({"mutant": wm, "mutated_sequence": [synth.apply_mutant(wseq, m) for m in wm]}),
           torch.from_numpy(workloads.synthetic_log_prior(80, 1)), torch.from_numpy(workloads.synthetic_log_prior(80, 2)))])  # warm-up
    _, per_rank, tw = timed(lambda: run5(jobs))
    record("config5: TranceptEVE (Tranception-L + MSA prior + EVE prior fused in the LM-head kernel), synthetic substitution assays shaped "
           "like DMS_substitutions with synthetic [L,25] log-priors (SURVEY.md §8d), LPT over the ranks",
           f"{len(picks)} of the {len(ents)} assays with L <= 1022 ({info.get('classes')} size classes evenly spaced over the cost-sorted list x {world} neighbours per class); L = "
           f"{[ents[i]['L'] for i in picks]}; mutants capped at 500 per assay",
           picks, costs, sum(nm[i] for i in picks), per_rank, tw,
           extra={"prefix_reuse_token_rows": {"plain": esc.reuse_rows[0], "run": esc.reuse_rows[1]} if esc.reuse_rows else None})
    esc.close()
    torch.cuda.empty_cache()

    # ---- MSA Transformer (SURVEY.md §8 f3): masked positions of one alignment, the launcher's 400 sampled rows ----
    try:
        log("MSA Transformer")
        from proteingym_b200 import msa_engine
        march = synth.MSA_1B
        mcfg = checkpoint.config_from_msa_synth(march)
        mstate = checkpoint.normalise_msa_synth_state(march, synth.make_msa_state(march, 0, device=dev))
        R, Lm, npos = 400, 512, 8
        toks = msa_engine.tokenize_alignment(synth.random_alignment(synth.random_protein(Lm, seed=100 + rank), R, seed=200 + rank))
        msc = msa_engine.MsaScorer(mcfg, mstate, precision=side_prec, device=local_rank,
                                   max_rows=msa_engine.default_max_rows(mcfg, R, Lm + 1, 1 if side_prec == "f16" else 2, want=4))
        del mstate
        pos = np.linspace(1, Lm, npos).astype(np.int32)
        msc.masked_marginal_rows(toks, pos[:4])  # warm-up
        _, per_rank, tw = timed(lambda: msc.masked_marginal_rows(toks, pos))
        msc.close()
        d_, f_, C_ = march.embed_dim, march.ffn_dim, Lm + 1
        flop = march.layers * (2.0 * R * C_ * (8 * d_ * d_ + 2 * d_ * f_) + 4.0 * C_ * C_ * R * d_ + 4.0 * R * R * C_ * d_)
        secs = max(per_rank) / 1e3
        out.append({"config": "MSA Transformer (MSA-1b: 12 x 768, 12 heads, ffn 3072; tied row attention + column attention) masked-marginals of one "
                              f"synthetic alignment per rank: {R} sampled rows x {Lm} residues (+BOS), {npos} masked positions, 4 per pass",
                    "sample": f"{npos} of the {Lm + 1} columns per rank; one alignment forward per masked position (compute_fitness.py:383-399)",
                    "precision_mode": side_prec, "n_gpus": world, "value": world * npos / secs, "unit": "masked positions/s",
                    "mutants_per_s_all_singles": 19 * world * npos / secs, "seconds": secs, "per_rank_ms": per_rank,
                    "algorithmic_tflop_per_position": flop / 1e12, "algorithmic_tflops": world * npos * flop / 1e12 / secs,
                    "frac_of_peak": npos * flop / 1e12 / secs / sustained, "clocks": sampler.window(*tw) if sampler else None})
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001  (keep the entries of configs 3-5; the shapes are the same on every rank, so is a failure)
        import traceback
        traceback.print_exc(file=sys.stderr)
        out.append({"config": "MSA Transformer", "error": f"{type(e).__name__}: {e}"})
    return out


def main():
    # stdout carries exactly one JSON line: everything else that writes to fd 1 (NCCL's version banner, the progress lines the
    # scoring engines print like the reference does) goes to stderr from here on
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    json_out = os.fdopen(json_fd, "w")
    a = parse()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from proteingym_b200 import synth
    arch = synth.EsmArch("esm1v", 2, 128, 2, 256) if a.small else synth.ESM1V_650M
    L = 64 if a.small else L_SEQ
    n_mut = 200 if a.small else N_MUT
    T = L + 2
    config = {"workload": f"config2: {N_ASSAYS} synthetic assays, L={L} (T={T}) x {n_mut} single mutants, ESM-1v 650M "
                          f"({arch.layers}x{arch.embed_dim}, {arch.heads} heads, ffn {arch.ffn_dim}), masked-marginals, "
                          "one assay per step",
              "assays_per_step": 1, "mutants_per_step": n_mut, "masked_positions_per_step": L,
              "parallelism": f"assay-sharded x{a.gpus} (weights broadcast once, scores gathered once)",
              "l2": "no flush needed: per-step working set (operand-format weights 1.3-2.6 GB + activations >6 GB) >> 126 MB L2"}

    # ------------------------------------------------------------------------------------------------ reference arm
    if a.impl == "reference":
        if rank != 0:
            return
        threads = os.cpu_count() or 1
        state = synth.make_esm_state(arch, seed=0)
        vals, info = [], None
        per_step = max(2.0, min(a.cpu_seconds, 150.0 / max(1, a.steps + a.warmup)))
        for s in range(a.warmup + a.steps):
            v, info = cpu_mutants_per_s(arch, state, per_step, threads, L, n_mut)
            if s >= a.warmup:
                vals.append(v)
        v = statistics.median(vals)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "mutants/s", "n_gpus": a.gpus,
                          "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * n_mut / v, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": "mutants/s", "cores": info["threads"], "host_cpus": threads,
                                           "kind": info["kind"], "sample": cpu_sample_text(info) + " (per step)",
                                           "extrapolated": True,
                                           "note": "one CPU process on rank 0 at every --gpus N (the reference's CPU path has no multi-GPU form)"},
                          "e2e": {"value": v, "unit": "mutants/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), file=json_out, flush=True)
        return

    # ------------------------------------------------------------------------------------------------------ our arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from proteingym_b200 import _lib, checkpoint
    from proteingym_b200.esm_engine import EsmScorer
    lib = _lib.load()

    # weights: rank 0 builds the seeded synthetic checkpoint, NCCL-broadcasts it (north_star: "broadcast of weights")
    state = None
    log("building synthetic weights")
    if rank == 0:
        state = checkpoint.normalise_synth_state(arch, synth.make_esm_state(arch, seed=0))
    if world > 1:
        from proteingym_b200 import sharding
        state = sharding.broadcast_state(state, src=0, device=torch.device("cuda", local_rank))
    sustained, burst, hbm, how = peaks()
    total = a.warmup + a.steps
    my_assays = [make_assay((rank + world * s) % N_ASSAYS, L, n_mut) for s in range(total)]
    sampler = ClockSampler(local_rank) if rank == 0 else None

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_scores(outs):
        """the single final gather of the per-mutant scores (north_star: "a final gather only")"""
        if dist is None:
            return
        mine = torch.stack(outs)
        gathered = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
        dist.gather(mine, gathered, dst=0)

    def measure(precision, with_e2e):
        """One full measurement (device-resident leg, roofline leg, optional end-to-end leg) at the given operand precision."""
        log(f"measure {precision}: upload")
        t_w0 = time.time()
        scorer = EsmScorer(checkpoint.config_from_synth(arch), state, precision=precision, device=local_rank,
                           max_rows=16384 if a.small else 0)
        load_s = time.time() - t_w0
        preps = [scorer.prepare_assay(seq, muts) for seq, muts in my_assays]
        devs = [h.to(scorer.device) for h, _ in preps]
        # ---- leg 1: HBM-resident (value). No profiling events in here. ----
        log(f"measure {precision}: resident leg")
        wout = None
        for s in range(a.warmup):
            wout = scorer.run_assay(preps[s][0], preps[s][1], dev=devs[s])
        # NCCL opens its send/recv channels on first use: run the exact gather once before the timed region
        gather_scores([wout if wout is not None else torch.zeros(n_mut, device=scorer.device)] * a.steps)
        barrier()
        launches0 = lib.pg_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_host0 = time.time()
        e0.record()
        outs = [scorer.run_assay(preps[s][0], preps[s][1], dev=devs[s]) for s in range(a.warmup, total)]
        gather_scores(outs)
        e1.record()
        barrier()
        t_host1 = time.time()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        per_rank = [ms.clone() for _ in range(world)]
        if dist is not None:
            dist.all_gather(per_rank, ms)
        per_rank = [float(x.item()) for x in per_rank]
        ms_total = max(per_rank)
        launches = lib.pg_launch_count() - launches0
        clocks = sampler.window(t_host0, t_host1) if sampler else None
        res = {"value": world * a.steps * n_mut / (ms_total / 1e3), "ms_per_step": ms_total / a.steps, "gpu_launches": int(launches),
               "clocks": clocks, "weight_load_s": load_s,
               "per_rank_ms": {"min": min(per_rank), "median": statistics.median(per_rank), "max": max(per_rank)},
               "last_scores": outs[-1].cpu().numpy()}
        # ---- leg 2: the same K steps with a CUDA-event pair around every kernel -> per-kernel times for the roofline ----
        log(f"measure {precision}: roofline leg")
        barrier()
        lib.pg_profile_begin()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for s in range(a.warmup, total):
            scorer.run_assay(preps[s][0], preps[s][1], dev=devs[s])
        r1.record()
        barrier()
        ncat = len(_lib.PROFILE_CATEGORIES)
        cat_ms = (C.c_float * ncat)(); cat_n = (C.c_int32 * ncat)()
        lib.pg_profile_end(cat_ms, cat_n, ncat)
        prof_ms = r0.elapsed_time(r1)
        # ---- leg 3: end to end through the public API with host buffers ----
        if with_e2e:
            log(f"measure {precision}: e2e leg")
            for s in range(min(2, a.warmup)):
                scorer.score_assay(*my_assays[s])
            barrier()
            t0 = time.time()
            e2e_scores = []
            for s in range(a.warmup, total):
                e2e_scores.append(scorer.score_assay(*my_assays[s]))
            barrier()
            e2e_s = torch.tensor([time.time() - t0], device="cuda")
            if dist is not None:
                dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
            same = all(np.array_equal(e2e_scores[i], outs[i].cpu().numpy()) for i in range(len(outs)))
            res["e2e"] = {"value": world * a.steps * n_mut / float(e2e_s.item()), "unit": "mutants/s",
                          "h2d_bytes_per_step": int(preps[a.warmup][0].numel() * 4), "d2h_bytes_per_step": int(n_mut * 4),
                          "bit_identical_to_resident_leg": bool(same)}
        # ---- leg 4 (N > 1): strong scaling — ONE assay per step, its masked positions partitioned over the ranks, the [P, vocab]
        #      table completed by one NCCL all-gather per step (compute_fitness --partition positions) ----
        if with_e2e and dist is not None:
            log(f"measure {precision}: strong-scaling leg")
            seq0, muts0 = make_assay(0, L, n_mut)
            h0, z0 = scorer.prepare_assay(seq0, muts0)
            d0 = h0.to(scorer.device)
            for s in range(max(1, a.warmup)):
                sc = scorer.run_assay(h0, z0, dev=d0, shard=(rank, world))
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for s in range(a.steps):
                sc = scorer.run_assay(h0, z0, dev=d0, shard=(rank, world))
            s1.record()
            barrier()
            sms = torch.tensor([s0.elapsed_time(s1)], device="cuda")
            dist.all_reduce(sms, op=dist.ReduceOp.MAX)
            ref = sc.clone()
            dist.broadcast(ref, src=0)
            same = torch.tensor([int(torch.equal(ref, sc))], device="cuda")
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            res["strong_scaling"] = {"workload": "ONE config-2 assay per step, masked positions partitioned over the ranks "
                                                 "(--partition positions), one all-gather of the table per step",
                                     "value": a.steps * n_mut / (float(sms.item()) / 1e3), "unit": "mutants/s", "scaling": "strong",
                                     "ms_per_step": float(sms.item()) / a.steps, "n_gpus": world,
                                     "scores_identical_on_every_rank": bool(same.item())}
        # ---- roofline of the dominant kernel (tcgen05 GEMM) from the event timings of leg 2 ----
        cats = {n: {"ms": float(cat_ms[i]), "launches": int(cat_n[i])} for i, n in enumerate(_lib.PROFILE_CATEGORIES) if cat_n[i]}
        P = preps[a.warmup][1]["P"]
        f_total, f_lin = algorithmic_flops(arch, T, P)
        gemm_ms = sum(cats[c]["ms"] for c in cats if c.startswith("gemm_"))
        gemm_launches = sum(cats[c]["launches"] for c in cats if c.startswith("gemm_"))
        achieved = (f_lin * a.steps / 1e12) / (gemm_ms / 1e3) if gemm_ms > 0 else None
        issued = (issued_linear_flops(arch, T, P, PASSES[precision]) * a.steps / 1e12) / (gemm_ms / 1e3) if gemm_ms > 0 else None
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
                traffic = json.load(fh).get(precision)
        except Exception:
            pass
        res["roofline"] = {
            "bound": "tensor", "kernel": "gemm_tc_kernel (CTA pairs: tcgen05.mma cta_group::2 kind::f16 [+ kind::f8f6f4 cross terms in f16f8; shared base "
                                         "rows added in the epilogue in f16d], 256x256 tile per pair, packed-fp32 epilogue, TMA 6-stage ring, "
                                         "chunked RN accumulation, TMA-store epilogue)",
            "achieved": achieved, "peak": sustained, "unit": "TFLOP/s", "frac": (achieved / sustained) if achieved else None,
            "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({how}); burst {burst}",
            "algorithmic_flops_per_launch": f_lin * a.steps / max(1, gemm_launches), "launches": gemm_launches,
            "avg_launch_ms": gemm_ms / max(1, gemm_launches), "tensor_pipe_work_multiplier": PASSES[precision],
            "issued_tflops": issued, "issued_frac": (issued / sustained) if issued else None, "traffic": traffic,
            "timed_in": f"separate roofline pass of the same {a.steps} steps ({prof_ms:.1f} ms with per-kernel events vs {ms_total:.1f} ms "
                        "in the value leg)",
            "whole_step": {"algorithmic_tflop_per_step": f_total / 1e12,
                           "achieved_per_gpu": f_total * a.steps / 1e12 / (ms_total / 1e3),
                           "frac_of_peak": f_total * a.steps / 1e12 / (ms_total / 1e3) / sustained},
            "kernel_ms_in_timed_region": cats,
            "secondary": secondary(cats, arch, T, P, a.steps, precision, hbm)}
        scorer.close()
        del scorer, devs
        torch.cuda.empty_cache()
        return res

    cpu_state = {k: v.cpu() for k, v in state.items()} if (rank == 0 and world == 1 and not a.no_cpu_baseline) else None
    main_res = measure(a.precision, with_e2e=True)
    if a.dump_outputs and rank == 0:
        os.makedirs(a.dump_outputs, exist_ok=True)
        np.save(os.path.join(a.dump_outputs, "scores.npy"), main_res["last_scores"].astype(np.float32))
    others = [] if (a.small or a.no_other_modes) else [(m, measure(m, with_e2e=False)) for m in ("f16d", "f16f8", "f16x3", "f16") if m != a.precision]
    del state
    torch.cuda.empty_cache()
    extra = None
    if not a.small and not a.no_other_workloads:
        try:
            extra = other_workloads(a, rank, world, local_rank, dist, sustained, sampler)
        except Exception as e:  # noqa: BLE001  (the headline line must survive a failure in the side workloads at N = 1)
            import traceback
            traceback.print_exc(file=sys.stderr)
            if dist is not None:
                raise  # the other ranks may be waiting in a collective: fail the whole job loudly instead of hanging
            extra = [{"error": f"{type(e).__name__}: {e}"}]
    if sampler:
        sampler.stop()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    DT = {"f16f8": "f16f8 (linear layers: fp16 hi*hi + e4m3 cross terms = 2 tensor-pipe units; attention fp16 hi/lo x3; chunked RN fp32 "
                   "accumulation; fp32 residual/LayerNorm/softmax/head; meets 1e-3 parity)",
          "f16x3": "f16x3 (fp16 hi+lo operand pairs, 3 tcgen05 passes, fp32 accumulate/residual/softmax; meets 1e-3 parity)",
          "f16d": "f16d (delta operands: every linear layer = shared base row at fp16 hi/lo x3, computed once per window, + ONE fp16 pass on "
                  "the per-copy difference = 1 tensor-pipe unit; masked rows exact (x3); attention fp16 hi/lo x3; fp32 residual/LayerNorm/"
                  "softmax/head; meets 1e-3 parity)",
          "f16": "f16 (single fp16 pass, fp32 accumulate; ~1e-2 abs error, Spearman > 0.999; does NOT meet the 1e-3 parity bar)"}
    out = {"metric": METRIC, "value": main_res["value"], "unit": "mutants/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": DT[a.precision], "data": "synthetic", "config": config, "precision_mode": a.precision,
           "e2e": main_res["e2e"], "gpu_launches": main_res["gpu_launches"], "clocks": main_res["clocks"],
           "per_rank_ms": main_res["per_rank_ms"], "roofline": main_res["roofline"], "weight_load_s": main_res["weight_load_s"]}
    out["other_precision_modes"] = [
        {"precision_mode": m, "dtype": DT[m], "value": r["value"], "unit": "mutants/s", "ms_per_step": r["ms_per_step"], "clocks": r["clocks"],
         "roofline": {k: r["roofline"][k] for k in ("achieved", "frac", "issued_tflops", "issued_frac", "whole_step",
                                                    "kernel_ms_in_timed_region", "secondary")}} for m, r in others]
    if "strong_scaling" in main_res:
        out["strong_scaling"] = main_res["strong_scaling"]
    if extra is not None:
        out["other_workloads"] = extra

    if not a.no_cpu_baseline and world == 1:
        log("cpu baseline")
        threads = os.cpu_count() or 1
        v, info = cpu_mutants_per_s(arch, cpu_state, a.cpu_seconds, threads, L, n_mut)
        out["cpu_baseline"] = {"value": v, "unit": "mutants/s", "cores": info["threads"], "host_cpus": threads, "kind": info["kind"],
                               "sample": cpu_sample_text(info), "extrapolated": True}
    print(json.dumps(out), file=json_out, flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
