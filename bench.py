#!/usr/bin/env python
"""bench.py -- CTU-analysis throughput (CTUs/s) of the B200 block-primitive path on the BASELINE.json configs.

  --config c3 (default) : 3840x2160  8-bit preset slow    : 4 refs, STAR, merange 57, subme 3, rect, chroma-SATD on (4:2:0)
  --config c4           : 3840x2160 10-bit preset slower  : 5 refs, subme 4, rect + AMP, chroma-SATD on
  --config c5           : 7680x4320 10-bit preset veryslow: 5 refs, subme 4, rect + AMP, chroma-SATD on
  --config c2           : 1920x1080  8-bit preset medium lookahead: Lowres init + intra + estimateFrameCost over a 20-frame
                          window (bframes 4); metric = lowres CUs/s; N>1 shards the lookahead FRAMES (owner(b) = b % N)

A step (c3/c4/c5) = one pass of the hot path over one frame per GPU: every PU of every CTU x every reference through
motionEstimate (STAR + sub-pel, chroma-SATD term as MotionEstimate::bChromaSATD runs it, motion.cpp:204-212), then per CU
the fused MC -> residual -> DCT -> quant -> dequant -> IDCT -> recon -> SSE chain, then the 35-mode intra SA8D search.

  value : whole-job units/s with inputs resident in HBM (kernels only, CUDA events, L2 flushed between steps)
  e2e   : same metric through the public call (x265_b200.Analyser.analyse / Lookahead) with pinned HOST buffers,
          H2D of the inputs and D2H of the results inside the timed region
  checks: order-sensitive checksums of the results; the CPU legs compute the same fields on the same geometry
          (full frame, or its first k CTU rows) and the GPU arm ASSERTS equality on that scope (exit code 3 otherwise)
  --impl reference : the same workload on the reference's own C code (oracle/_ref: MotionEstimate class + C primitive
          table compiled from /root/reference) on all host cores.

Multi-GPU (torchrun, one process per GPU):
  --shard frames (default): each rank analyses its own frame (weak scaling); the one exchange is the NCCL broadcast of the
          newest reconstructed reference plane from its owner, issued on a side stream and overlapped with the step.
  --shard rows : ONE frame per step, its CTU rows dealt to the ranks (strong scaling, BASELINE configs[4]), every owner
          broadcasting its reconstructed rows afterwards.

  --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned to its caller as
          DIR/<name>.npy (float64, exact for these integer results; at most 64 MB, larger outputs as a fixed seeded
          row sample whose indices are written beside it).  The inputs are seeded, so two builds run with the same
          arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# the benchmark may run from a read-only tree: no bytecode caches next to the sources
sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# preset table: common/param.cpp:478-534 (slow / slower / veryslow), search.cpp:2059-2060 (bChromaSATD for 4:2:0)
CONFIGS = {
    "c3": dict(W=3840, H=2160, depth=8, refs=4, method=3, subme=3, merange=57, rect=1, amp=0, chroma=True, qp=30,
               label="3840x2160 8-bit preset slow: full ME + sub-pel interp (chroma-SATD on) + DCT/quant + intra primitives on device (BASELINE configs[2])"),
    "c4": dict(W=3840, H=2160, depth=10, refs=5, method=3, subme=4, merange=57, rect=1, amp=1, chroma=True, qp=30,
               label="3840x2160 10-bit Main10 preset slower: 5 refs, subme 4, rect + AMP PUs, chroma-SATD on (BASELINE configs[3] analysis part)"),
    "c5": dict(W=7680, H=4320, depth=10, refs=5, method=3, subme=4, merange=57, rect=1, amp=1, chroma=True, qp=30,
               label="7680x4320 10-bit preset veryslow: 5 refs, subme 4, rect + AMP PUs, chroma-SATD on (BASELINE configs[4])"),
    "c2": dict(W=1920, H=1080, depth=8, frames=20, bframes=4, lookahead=True, lslices=0,
               label="1920x1080 8-bit preset medium lookahead: Lowres init + lowresIntraEstimate + estimateFrameCost (HEX, subme 1 lowres) on device (BASELINE configs[1])"),
}
CFG = None          # the selected config dict (set in main)
CFG_NAME = "c3"


def ctus_per_frame():
    return ((CFG["W"] + 63) // 64) * ((CFG["H"] + 63) // 64)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def host_cores():
    """Usable host cores: os.cpu_count() capped by the cgroup CPU quota and the affinity mask."""
    n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    return n


def asm_status():
    """The reference's AVX2/AVX-512 primitives are NASM sources (common/x86/*.asm); they can only be built where an
    assembler exists.  Reported with every CPU number so that a ratio is never read as 'vs AVX-512'."""
    for tool in ("nasm", "yasm"):
        for d in os.environ.get("PATH", "").split(os.pathsep):
            if d and os.path.exists(os.path.join(d, tool)):
                return "%s present at %s but oracle/_ref is the C-primitive build (no asm objects were assembled)" % (tool, d)
    return "unavailable (no nasm/yasm on this box): CPU arm = the reference's C primitives (--no-asm path)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
def workload_config(shard="frames"):
    """The config dict of BOTH arms (identical by construction)."""
    c = CFG
    if c.get("lookahead"):
        return {"workload": c["label"], "config": CFG_NAME, "frames": c["frames"], "bframes": c["bframes"],
                "lowres_cus_per_frame": ((c["W"] // 2 + 7) // 8) * ((c["H"] // 2 + 7) // 8),
                "estimates": "P costs at every anchor distance <= bframes+1 and the B costs between them (x265_b200.lookahead.window_triples)",
                "unit_definition": "lowres CUs of estimateFrameCost per second (frame costs x CUs per frame); the GPU step ALSO does Lowres init + intra of all frames",
                "l2": "256 MiB memset between timed steps (untimed)",
                "shard": "lookahead frames: owner(b) = b % N runs every estimate of frame b; each frame's 4 lowres planes are broadcast once from its owner (N>1 only)"}
    out = {"workload": c["label"], "config": CFG_NAME, "ctus_per_frame": ctus_per_frame(), "refs": c["refs"], "search": "star", "merange": c["merange"],
           "subme": c["subme"], "rect": c["rect"], "amp": c["amp"], "chroma_satd": bool(c["chroma"]), "qp": c["qp"], "bit_depth": c["depth"],
           "l2": "256 MiB memset between timed steps (untimed) + >300 MB per-step working set",
           "frames": "rank k: frame refs+k against frames refs-1+k..k (frame-parallel: own nearest references per frame)"}
    if shard == "rows":
        out["frames_per_step"] = "1 per step, CTU rows sharded over the GPUs (contiguous row blocks)"
        out["exchange"] = "NCCL broadcast of every owner's reconstructed CTU rows (one luma plane in total) per step (N>1 only)"
    else:
        out["frames_per_step"] = "1 per GPU"
        out["exchange"] = "NCCL broadcast of one reference luma plane per step on a side stream, overlapped with the analysis (N>1 only)"
    return out


def checks_of(cost, mvx, mvy, numsig, sse, intra, nj, nc):
    """Order-sensitive checksums over the first nj PU jobs / nc CUs (both arms compute exactly these)."""
    cost = np.asarray(cost[:nj]).astype(np.int64)
    mvx = (np.asarray(mvx[:nj]).astype(np.int64) & 0xffff).astype(np.uint64)
    mvy = (np.asarray(mvy[:nj]).astype(np.int64) & 0xffff).astype(np.uint64)
    idx = np.arange(nj, dtype=np.uint64)
    mv_hash = int(((mvx * (idx % np.uint64(251) + np.uint64(1))) + (mvy * (idx % np.uint64(241) + np.uint64(1)))).sum(dtype=np.uint64) & np.uint64((1 << 62) - 1))
    intra = np.asarray(intra[:nc])
    return {"jobs": int(nj), "cus": int(nc), "me_cost_sum": int(cost.sum()), "mv_hash": mv_hash,
            "numsig_sum": int(np.asarray(numsig[:nc]).astype(np.int64).sum()), "sse_sum": int(np.asarray(sse[:nc]).astype(np.uint64).sum()),
            "intra_cost_sum": int(intra[:, :35].astype(np.int64).sum()), "intra_mode_hist_hash": int((intra[:, 35].astype(np.int64) * (np.arange(nc) % 97 + 1)).sum())}


def cpu_reference(max_rows, threads, kind_pref="reference", steps=1, warmup=0, wl=None):
    """The same workload on host cores: reference-from-source driver (oracle/_ref) or the oracle port, over the first
    `max_rows` CTU rows of the FULL-frame geometry (0 = the whole frame)."""
    from common import load_ref, load_oracle
    from frame_helpers import Workload, cpu_analyse, lambda_for
    from me_helpers import mvcost_table
    c = CFG
    O = load_oracle(c["depth"])
    R = load_ref(c["depth"]) if kind_pref == "reference" else None
    lib, fn, kind = (R, "x265ref_analyse_frame", "reference") if R is not None else (O, "orc_analyse_frame", "port")
    if wl is None:
        wl = Workload(c["W"], c["H"], depth=c["depth"], numRefs=c["refs"], method=c["method"], subme=c["subme"], merange=c["merange"],
                      rect=c["rect"], qp=c["qp"], chroma=c["chroma"], amp=c["amp"])
    tab = mvcost_table(O, lambda_for(c["qp"], c["depth"]))
    total_rows = (c["H"] + 63) // 64
    rows = total_rows if max_rows <= 0 or max_rows >= total_rows else max_rows
    ctus = ((c["W"] + 63) // 64) * rows
    for _ in range(warmup):
        cpu_analyse(lib, fn, wl, tab, threads=threads, max_ctu_rows=rows)
    t0 = time.perf_counter()
    for _ in range(steps):
        res = cpu_analyse(lib, fn, wl, tab, threads=threads, max_ctu_rows=rows)
    dt = time.perf_counter() - t0
    nj, nc = res["njobs_run"], res["ncu_run"]
    chk = checks_of(res["me_out"][:, 0], res["me_out"][:, 1], res["me_out"][:, 2], res["cu_numsig"], res["cu_sse"], res["intra_cost"], nj, nc)
    scope = "whole frame" if rows == total_rows else "CTU rows [0, %d) of %d (full-frame geometry)" % (rows, total_rows)
    return {"ctus_per_s": ctus * steps / dt, "seconds": dt, "ctus": ctus, "kind": kind, "threads": threads, "rows": rows, "whole": rows == total_rows,
            "sample": "%s of the %dx%d workload, %d refs, all PUs, %d step(s)" % (scope, c["W"], c["H"], c["refs"], steps),
            "checks": chk, "scope": scope, "wl": wl, "jobs": res["jobs"][:nj], "me_out": res["me_out"][:nj]}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    if CFG.get("lookahead"):
        return run_lookahead_reference(args)
    threads = host_cores()
    total_rows = (CFG["H"] + 63) // 64
    # size the per-step sample so that the whole run stays within a few minutes; the probe step is the warm-up
    probe = cpu_reference(1, threads, steps=1)
    per_row = probe["seconds"]
    budget = 170.0 / max(1, args.steps)
    rows = int(max(1, min(total_rows, budget / max(per_row, 1e-3))))
    r = cpu_reference(rows, threads, steps=args.steps, warmup=0, wl=probe["wl"])
    line = {"impl": "reference", "metric": "2160p preset-slow CTU-analysis throughput", "value": r["ctus_per_s"], "unit": "CTUs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * r["seconds"] / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.shard == "rows" else "weak", "vs_baseline": None,
            "dtype": "u8" if CFG["depth"] == 8 else "u16", "data": "synthetic",
            "config": workload_config(args.shard),
            "cpu_baseline": {"value": r["ctus_per_s"], "unit": "CTUs/s", "cores": threads, "kind": r["kind"], "sample": r["sample"], "asm": asm_status(),
                             "warmup_note": "one 1-row probe step is the warm-up (the CPU arm has no caches worth more)"},
            "e2e": {"value": r["ctus_per_s"], "unit": "CTUs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "checks": r["checks"], "checks_scope": r["scope"], "gpu_launches": 0}
    if CFG["chroma"] and not args.no_pred:
        # the prediction costs around the motion search (Search::selectMVP / mergeEstimation / bidir) of the rows just analysed, on
        # the reference's own Predict / MotionEstimate classes: the same job list the GPU arm's `pred_cost` leg evaluates
        try:
            pj = pred_jobs_of(r["jobs"], r["me_out"], CFG["refs"], True)
            pr = pred_cpu(r["wl"], pj, threads, 8.0)
            if pr is not None:
                line["pred_cost"] = {"jobs_per_s": pr["jobs_per_s"], "cores": pr["threads"], "kind": "reference", "sample": "first %d of %d jobs (4 per motion-search job of %s)" % (pr["jobs"], len(pj), r["scope"]),
                                     "checks": pred_checks(pr["cost"])}
        except Exception as e:
            line["pred_cost_error"] = repr(e)
    print(json.dumps(line), flush=True)


DUMP_LIMIT = 64 << 20


def sample_rows(n, k, seed):
    """Sorted indices of a fixed, seeded sample of k of n rows (all n rows when n <= k)."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def write_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float64 (the results are integers below 2**53)."""
    arrays = {k: np.ascontiguousarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise ValueError("outputs to dump take %d bytes, more than %d" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def analysis_outputs(an):
    """What Analyser.analyse hands its caller: per motion-search job the cost and the vector (quarter-pel), per CU the SSE,
    the significant-coefficient count, the chosen reference and the 35 intra costs + the best mode.  A 2160p frame has
    millions of jobs, so jobs and CUs are sampled at fixed seeded rows (job_index, cu_index)."""
    jobs = sample_rows(an.njobs, 1 << 18, 1)
    cus = sample_rows(an.ncu, 1 << 16, 2)
    mvp = an.me_packed[jobs, 1].view(np.uint32)
    return {"job_index": jobs, "me_cost": an.me_packed[jobs, 0],
            "mv_x": (mvp & 0xffff).astype(np.uint16).view(np.int16), "mv_y": (mvp >> 16).astype(np.uint16).view(np.int16),
            "cu_index": cus, "cu_sse": an.cu_sse[cus], "cu_numsig": an.cu_numsig[cus], "cu_ref": an.cu_ref[cus],
            "intra_cost": an.intra_cost[cus]}


def plane_as_tensor(torch, ptr, nbytes, device):
    class _Wrap:
        pass
    w = _Wrap()
    w.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}
    return torch.as_tensor(w, device=device)


def primitives_leg(lib, reps=3):
    """Per-primitive half of the metric: achieved HBM GB/s of every primitive class at frame scale, 8- and 10-bit
    (profiles/primitive_bench.py), with the ncu DRAM bytes of the committed capture of the same launches when present."""
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import primitive_bench
    dram = {}
    try:
        for row in json.load(open(os.path.join(ROOT, "profiles", "primitives_r2_ncu.json")))["rows"]:
            dram[(row["kernel"], row["depth"])] = row.get("dram_bytes")
    except Exception:
        pass
    out = []
    for depth in (8, 10):
        for row in primitive_bench.run(lib, depth=depth, reps=reps, frames=24, quiet=True):
            out.append({"kernel": row["kernel"], "depth": depth, "GBps": round(row["GBps"], 1), "frac": round(row["frac_of_measured_peak"], 4),
                        "algorithmic_bytes": int(row["algorithmic_MB"] * 1e6), "dram_bytes": dram.get((row["kernel"], depth)), "note": row["note"]})
    return out


def pred_jobs_of(jobs, me_out, nrefs, chroma):
    """Four prediction costs per motion-search job (PU, reference r), as predInterSearch asks around motionEstimate:
    the two AMVP candidates' SADs (Search::selectMVP: the job's MVP and its first MV candidate), one merge candidate's SATD
    (uni, the second MV candidate) and one bi-prediction (the search result on r with the MVP on the next reference).  Vectors
    are clipped to the job's search window (quarter-pel), as CUData::clipMv / setSearchRange keep them inside the padded
    picture.  With the chroma-SATD term on (presets >= subme 3) the SATD jobs carry it and the bi job is the addAvg path;
    without it the bi job is the pixelavg_pp estimate (search.cpp:2499-2510)."""
    from x265_b200.lib import PRED_JOB, PRED_CHROMA, PRED_AVG_PP
    n = len(jobs)
    lo = jobs["mvmin"].astype(np.int32) * 4; hi = jobs["mvmax"].astype(np.int32) * 4
    clip = lambda v: np.clip(v.astype(np.int32), lo, hi).astype(np.int16)
    pj = np.zeros((n, 4), PRED_JOB)
    for k in range(4):
        pj[:, k]["offset"] = jobs["offset"]; pj[:, k]["pw"] = jobs["pw"]; pj[:, k]["ph"] = jobs["ph"]
        pj[:, k]["ref0"] = jobs["ref"]; pj[:, k]["ref1"] = -1
    pj[:, 0]["mv0"] = clip(jobs["qmvp"]); pj[:, 1]["mv0"] = clip(jobs["mvc"][:, 0:2]); pj[:, 2]["mv0"] = clip(jobs["mvc"][:, 2:4])
    pj[:, 2]["cost"] = 1; pj[:, 3]["cost"] = 1
    pj[:, 2]["flags"] = PRED_CHROMA if chroma else 0
    pj[:, 3]["flags"] = PRED_CHROMA if chroma else PRED_AVG_PP
    pj[:, 3]["mv0"] = me_out[:n, 1:3].astype(np.int16)
    pj[:, 3]["ref1"] = (jobs["ref"] + 1) % nrefs
    pj[:, 3]["mv1"] = clip(jobs["qmvp"])
    return pj.reshape(-1)


def pred_checks(cost):
    cost = np.asarray(cost).astype(np.int64)
    idx = np.arange(cost.size, dtype=np.int64)
    return {"jobs": int(cost.size), "cost_sum": int(cost.sum()), "cost_hash": int((cost * (idx % 239 + 1)).sum() & ((1 << 62) - 1))}


def pred_cpu(wl, pj, threads, budget_s):
    """Reference arm of the prediction-cost leg: the real Predict / MotionEstimate classes (oracle/_ref: x265ref_pred_cost_batch)
    over the first jobs of the list, sized to `budget_s` seconds of host time."""
    from common import load_ref
    c = CFG
    R = load_ref(c["depth"])
    if R is None:
        return None
    es = 1 if c["depth"] == 8 else 2
    nref = len(wl.refs)
    PA = C.c_void_p * nref
    refs = PA(*[r.ctypes.data + wl.org * es for r in wl.refs])
    rcb = PA(*[wl.refC[r][0].ctypes.data + wl.corg * es for r in range(nref)])
    rcr = PA(*[wl.refC[r][1].ctypes.data + wl.corg * es for r in range(nref)])
    R.x265ref_pred_cost_batch.restype = C.c_int
    R.x265ref_pred_cost_batch.argtypes = [C.c_void_p] * 6 + [C.c_ssize_t, C.c_ssize_t, C.c_void_p, C.c_int, C.c_void_p, C.c_int]

    def run(m):
        out = np.zeros(m, np.int32)
        t0 = time.perf_counter()
        R.x265ref_pred_cost_batch(wl.fenc.ctypes.data + wl.org * es, wl.fencC[0].ctypes.data + wl.corg * es, wl.fencC[1].ctypes.data + wl.corg * es,
                                  refs, rcb, rcr, wl.stride, wl.cstride, pj.ctypes.data, m, out.ctypes.data, threads)
        return out, time.perf_counter() - t0
    m0 = min(len(pj), 40000)
    out, dt = run(m0)
    m = int(min(len(pj), max(m0, m0 * budget_s / max(dt, 1e-4))))
    if m > m0:
        out, dt = run(m)
    return {"jobs": m, "seconds": dt, "jobs_per_s": m / dt, "cost": out, "threads": threads}


def pred_cost_leg(lib, an, wl, cpu_seconds, reps=3):
    """The prediction costs around the motion search (x265cu_pred_cost_batch) for the analysed frame: job list derived from
    the frame's motion-search jobs and results (pred_jobs_of), planes as the analyser holds them, device time by CUDA events;
    the CPU arm runs the reference's own classes on the first jobs of the same list and the costs are compared exactly."""
    c = CFG
    es = 1 if c["depth"] == 8 else 2
    jobs = an.fetch("jobs"); me = an.fetch("me_out").reshape(-1, 4)
    pj = pred_jobs_of(jobs, me, c["refs"], True)
    d_f = lib.to_device(wl.fenc); d_r = [lib.to_device(r) for r in wl.refs]
    d_fc = [lib.to_device(x) for x in wl.fencC]; d_rc = [[lib.to_device(x) for x in rc] for rc in wl.refC]
    tab = lib.to_device(np.array([d.ptr + wl.org * es for d in d_r], np.uint64))
    tcb = lib.to_device(np.array([rc[0].ptr + wl.corg * es for rc in d_rc], np.uint64))
    tcr = lib.to_device(np.array([rc[1].ptr + wl.corg * es for rc in d_rc], np.uint64))
    d_j = lib.to_device(pj); d_o = lib.alloc(4 * len(pj))

    class _At:                      # a device pointer at the plane's pixel (0, 0)
        def __init__(self, buf, off): self.ptr = buf.ptr + off
    chroma = (_At(d_fc[0], wl.corg * es), _At(d_fc[1], wl.corg * es), tcb, tcr, wl.cstride)
    call = lambda: lib.pred_cost_batch(c["depth"], _At(d_f, wl.org * es), wl.stride, tab, wl.stride, chroma, d_j, len(pj), d_o)
    call(); lib.sync()
    ts = []
    for _ in range(reps):
        lib.timer_begin(); call(); ts.append(lib.timer_end())
    ms = float(np.median(ts))
    got = d_o.download(np.int32)
    out = {"what": "AMVP candidate SADs (Search::selectMVP), merge-candidate and bi-prediction SATD + chroma SATD (mergeEstimation, predInterSearch bidir) on Predict::motionCompensation: 4 costs per motion-search job",
           "jobs": int(len(pj)), "ms": ms, "jobs_per_s": len(pj) / (ms / 1000.0), "checks": pred_checks(got), "launches_per_call": 4}
    if cpu_seconds > 0:
        r = pred_cpu(wl, pj, host_cores(), cpu_seconds)
        if r is not None:
            m = r["jobs"]
            out["cpu"] = {"jobs_per_s": r["jobs_per_s"], "cores": r["threads"], "kind": "reference", "sample": "first %d jobs of the list" % m,
                          "checks": pred_checks(r["cost"])}
            out["gpu_checks_on_sample"] = pred_checks(got[:m])
            out["checks_equal"] = bool(np.array_equal(got[:m], r["cost"]))
    for d in [d_f, tab, tcb, tcr, d_j, d_o] + d_r + d_fc + [x for rc in d_rc for x in rc]:
        d.free()
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    import x265_b200
    from x265_b200 import shard
    from frame_helpers import gen_luma, gen_chroma, make_field, MARGIN_X, MARGIN_Y
    c = CFG
    W, H, DEPTH, NREFS, CHROMA = c["W"], c["H"], c["depth"], c["refs"], c["chroma"]
    pdt = np.uint8 if DEPTH == 8 else np.uint16
    es = 1 if DEPTH == 8 else 2
    dist = None
    if world > 1:
        import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = x265_b200.load(local_rank)
    an = x265_b200.Analyser(lib, W, H, depth=DEPTH, numRefs=NREFS, method=c["method"], subme=c["subme"], merange=c["merange"], rect=c["rect"],
                            qp=c["qp"], amp=c["amp"])
    # synthetic clip (BASELINE.md generator).  Frame shards: rank k analyses frame NREFS + k against ITS nearest previous frames,
    # as frame-parallel encoding does, so every rank has the same temporal distances and the same search problem.
    # Row shards: one frame and one reference set for all ranks.
    rows_mode = args.shard == "rows"
    k_frame = 0 if rows_mode else shard.frame_of(0, rank, world)
    for r in range(NREFS):
        an.set_ref(r, gen_luma(W, H, NREFS - 1 - r + k_frame, bits=DEPTH))
    cur = gen_luma(W, H, NREFS + k_frame, bits=DEPTH)
    my_rows = shard.row_blocks(an.ctu_rows, rank, world, "block") if rows_mode else [(0, an.ctu_rows)]
    field = make_field(W, H, NREFS)
    # pinned host buffers: these are what the user hands to the public call
    pin = lib.L.x265cu_host_alloc(W * H * es)
    h_fenc = np.frombuffer((C.c_uint8 * (W * H * es)).from_address(pin), pdt).reshape(H, W)
    h_fenc[:] = cur
    pinf = lib.L.x265cu_host_alloc(field.nbytes)
    h_field = np.frombuffer((C.c_uint8 * field.nbytes).from_address(pinf), np.int16).reshape(field.shape)
    h_field[:] = field
    h_cb = h_cr = None
    if CHROMA:
        # the reference runs subme >= 3 on a 4:2:0 source with MotionEstimate::bChromaSATD on (motion.cpp:204-212)
        an.enable_chroma()
        for r in range(NREFS):
            an.set_ref_chroma(r, gen_chroma(W, H, NREFS - 1 - r + k_frame, 1, bits=DEPTH), gen_chroma(W, H, NREFS - 1 - r + k_frame, 2, bits=DEPTH))
        cf = NREFS + k_frame
        cbytes = W * H // 4 * es
        pc = [lib.L.x265cu_host_alloc(cbytes) for _ in range(2)]
        h_cb, h_cr = [np.frombuffer((C.c_uint8 * cbytes).from_address(p), pdt).reshape(H // 2, W // 2) for p in pc]
        h_cb[:] = gen_chroma(W, H, cf, 1, bits=DEPTH); h_cr[:] = gen_chroma(W, H, cf, 2, bits=DEPTH)
        an.load_chroma(h_cb, h_cr)
    flush = lib.alloc(256 << 20)
    ref0 = incoming = None
    side = None
    if world > 1:
        ptr, stride = an.recon_plane_ptr(1) if rows_mode else an.ref_plane_ptr(0)
        base = ptr - (MARGIN_Y * stride + MARGIN_X) * es
        nb = stride * (H + 2 * MARGIN_Y) * es
        ref0 = plane_as_tensor(torch, base, nb, dev)
        side = torch.cuda.Stream(device=dev)
        if not rows_mode:
            # incoming-reference plane: the owner's newest reference lands here on the other ranks (making it a reference is a
            # pointer swap the bench does not do, so that every step analyses the same frames)
            inc = lib.alloc(nb)
            incoming = plane_as_tensor(torch, inc.ptr, nb, dev)

    # All step timing is on the device: CUDA events on the library's own stream (wrapped as a torch ExternalStream) bracket
    # the kernels AND, through event waits, the exchange that runs on the side stream.
    lib_stream = torch.cuda.ExternalStream(lib.L.x265cu_stream(lib.ctx), device=dev)
    pending = []

    def exchange(step):
        """Newest reconstructed reference plane from its owner (producer side of m_reconRowFlag, framefilter.cpp:664).  Issued
        on a SIDE stream with no host synchronisation: it overlaps with this step's kernels (which read the current
        references, not the incoming plane); the library stream waits for it at the END of the step (where the consumer
        would swap the plane in)."""
        if world > 1 and not rows_mode:
            e0 = torch.cuda.Event()
            e0.record(lib_stream)
            side.wait_event(e0)                            # the broadcast starts when the step starts
            with torch.cuda.stream(side):
                shard.exchange_ref(dist, ref0, step, world, recv=incoming)
                e1 = torch.cuda.Event()
                e1.record(side)
            pending.append(e1)

    def exchange_rows():
        # rows mode: every owner publishes the CTU rows it reconstructed (CU-size-32 recon plane) once its kernels are done
        if world > 1 and rows_mode:
            e0 = torch.cuda.Event()
            e0.record(lib_stream)
            side.wait_event(e0)
            with torch.cuda.stream(side):
                shard.exchange_rows(dist, ref0, an.ctu_rows, world, H, an.stride, MARGIN_Y, es=es)
                e1 = torch.cuda.Event()
                e1.record(side)
            pending.append(e1)

    def exchange_join():
        """The step ends when its exchange has landed too: the library stream waits for the side stream (device-side)."""
        while pending:
            lib_stream.wait_event(pending.pop())

    def analyse_e2e():
        if CHROMA:
            an.load_chroma(h_cb, h_cr)                     # the frame's chroma travels with it (H2D inside the timed region)
        for r0, r1 in my_rows:
            an.analyse_rows(h_fenc, h_field, r0, r1)

    def run_resident():
        for r0, r1 in my_rows:
            an.run_rows(r0, r1, 7)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (both paths) ----
    for s in range(args.warmup):
        exchange(s)
        analyse_e2e()
        exchange_rows()
        exchange_join()
    an.load_inputs(h_fenc, h_field)
    lib.sync()
    sampler = ClockSampler(local_rank)
    launches0 = lib.launch_count()

    # ---- resident: kernels only, per-step CUDA events, L2 flushed between steps ----
    barrier()
    sampler.start()
    res_ms, stage, phases = [], np.zeros(4), np.zeros(3)
    for s in range(args.steps):
        lib.check(lib.L.x265cu_memset(lib.ctx, flush.ptr, s & 255, flush.nbytes))
        lib.sync()
        if world > 1:
            # untimed, like the flush: line the ranks up before the step.  The exchange inside the step is a collective, so
            # without this the step of an early rank would absorb the host-side skew (Python, the memset) of the latest one
            dist.barrier()
            torch.cuda.synchronize()
        t0e = torch.cuda.Event(enable_timing=True); t1e = torch.cuda.Event(enable_timing=True)
        t0e.record(lib_stream)
        exchange(s)                                        # side stream: overlaps with the kernels below
        run_resident()
        exchange_rows()
        exchange_join()
        t1e.record(lib_stream)
        t1e.synchronize()
        res_ms.append(t0e.elapsed_time(t1e))               # device time: kernels + (overlapped) exchange
        stage += np.array(an.stage_ms())
        phases += np.array(lib.me_phase_ms())
    barrier()
    launches = lib.launch_count() - launches0
    t_res = float(np.sum(res_ms))

    # ---- e2e: public call with host buffers, H2D + D2H inside ----
    barrier()
    t0 = time.perf_counter()
    for s in range(args.steps):
        exchange(s)
        analyse_e2e()
        exchange_rows()
        exchange_join()
    lib.sync()
    torch.cuda.synchronize()
    t_e2e = (time.perf_counter() - t0) * 1000.0
    barrier()
    clocks = sampler.stop()
    # the host buffers now hold the last timed step's results.  With CTU rows sharded over N > 1 GPUs rank 0 holds only its
    # own rows (the rest of its buffers was never written), so there is no whole-frame result to dump
    if args.dump_outputs and rank == 0 and not (rows_mode and world > 1):
        write_outputs(args.dump_outputs, analysis_outputs(an))
    elif args.dump_outputs and rank == 0 and not args.shard_auto:
        print("bench.py: --dump-outputs skipped: with --shard rows no rank holds the whole frame's results", file=sys.stderr)

    if world > 1:
        t = torch.tensor([t_res, t_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_res, t_e2e = float(t[0]), float(t[1])

    rc = 0
    line = None
    if rank == 0:
        stage /= args.steps
        phases /= args.steps
        units = ctus_per_frame() * (1 if rows_mode else world) * args.steps
        value = units / (t_res / 1000.0)
        e2e = units / (t_e2e / 1000.0)
        peak, peak_src = peaks()
        plane = W * H * es
        # Dominant kernel = the longest of the three motion-estimation phases (each phase = the launches of one kernel family).
        # Algorithmic (compulsory) bytes per phase (SURVEY 8(d), DESIGN.md): the source plane + every reference plane read
        # once (+ the 4:2:0 chroma planes where the phase evaluates the chroma-SATD term) + per job the 40 B record and the
        # 24 B phase state read and written (the sub-pel phase writes the 16 B result instead of the state).
        my_jobs = sum(an.row_range(r0, r1)[1] for r0, r1 in my_rows)
        my_share = sum(r1 - r0 for r0, r1 in my_rows) / float(an.ctu_rows)
        luma_bytes = int(plane * (1 + NREFS) * my_share)
        chroma_bytes = int(plane // 2 * (1 + NREFS) * my_share) if CHROMA else 0
        phase_info = [
            ("prechecks", "k_me_chroma<P,1,*>" if CHROMA else "k_me<P,1,*>", "pre-check launches of the batched motionEstimate (MVP / zero / candidate costs; small-PU and large-PU kernels)",
             luma_bytes + chroma_bytes + my_jobs * (40 + 24)),
            ("integer_search", "k_me_window<P,*> (+ k_me<P,2,-1> for groups that do not fit)", "STAR integer search out of TMA-staged shared-memory search windows, one CTA per CU group / 16x16 cell",
             luma_bytes + my_jobs * (40 + 24 + 24)),
            ("subpel", "k_me_chroma<P,3,*>" if CHROMA else "k_me<P,3,*>", "sub-pel refinement launches (interpolation + SATD%s; small-PU and large-PU kernels)" % (" + chroma-SATD term" if CHROMA else ""),
             luma_bytes + chroma_bytes + my_jobs * (40 + 24 + 16))]
        dom = int(np.argmax(phases))
        me_bytes = phase_info[dom][3]
        me_ms = phases[dom]
        achieved = me_bytes / (me_ms / 1000.0) / 1e9
        traffic = None
        traffic_src = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "me_r2_traffic.json")))
            key = "%s_%dx%d_%dbit_%s" % (CFG_NAME, W, H, DEPTH, phase_info[dom][0])
            if key in tr.get("phases", {}):
                traffic = float(tr["phases"][key]["dram_bytes_per_step"]); traffic_src = "profiles/me_r2_traffic.json (" + tr.get("how", "ncu") + ")"
        except Exception:
            pass
        cfg = workload_config(args.shard)
        sizes = {"resid_bytes": plane * 2 + an.ncoef * 2 + 4 * plane, "intra_bytes": plane + an.ncu * 36 * 4}
        line = {
            "metric": "2160p preset-slow CTU-analysis throughput", "value": value, "unit": "CTUs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_res / args.steps, "higher_is_better": True,
            "scaling": "strong" if rows_mode else "weak", "vs_baseline": None, "dtype": "u8" if DEPTH == 8 else "u16", "data": "synthetic", "config": cfg,
            "pu_jobs_per_frame": an.njobs,
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "CTUs/s", "ms_per_step": t_e2e / args.steps,
                    "h2d_bytes_per_step": int(an.h2d_bytes(field)) + (W * H // 2 * es if CHROMA else 0), "d2h_bytes_per_step": int(sum(an.d2h_bytes_rows(r0, r1) for r0, r1 in my_rows))},
            "gpu_launches": int(launches),
            "roofline": {"kernel": phase_info[dom][1], "what": phase_info[dom][2], "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(me_bytes), "kernel_ms": float(me_ms),
                         "note": "the dominant launches of the step (longest motion-estimation phase); not an HBM-bound kernel family: hundreds of SAD / SATD candidates per job against < 100 B of compulsory traffic, planes L2-resident; the binding resources are the SM's ALU pipe, shared-memory bandwidth and instruction cache (DESIGN.md section 5, profiles/)"},
            "phase_rooflines": {pi[0]: {"kernel": pi[1], "ms": float(phases[i]), "algorithmic_bytes": int(pi[3]), "GBps": pi[3] / (phases[i] / 1000.0) / 1e9,
                                        "frac": pi[3] / (phases[i] / 1000.0) / 1e9 / peak} for i, pi in enumerate(phase_info)},
            "stages_ms": {"me_stage": float(stage[0]), "me_prechecks": float(phases[0]), "me_integer_search": float(phases[1]), "me_subpel": float(phases[2]), "residual": float(stage[1]), "intra": float(stage[2])},
            "stage_rooflines": {
                "k_cu_residual": {"achieved": sizes["resid_bytes"] / (stage[1] / 1000.0) / 1e9, "unit": "GB/s", "frac": sizes["resid_bytes"] / (stage[1] / 1000.0) / 1e9 / peak},
                "k_intra_search": {"achieved": sizes["intra_bytes"] / (stage[2] / 1000.0) / 1e9, "unit": "GB/s", "frac": sizes["intra_bytes"] / (stage[2] / 1000.0) / 1e9 / peak}},
        }
        # ---- results of the last e2e step (host arrays) -> checks ----
        mvp = an.me_packed[:, 1].view(np.uint32)
        mvx = (mvp & 0xffff).astype(np.int64); mvy = (mvp >> 16).astype(np.int64)
        full_scope = (not rows_mode) or world == 1
        if full_scope:
            line["checks"] = checks_of(an.me_packed[:, 0], mvx, mvy, an.cu_numsig, an.cu_sse, an.intra_cost, an.njobs, an.ncu)
            line["checks_scope"] = "whole frame"
        # ---- CPU baseline on this box's host cores (rank 0, N=1 only; bounded sample) + parity assertion on its scope ----
        if world == 1 and not args.no_cpu:
            threads = host_cores()
            probe = cpu_reference(1, threads)
            total_rows = (H + 63) // 64
            rows = int(max(1, min(total_rows, args.cpu_seconds / max(probe["seconds"], 1e-3))))
            r = cpu_reference(rows, threads, wl=probe["wl"]) if rows > 1 else probe
            line["cpu_baseline"] = {"value": r["ctus_per_s"], "unit": "CTUs/s", "cores": threads, "kind": r["kind"], "sample": r["sample"], "asm": asm_status()}
            cj, cc = r["checks"]["jobs"], r["checks"]["cus"]
            mine = checks_of(an.me_packed[:, 0], mvx, mvy, an.cu_numsig, an.cu_sse, an.intra_cost, cj, cc)
            line["checks_vs_cpu"] = {"scope": r["scope"], "gpu": mine, "cpu": r["checks"], "equal": mine == r["checks"]}
            line["checks_equal"] = bool(mine == r["checks"])
            if not line["checks_equal"]:
                rc = 3
        if world == 1 and CHROMA and not args.no_pred:
            try:
                from frame_helpers import Workload
                wl = r["wl"] if (not args.no_cpu) else Workload(W, H, depth=DEPTH, numRefs=NREFS, method=c["method"], subme=c["subme"], merange=c["merange"],
                                                               rect=c["rect"], qp=c["qp"], chroma=True, amp=c["amp"])
                an.analyse(h_fenc, h_field)                   # whole-frame results resident for the job list
                line["pred_cost"] = pred_cost_leg(lib, an, wl, 0.0 if args.no_cpu else min(8.0, args.cpu_seconds))
                if line["pred_cost"].get("checks_equal") is False:
                    rc = rc or 4
                    print("bench.py: PARITY FAILURE: prediction costs differ from the reference on the CPU sample", file=sys.stderr)
            except Exception as e:
                line["pred_cost_error"] = repr(e)
        if world == 1 and not args.no_primitives:
            try:
                line["primitives"] = primitives_leg(lib)
            except Exception as e:          # the per-primitive table must never cost the headline line
                line["primitives_error"] = repr(e)
        if rc:
            print("bench.py: PARITY FAILURE: GPU checks differ from the CPU reference on %s" % line["checks_vs_cpu"]["scope"], file=sys.stderr)
    an.close()
    flush.free()
    return (line if rank == 0 else None), rc


# ----------------------------------------------------------------------------------------------
# c2: the lookahead (BASELINE configs[1]); N>1 shards the frames (BASELINE configs[3]'s lookahead partition)
def lookahead_frames():
    from frame_helpers import gen_luma
    c = CFG
    return [gen_luma(c["W"], c["H"], i, bits=c["depth"]) for i in range(c["frames"])]


def run_lookahead_ours(args, rank, world, local_rank):
    import torch
    import x265_b200
    from x265_b200.lookahead import Lookahead, window_triples, conflict_free_batches, owner
    c = CFG
    dist = None
    if world > 1:
        import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = x265_b200.load(local_rank)
    frames = lookahead_frames()
    n = len(frames)
    # pinned host copies: what the caller (the encoder's input queue) hands over; H2D is then real asynchronous DMA
    pinned = []
    for f in frames:
        p = lib.L.x265cu_host_alloc(f.nbytes)
        a = np.frombuffer((C.c_uint8 * f.nbytes).from_address(p), f.dtype).reshape(f.shape)
        a[:] = f
        pinned.append(a)
    frames = pinned
    la = Lookahead(lib, c["W"], c["H"], c["depth"], n, lookahead_slices=c.get("lslices", 0))
    triples = window_triples(n, c["bframes"])
    mine = [t for t in triples if owner(t[2], world) == rank]
    batches = conflict_free_batches(mine)
    flush = lib.alloc(256 << 20)
    blocks = [plane_as_tensor(torch, *la.plane_block(i), dev) for i in range(n)] if world > 1 else None

    def publish():
        # every frame's 4 lowres planes: produced on the owner, ONE broadcast per frame (the only data-path exchange)
        if world > 1:
            lib.sync()
            works = [dist.broadcast(blocks[i], src=owner(i, world), async_op=True) for i in range(n)]
            for w in works:
                w.wait()
            torch.cuda.current_stream().synchronize()
            for i in range(n):
                la.planes_received(i)

    def step(e2e):
        la.forget_results()
        for f in la.fr:
            f["has_intra"] = False
        own = [i for i in range(n) if owner(i, world) == rank]
        for i in own:
            la.init_frame(i, frames[i], sync=False)   # H2D of the full-res luma + border extension + Lowres::init, stream-ordered
        publish()
        la.intra_batch(own)
        preps = [la.prepare_batch(b) for b in batches]
        for p in preps:
            la.launch_batch(p)
        lib.sync()
        for p in preps:
            la.collect_batch(p, full=e2e)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(True)
    sampler = ClockSampler(local_rank)
    launches0 = lib.launch_count()
    barrier()
    sampler.start()
    # resident: planes + intra in place; time the estimate launches only (CUDA events)
    t_res = 0.0
    for s in range(args.steps):
        la.forget_results()
        preps = [la.prepare_batch(b) for b in batches]
        lib.check(lib.L.x265cu_memset(lib.ctx, flush.ptr, s & 255, flush.nbytes))
        lib.sync()
        lib.timer_begin()
        for p in preps:
            la.launch_batch(p)
        t_res += lib.timer_end()
        for p in preps:
            la.collect_batch(p, full=False)
    barrier()
    launches = lib.launch_count() - launches0
    t0 = time.perf_counter()
    for s in range(args.steps):
        step(True)
    torch.cuda.synchronize()
    t_e2e = (time.perf_counter() - t0) * 1000.0
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # what collect_batch(full=True) returned for this rank's frame-cost estimates in the last timed step
        res = [la.fr[b]["res"][(b - p0, p1 - b)] for (p0, p1, b) in mine]
        write_outputs(args.dump_outputs, {"triples": np.array(mine).reshape(-1, 3), "frame_cost": [r["score"] for r in res],
                                          "cost_est_aq": [r["costEstAq"] for r in res], "intra_mbs": [r["intraMbs"] for r in res],
                                          "lowres_costs": np.array([r["lowresCosts"] for r in res]),
                                          "row_satds": np.array([r["rowSatds"] for r in res])})
    costs = {t: la.fr[t[2]]["res"][(t[2] - t[0], t[1] - t[2])]["score"] for t in mine}
    csum = sum(v * (1 + (t[0] * 31 + t[1] * 17 + t[2]) % 13) for t, v in costs.items())
    if world > 1:
        t = torch.tensor([t_res, t_e2e, float(csum)], dtype=torch.float64, device=dev)
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        t_res, t_e2e, csum = float(tm[0]), float(tm[1]), int(ts[2])
    rc = 0
    if rank == 0:
        units = len(triples) * la.ncu * args.steps
        peak, peak_src = peaks()
        plane_b = la.plane_bytes
        algo = sum((5 if t[1] == t[2] else 9) * plane_b + la.ncu * 32 for t in mine)      # fenc + 4 (P) / 8 (B) hpel planes read once + 32 B per CU
        achieved = algo / (t_res / args.steps / 1000.0) / 1e9
        line = {"metric": "1080p lookahead estimateFrameCost throughput", "value": units / (t_res / 1000.0), "unit": "lowres CUs/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_res / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u8" if c["depth"] == 8 else "u16", "data": "synthetic", "config": workload_config(), "clocks": clocks,
                "e2e": {"value": units / (t_e2e / 1000.0), "unit": "lowres CUs/s", "ms_per_step": t_e2e / args.steps,
                        "h2d_bytes_per_step": int(sum(frames[i].nbytes for i in range(n) if owner(i, world) == 0)),
                        "d2h_bytes_per_step": int(len(mine) * (24 + 2 * la.ncu + 4 * la.h8))},
                "gpu_launches": int(launches), "frame_costs": len(triples), "launches_per_step": len(batches),
                "roofline": {"kernel": "k_lookahead_cost (cluster wavefront, one cluster per (p0,p1,b))", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(algo / max(1, len(batches))),
                             "note": "latency bound: one dependent chain of ~250 CU searches per triple (anti-diagonal wavefront)"},
                "checks": {"frame_cost_hash": int(csum), "triples": len(triples)}}
        if world == 1 and not args.no_cpu:
            r = lookahead_cpu(frames, triples, budget_s=args.cpu_seconds)
            line["cpu_baseline"] = {"value": r["cus_per_s"], "unit": "lowres CUs/s", "cores": r["procs"], "kind": r["kind"], "sample": r["sample"], "asm": asm_status()}
            mine_h = sum(costs[t] * (1 + (t[0] * 31 + t[1] * 17 + t[2]) % 13) for t in r["triples"])
            line["checks_vs_cpu"] = {"scope": r["sample"], "gpu": int(mine_h), "cpu": int(r["hash"]), "equal": int(mine_h) == int(r["hash"])}
            line["checks_equal"] = line["checks_vs_cpu"]["equal"]
            if not line["checks_equal"]:
                rc = 3
        print(json.dumps(line), flush=True)
    la.close()
    return rc


def _la_worker(args):
    """One host process of the CPU lookahead arm: its own reference Lookahead over the window, a subset of the triples."""
    depth, W, H, nframes, bframes, triples, kind = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from common import load_ref, load_oracle
    from frame_helpers import gen_luma
    frames = [gen_luma(W, H, i, bits=depth) for i in range(nframes)]
    if kind == "reference":
        from test_lookahead_oracle_vs_ref import RefLookahead
        h = RefLookahead(load_ref(depth), frames, bframes)
    else:
        from lookahead_helpers import OracleLookahead
        h = OracleLookahead(load_oracle(depth), frames, depth)
    t0 = time.perf_counter()
    out = [(t, h.cost(*t)) for t in triples]
    return out, time.perf_counter() - t0


def lookahead_cpu(frames, triples, budget_s=20.0, steps=1):
    """estimateFrameCost of (a bounded subset of) the window's triples with the REAL reference classes, one process per host
    core (the reference's serial per-TLD path in each), triples dealt by frame b."""
    from concurrent.futures import ProcessPoolExecutor
    from common import load_ref
    c = CFG
    kind = "reference" if load_ref(c["depth"]) is not None else "port"
    procs = max(1, min(host_cores(), c["frames"] - 1))
    ncu = ((c["W"] // 2 + 7) // 8) * ((c["H"] // 2 + 7) // 8)
    # ~0.7 M CUs/s per thread (profiles/lookahead_r1.txt): bound the sample
    per_triple = ncu / 0.5e6
    maxn = int(max(procs, min(len(triples), budget_s * procs / per_triple)))
    sub = triples[:maxn]
    parts = [[t for t in sub if t[2] % procs == k] for k in range(procs)]
    parts = [p for p in parts if p]
    t0 = time.perf_counter()
    with ProcessPoolExecutor(max_workers=len(parts)) as ex:
        res = list(ex.map(_la_worker, [(c["depth"], c["W"], c["H"], c["frames"], c["bframes"], p, kind) for p in parts]))
    wall = time.perf_counter() - t0
    busy = max(r[1] for r in res)                     # the estimate loops run concurrently: the slowest worker is the step
    costs = dict(kv for r in res for kv in r[0])
    h = sum(v * (1 + (t[0] * 31 + t[1] * 17 + t[2]) % 13) for t, v in costs.items())
    return {"cus_per_s": len(sub) * ncu / busy, "procs": len(parts), "kind": kind, "hash": h, "triples": sub, "seconds": busy, "wall": wall,
            "sample": "%d of the %d frame-cost estimates of the window, %d processes (frame setup untimed)" % (len(sub), len(triples), len(parts))}


def run_lookahead_reference(args):
    from x265_b200.lookahead import window_triples
    c = CFG
    triples = window_triples(c["frames"], c["bframes"])
    budget = 170.0 / max(1, args.steps)
    t0 = time.perf_counter()
    r = None
    for _ in range(args.steps):
        r = lookahead_cpu(None, triples, budget_s=budget * 0.5)
    dt = time.perf_counter() - t0
    line = {"impl": "reference", "metric": "1080p lookahead estimateFrameCost throughput", "value": r["cus_per_s"], "unit": "lowres CUs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * r["seconds"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(),
            "cpu_baseline": {"value": r["cus_per_s"], "unit": "lowres CUs/s", "cores": r["procs"], "kind": r["kind"], "sample": r["sample"], "asm": asm_status()},
            "e2e": {"value": r["cus_per_s"], "unit": "lowres CUs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "checks": {"frame_cost_hash_of_sample": int(r["hash"]), "triples": len(r["triples"])}, "gpu_launches": 0, "wall_s": dt}
    print(json.dumps(line), flush=True)


def main():
    # keep stdout clean for the ONE JSON line: library chatter (e.g. "NCCL version ...") goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS), help="BASELINE.json config (c2 lookahead, c3 slow [default], c4 slower Main10, c5 8K veryslow)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (and with it the parity assertion)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="host time budget of the cpu_baseline sample")
    ap.add_argument("--shard", default="auto", choices=["auto", "frames", "rows"],
                    help="N>1 partition: a frame per GPU (weak scaling) or the CTU rows of one frame per GPU (strong scaling); "
                         "auto (default) = the frame shard as the line, with the row shard measured in the same run and attached")
    ap.add_argument("--no-chroma", action="store_true", help="luma-only motion estimation (round-1 line; the presets run with the chroma-SATD term)")
    ap.add_argument("--no-pred", action="store_true", help="skip the prediction-cost leg (AMVP / merge / bidir costs) of the N=1 line")
    ap.add_argument("--no-primitives", action="store_true", help="skip the per-primitive HBM GB/s table (8- and 10-bit) of the N=1 line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the project's own path (--impl ours)")
    global CFG, CFG_NAME
    CFG_NAME = args.config
    CFG = dict(CONFIGS[args.config])
    if args.no_chroma and "chroma" in CFG:
        CFG["chroma"] = False
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    args.shard_auto = args.shard == "auto"
    if args.shard == "auto":
        args.shard = "frames"
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return 0
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world)
    if CFG.get("lookahead"):
        rc = run_lookahead_ours(args, rank, world, local_rank)
    else:
        # N > 1 without an explicit --shard: the headline line is the frame shard (weak scaling: CTUs/s of N frames in flight);
        # the same run then measures the CTU-ROW shard of ONE frame (strong scaling, BASELINE configs[4]) and attaches it
        shard_mode = args.shard if args.shard != "auto" else "frames"
        args.shard = shard_mode
        line, rc = run_ours(args, rank, world, local_rank)
        if world > 1 and args.shard_auto:
            args.shard = "rows"
            rows_line, rc2 = run_ours(args, rank, world, local_rank)
            rc = rc or rc2
            if rank == 0:
                line["strong_scaling_rows"] = {k: rows_line[k] for k in ("value", "unit", "ms_per_step", "scaling", "e2e", "stages_ms", "gpu_launches")}
                line["strong_scaling_rows"]["config"] = rows_line["config"]
        if rank == 0:
            print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main() or 0)
