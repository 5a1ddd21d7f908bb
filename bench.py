"""bench.py -- stage-II re-ranked triplets/s (BASELINE.json metric) on N B200s of one node.

A "step" is one pass of the hot path over one batch of synthetic input: for every query of a Fashion-IQ-val-shaped
category (Q = 2,017 queries x top-K = 100 candidates, BASELINE configs[3]; `--job cirr`: Q = 4,181 x K = 50, configs[2])
compute z_t (stage-I encoder on the reference image's tokens), score all Q*K triplets with the dual-stream stage-II
encoder (candidate-major, K/V once per unique candidate), re-sort each row and count Recall@{10,50}.  Gallery ViT tokens
are the resident cache the reference also keeps on the device (src/utils.py:43-55); they are produced once, outside the
timed region, by the ViT kernel path.

  value : whole-job triplets/s with the step's inputs already resident in HBM
  e2e   : the same metric through the public validate_stage2.compute_fiq_val_metrics call with HOST (pinned) token ids /
          masks / candidate names / labels: name -> row join, H2D of ids, masks, reference rows, per-chunk triplet lists
          and labels inside the timed region; the recall counters AND the re-ranked order [Q,K] are read back D2H
  roofline : the dominant kernel (tcgen05 GEMM): algorithmic FLOPs / CUDA-event duration per launch against the measured
          sustained bf16 peak in MEASURED_PEAKS.json; `secondary` holds the same for the tcgen05 attention, the masked
          self-attention and LayerNorm (HBM) kernels; `traffic` = DRAM bytes per launch from the committed ncu capture
  cpu_baseline : the reference's CPU arithmetic on the host cores on a bounded sample of the same workload (the reference
          itself through tests/golden/ref_shim.py where its sources are reachable, else the oracle port)

N > 1 (torchrun): STRONG scaling -- the job is fixed and split over the ranks.  z_t is computed for a block of queries per
rank and all-gathered; the candidate-sorted triplet list is cut into N contiguous candidate ranges, so each gallery image's
K/V projections are computed on one rank only and the per-GPU K/V reuse does not fall with N (`--partition query` splits
by query block instead); ranks all-gather (position, score) pairs and every rank re-sorts.  After the timed region rank 0
re-scores a sample of rows alone (single-GPU path) and the line carries the comparison (`cross_rank_check`).
`--impl reference` times the reference's CPU implementation of the path instead (rank 0 only).

`--dump-outputs DIR` writes what the last timed step returned, so that two builds can be compared output for output on
the same seeded inputs: scores.npy [Q,K] float32, order.npy [Q,K] (re-ranked positions, as float32),
recall_hits_at_10_50.npy [2] float64 and rows.npy (the query rows written, float64).  Above 64 MB in all, a fixed
seeded sample of the query rows is written.
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
sys.path.insert(0, ROOT)

import numpy as np
import torch

F_REF_GF = 47.247          # SURVEY.md 8(d): algorithmic GFLOP per triplet as the reference executes them (L=32)
METRIC = "stage2_reranked_triplets_per_s"
UNIT = "triplets/s"
JOBS = {"fiq": (2017, 100), "cirr": (4181, 50)}      # analysis_plot/fiq_stageII_labels_val_dress.pt / cirr_stageII_labels_val.pt row counts


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--job", default="fiq", choices=sorted(JOBS))
    ap.add_argument("--queries", type=int, default=None)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--gallery", type=int, default=2297)      # CIRR-val-sized token gallery (BASELINE configs[1])
    ap.add_argument("--length", type=int, default=32)
    ap.add_argument("--partition", default="candidate", choices=["candidate", "query"])
    ap.add_argument("--cpu-sample-queries", type=int, default=4)      # ~13 s of CPU work on the box's 16 cores
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    q, k = JOBS[a.job]
    a.queries = a.queries or q
    a.k = a.k or k
    return a


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return (d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs", 6500.0),
                "measured (MEASURED_PEAKS.json: bf16_tflops_sustained for kernels timed inside a long step, hbm_gbs)")
    return 1400.0, 6500.0, "fallback (B200_PROFILING.md: sustained ~1.4 PFLOP/s bf16, ~6.5 TB/s HBM copy)"


def committed_traffic():
    """DRAM bytes per launch of this repo's kernels from the committed ncu capture (profiles/r02_dram_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons}


def synth_workload(args, seed=0):
    """The job (identical on every rank): queries, stage-I-like candidate lists (K distinct gallery rows per query, never the
    reference; the target planted in ~98 % of the lists), labels."""
    import cir_b200 as cir
    syn = cir.synthetic
    Q, K, G, L = args.queries, args.k, args.gallery, args.length
    ref, tgt, ids, mask = syn.make_queries(Q, G, L, seed=300 + seed)
    g = torch.Generator().manual_seed(400 + seed)
    scores = torch.rand(Q, G, generator=g)
    scores[torch.arange(Q), ref] = -1.0
    hit = torch.rand(Q, generator=g) < 0.98
    scores[torch.arange(Q)[hit], tgt[hit]] = 2.0
    scores[torch.arange(Q)[~hit], tgt[~hit]] = -1.0
    cand = scores.topk(K, dim=1).indices
    cand = cand[:, torch.randperm(K, generator=g)].to(torch.int32)
    labels = cand.long() == tgt[:, None]
    return ref.int(), tgt, ids.int(), mask.int(), cand, labels


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, scores, order, hits, limit=DUMP_LIMIT_BYTES):
    """Write one step's outputs as .npy files (float32 / float64).  When all rows would exceed ``limit`` bytes, a fixed
    seeded sample of query rows is written instead; rows.npy names them."""
    scores = np.asarray(scores, dtype=np.float32)
    order = np.asarray(order, dtype=np.float32)          # positions < K <= 2**24: exact in float32
    Q, K = scores.shape
    per_row = K * 4 * 2 + 8
    fixed = 16 + 4 * 128                                  # recall counters + .npy headers
    rows = np.arange(Q)
    if fixed + Q * per_row > limit:
        n = max(0, (limit - fixed) // per_row)
        rows = np.sort(np.random.default_rng(0).choice(Q, size=n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scores.npy"), scores[rows])
    np.save(os.path.join(out_dir, "order.npy"), order[rows])
    np.save(os.path.join(out_dir, "recall_hits_at_10_50.npy"), np.asarray(hits, dtype=np.float64))
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


def workload_text(args):
    return (f"stage2_rerank_{args.job}_shape: Q={args.queries} queries x K={args.k} candidates (whole job), L={args.length} tokens, "
            f"G={args.gallery} gallery images (577 ViT-B/16 tokens each, resident), z_t + stage-II + re-sort + recall")


# ----------------------------------------------------------------------------------------------- CPU arms
def find_reference():
    """The reference's own sources, if reachable: $CIR_REFERENCE or ./baseline/_ref."""
    for p in (os.environ.get("CIR_REFERENCE"), os.path.join(ROOT, "baseline", "_ref")):
        if p and os.path.exists(os.path.join(p, "src", "blip_stage2.py")):
            return p
    return None


def cpu_scorer(args):
    """-> (score_one_query(qi), kind, note).  The UNMODIFIED reference modules behind tests/golden/ref_shim.py when the
    reference's sources are reachable, otherwise the CPU oracle (a restatement of the same arithmetic)."""
    import cir_b200 as cir
    syn = cir.synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd1 = syn.make_stage1_state_dict(0, 384, "reference")
    sd2 = syn.make_stage2_state_dict(0, 384, "reference")
    L, K = args.length, args.k
    g = torch.Generator().manual_seed(0)
    tokens = torch.randn(K + 1, 577, 768, generator=g)          # LayerNorm-like statistics (mean 0, std 1)
    ids, mask = syn.make_token_ids(8, L, seed=2)
    ids[:, 0] = syn.ENC_TOKEN_ID
    ref_path = find_reference()
    if ref_path is not None:
        try:
            os.environ["CIR_REFERENCE"] = ref_path
            sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            from ref_shim import build_models
            m1, m2, tok, _ = build_models(sd1, sd2)

            def one(qi):
                q = qi % 8
                with torch.no_grad():
                    tok.push(ids[q:q + 1], mask[q:q + 1])
                    z = m1.img_txt_fusion(tokens[:1], None, ["x"], train=False, return_raw=True)        # validate_stage2.py:105-106
                    tok.push(ids[q:q + 1], mask[q:q + 1])
                    s = m2.img_txt_fusion_val(z, tokens[1:], ["x"])                                     # :118
                    torch.argsort(s[None], dim=-1, descending=True)                                     # :53
            return one, "reference", f"unmodified reference modules from {ref_path} (import shims: tests/golden/ref_shim.py)", cores
        except Exception as ex:                                  # fall through to the port
            print(f"bench: reference at {ref_path} not usable ({type(ex).__name__}: {ex}); using the oracle port", file=sys.stderr)
    from oracle import cir_oracle as O

    def one(qi):
        q = qi % 8
        with torch.no_grad():
            z = O.stage1_hidden(sd1, tokens[:1], ids[q:q + 1], mask[q:q + 1])
            s = O.stage2_score(sd2, z, ids[q:q + 1], mask[q:q + 1], tokens[1:])
            O.rerank_order(s[None])
    return one, "port", "oracle/cir_oracle.py (the reference's sources are not reachable on this box)", cores


def run_reference(args, rank, emit):
    """Reference arm: the reference's CPU implementation of the path on all host threads; each step = one query x K candidates
    of the workload (z_t + img_txt_fusion_val + argsort, as src/validate_stage2.py:94-125)."""
    if rank != 0:
        return
    one, kind, note, cores = cpu_scorer(args)
    K = args.k
    for i in range(args.warmup):
        one(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        one(args.warmup + i)
    dt = (time.perf_counter() - t0) / args.steps
    v = K / dt
    sample = f"1 query x K={K} candidates per step (z_t + stage-II + sort), fp32, torch CPU {cores} threads; {note}"
    emit({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
          "dtype": "f32", "data": "synthetic",
          "config": {"workload": workload_text(args), "sample": f"each step = 1 query x {K} candidates of that workload on the host CPU"},
          "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
          "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
          "gpu_launches": 0})


def cpu_baseline(args):
    one, kind, note, cores = cpu_scorer(args)
    nq = max(1, args.cpu_sample_queries)
    one(7)                                                       # warm-up
    t0 = time.perf_counter()
    for q in range(nq):
        one(q)
    dt = time.perf_counter() - t0
    return {"value": nq * args.k / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{nq} queries x K={args.k} candidates (z_t + stage-II + sort per query, as src/validate_stage2.py:94-125), fp32, "
                      f"torch CPU {cores} threads; {note}"}


# ----------------------------------------------------------------------------------------------- GPU arm
def main():
    # stdout carries exactly ONE JSON line: everything else a library prints there (e.g. "NCCL version ..." on the
    # first collective) is routed to stderr by pointing fd 1 at fd 2 until the line is ready
    sys.stdout.flush()
    _stdout_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(_stdout_fd, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, emit)
        return
    import cir_b200 as cir
    import torch.distributed as dist
    N = cir.native
    D = cir.distributed
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    syn = cir.synthetic
    Q, K, G, L = args.queries, args.k, args.gallery, args.length

    # ---- models (random-init, reference init style) and the resident gallery token cache (replicated: 2 GB of 180)
    sd1 = syn.make_stage1_state_dict(0, 384, "reference")
    sd2 = syn.make_stage2_state_dict(0, 384, "reference")
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16", device=dev)
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16", device=dev)
    eng = m2.engine
    del sd1, sd2
    tokens = torch.empty(G, 577, 768, dtype=torch.bfloat16, device=dev)
    gi = torch.Generator().manual_seed(1)
    for g0 in range(0, G, 64):                                   # ViT-B/16 on synthetic 384x384 images (not timed)
        n = min(64, G - g0)
        tokens[g0:g0 + n] = m2.img_embed(torch.randn(n, 3, 384, 384, generator=gi))
    torch.cuda.synchronize()

    ref, tgt, ids, mask, cand, labels = synth_workload(args)
    names = syn.index_names_for(G)
    ref_d, ids_d, mask_d = ref.to(dev), ids.to(dev), mask.to(dev)
    cand_np = cand.numpy()
    labels_d = labels.to(dev)
    row_active = labels.any(1).numpy()
    n_trip = int(row_active.sum()) * K                            # rows without a positive are filled, not scored (:95,:123)

    def step_resident():
        if args.partition == "candidate":
            z_all = D.encode_queries_sharded(m1, tokens, ref_d, ids_d, mask_d)
            scores = D.score_matrix_sharded(m2, tokens, z_all, ids_d, mask_d, cand_np, row_active)
        else:
            scores = D.stage2_scores_gpu(m1, m2, tokens, ref_d, ids_d, mask_d, cand_np, row_active, mode="query")
        order = eng.rerank_sort(scores)
        hits = eng.recall_counts(labels_d, order, (10, 50), sync=False)     # stays on the device: the host plans the next step meanwhile
        return scores, order, hits

    # host-resident inputs for the e2e leg (pinned)
    tb = syn.TokenBatch(input_ids=ids.long().pin_memory(), attention_mask=mask.long().pin_memory())
    ds = syn.SyntheticRelativeDataset(names, ref, tgt, ["x"] * Q, cand_np, kind="fiq", token_batch=tb)
    V2 = cir.validate_stage2

    def step_e2e():
        # the reference's own entry point for this path (src/validate_stage2.py:33-66) on a dataset object whose token ids /
        # masks / candidate names / labels live in HOST memory: every step joins names to gallery rows, uploads ids, masks,
        # reference rows, the per-chunk triplet lists and the labels (H2D), scores, re-sorts, and reads the recall counters
        # and the re-ranked order back (D2H).  Under torchrun the same call shards itself over the ranks.
        r10, r50, order = V2.compute_fiq_val_metrics(ds, m2, m1, tokens, names, return_order=True)
        return r10, r50, order

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, out

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local)
    sampler.start()
    eng.launch_count(reset=True)
    eng.profile_gemm(True)
    ms_step, (scores_last, order_last, hits_last) = timed(step_resident, args.steps)
    eng.profile_gemm(False)
    launches = eng.launch_count()
    prof = {k: eng.profile_read(k) for k in (N.PROF_GEMM, N.PROF_ATTN_TC, N.PROF_ATTN_SELF, N.PROF_LAYERNORM, N.PROF_QKV_ATTN)}
    gemm_ms, gemm_flops, gemm_n = prof[N.PROF_GEMM]
    plan = dict(eng.last_plan)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, scores_last.cpu().numpy(), order_last.cpu().numpy(), hits_last.cpu().numpy())
    step_e2e()
    eng.h2d_bytes = 0
    ms_e2e, (r10, r50, order_host) = timed(step_e2e, args.steps)
    # bytes per step counted from the tensors the call copies: engine uploads (per-chunk lists, counted by the engine) +
    # int64 ids/mask (tokenize) + bool labels; D2H: the order [Q,K] int32 and two int64 counters
    h2d = eng.h2d_bytes // args.steps + 2 * Q * L * 8 + 2 * Q * L * 4 + Q * 4 + Q * K
    d2h = Q * K * 4 + 2 * 8
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- N-GPU == 1-GPU: rank 0 re-scores a sample of rows alone, through the single-process path (no partition, no
    #      collectives), and compares with the rows the sharded step produced
    check = None
    if world > 1:
        if rank == 0:
            rows = np.flatnonzero(row_active)[:: max(1, int(row_active.sum()) // 48)][:48]
            r_t = torch.from_numpy(rows).to(dev)
            z1, _ = m1.encode_queries(tokens, ref_d[r_t], ids_d[r_t], mask_d[r_t], want_z=True, want_emb=False)
            pos, sc = eng.stage2_score_pairs(m2._w, tokens, z1, ids_d[r_t], mask_d[r_t], cand_np[rows], None, part=None)
            alone = torch.empty(len(rows) * K, dtype=torch.float32, device=dev)
            alone.index_copy_(0, pos, sc)
            alone = alone.view(len(rows), K)
            diff = (alone - scores_last[r_t]).abs().max().item()
            same_order = bool(torch.equal(eng.rerank_sort(alone), order_last[r_t]))
            check = {"rows": int(len(rows)), "triplets": int(len(rows) * K), "bit_equal": bool(torch.equal(alone, scores_last[r_t])),
                     "max_abs_diff": diff, "order_equal": same_order}
            assert diff <= 1e-6, f"N-GPU scores differ from the single-GPU path by {diff}"
        barrier()

    # ---- secondary figures of the same path (outside the timed region, rank 0)
    def _time(fn, it=3):
        fn(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(it):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / it
    # ---- weak-scaling figure for comparison with round 1 (every rank re-ranks the WHOLE job by itself, no collectives)
    extras = {}
    if world > 1 and not args.no_extras:
        def step_alone():
            z, _ = m1.encode_queries(tokens, ref_d, ids_d, mask_d, want_z=True, want_emb=False)
            s = m2.score_triplets(z, ids_d, mask_d, tokens, cand_np, row_active)
            return eng.rerank_sort(s)
        step_alone()
        ms_weak, _ = timed(step_alone, 2)
        extras["weak_scaling"] = {"value": world * n_trip / (ms_weak / 1e3), "unit": UNIT, "ms_per_step": ms_weak,
                                  "note": "every rank re-ranks the whole job independently (round-1 definition), 2 steps"}

    # ---- stage I over a 1 M-image gallery (BASELINE configs[4]): the gallery rows are block-partitioned over the ranks, every rank
    #      finds its local top-200 (tensor-core candidate filter + exact fp32 re-check), one all-gather of the [Q, 200] (distance,
    #      index) lists, cir_topk_merge.  All ranks take part; timed like the main step (max over ranks).
    if not args.no_extras:
        try:
            G1, K1, Q1 = 1_000_000, 200, 4181
            gq = torch.Generator().manual_seed(5)
            qe = torch.nn.functional.normalize(torch.randn(Q1, 256, generator=gq), dim=-1).to(dev)
            rows1 = cir.schedule.shard_rows(G1, rank, world)
            gl = torch.Generator(device=dev).manual_seed(50 + rank)
            big = torch.nn.functional.normalize(torch.randn(rows1.stop - rows1.start, 256, generator=gl, device=dev), dim=-1)

            def stage1_step():
                return D.sharded_stage1_topk(lambda sl: eng.stage1_topk(qe, big, K1, exclude=None, col_offset=sl.start), eng.topk_merge, G1)
            stage1_step()
            ms1m, (d1m, i1m) = timed(stage1_step, 3)
            fl = 2.0 * 256 * Q1 * G1
            extras["stage1_topk_1M"] = {
                "queries_per_s": Q1 / (ms1m / 1e3), "Q": Q1, "G": G1, "K": K1, "ms": ms1m, "n_gpus": world,
                "gallery_rows_per_rank": rows1.stop - rows1.start,
                "roofline": {"bound": "tensor", "achieved": fl / (ms1m / 1e3) / 1e12, "peak": measured_peaks()[0] * world, "unit": "TFLOP/s",
                             "frac": fl / (ms1m / 1e3) / 1e12 / (measured_peaks()[0] * world),
                             "note": "algorithmic 2*256*Q*G flop over the whole call (bf16 conversion of the gallery, tcgen05 filter tiles, "
                                     "per-block select, exact fp32 re-check, merge); HBM floor = one read of the fp32 gallery (1.02 GB)"},
                "sorted": bool((d1m[:, 1:] >= d1m[:, :-1]).all().item())}
            if world == 1 and rank == 0:                         # the fp32 CUDA-core path it replaces, and the CPU (oracle) on a bounded sample
                eng.set_stage1_tensor_cores(False)
                ms_old = _time(lambda: eng.stage1_topk(qe, big, K1), it=1)
                eng.set_stage1_tensor_cores(True)
                d_old, i_old = eng.stage1_topk(qe[:512], big, K1)
                eng.set_stage1_tensor_cores(False)
                d_ref, i_ref = eng.stage1_topk(qe[:512], big, K1)
                eng.set_stage1_tensor_cores(True)
                extras["stage1_topk_1M"]["fp32_path_queries_per_s"] = Q1 / (ms_old / 1e3)
                extras["stage1_topk_1M"]["bit_equal_to_fp32_path_512_queries"] = bool(torch.equal(i_old, i_ref) and torch.equal(d_old, d_ref))
                if not args.no_cpu_baseline:
                    from oracle import cir_oracle as O
                    torch.set_num_threads(os.cpu_count() or 1)
                    qc, gc_ = qe[:64].cpu(), big[:200_000].cpu()
                    t0 = time.perf_counter()
                    O.stage1_topk(qc, gc_, None, K1)
                    dtc = time.perf_counter() - t0
                    extras["stage1_topk_1M"]["cpu_baseline"] = {
                        "value": 64 / dtc / 5.0, "unit": "queries/s", "cores": os.cpu_count() or 1, "kind": "port",
                        "sample": "64 queries x 200,000 gallery rows (1 - q @ G^T, full stable argsort, [:200], src/validate.py:57-58), "
                                  "scaled x 1/5 to the 1 M gallery (the work is linear in G up to the log factor of the sort)"}
            del big
        except Exception as ex_:                                 # never let a secondary leg break the bench line
            extras["stage1_topk_1M"] = {"error": repr(ex_)[:300]}
    if rank == 0 and not args.no_extras:
        gq = torch.Generator().manual_seed(5)
        qe = torch.nn.functional.normalize(torch.randn(4181, 256, generator=gq), dim=-1).to(dev)
        ge = m1.engine.stage1_gallery_embed(m1._w, tokens)
        ex = torch.randint(0, G, (4181,), generator=gq)
        ms1 = _time(lambda: eng.stage1_topk(qe, ge, 100, exclude=ex))
        extras["stage1_topk"] = {"queries_per_s": 4181 / (ms1 / 1e3), "Q": 4181, "G": G, "K": 100, "ms": ms1,
                                 "note": "BASELINE configs[1]: fused 1 - q @ G^T + per-query top-100 with the reference index excluded"}
        img = torch.randn(64, 3, 384, 384, device=dev)
        msv = _time(lambda: eng.vit_forward(m2._vit, img, batch=64), it=2)
        extras["vit_b16_384"] = {"images_per_s": 64 / (msv / 1e3), "batch": 64, "ms": msv}
        # K/V reuse = 1: every triplet names a different gallery image (what a 1 M-image gallery with disjoint lists looks like)
        try:
            q1 = min(22, Q)
            perm = torch.randperm(G, generator=gq)[: q1 * min(K, G // q1)].view(q1, -1).int().numpy()
            z1, _ = m1.encode_queries(tokens, ref_d[:q1], ids_d[:q1], mask_d[:q1], want_z=True, want_emb=False)
            old = eng.max_candidates
            eng.max_candidates = 512
            ms_r1 = _time(lambda: m2.score_triplets(z1, ids_d[:q1], mask_d[:q1], tokens, perm), it=2)
            eng.max_candidates = old
            extras["reuse_1"] = {"triplets_per_s": perm.size / (ms_r1 / 1e3), "triplets": int(perm.size), "ms": ms_r1,
                                 "note": "no K/V reuse: every triplet projects its own candidate's K/V (32.7 GF extra per triplet); chunk = 512 candidates"}
        except Exception as ex_:
            extras["reuse_1"] = {"error": repr(ex_)[:200]}
        # the reference's per-query formulation on stock PyTorch (ATen / cuBLAS) on this same B200: the oracle's torch code
        # with weights and inputs moved to the GPU -- the library baseline SURVEY 8(d) asks for
        try:
            from oracle import cir_oracle as O
            sd1c = {k: v.to(dev) for k, v in syn.make_stage1_state_dict(0, 384, "reference").items()}
            sd2c = {k: v.to(dev) for k, v in syn.make_stage2_state_dict(0, 384, "reference").items()}
            tok32 = tokens[: K + 1].float()
            ids_l, mask_l = ids_d[:4].long(), mask_d[:4].long()

            def torch_pass():
                with torch.no_grad():
                    for q in range(4):
                        z = O.stage1_hidden(sd1c, tok32[:1], ids_l[q:q + 1], mask_l[q:q + 1])
                        sc = O.stage2_score(sd2c, z, ids_l[q:q + 1], mask_l[q:q + 1], tok32[1:])
                        torch.argsort(sc, descending=True)
            ms32 = _time(torch_pass, it=2)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                ms16 = _time(torch_pass, it=2)
            extras["stock_pytorch_b200"] = {"fp32_triplets_per_s": 4 * K / (ms32 / 1e3), "bf16_autocast_triplets_per_s": 4 * K / (ms16 / 1e3),
                                            "sample": f"4 queries x {K} candidates, per-query loop as in src/validate_stage2.py:94-125 (z_t + "
                                                      "img_txt_fusion_val + argsort), oracle torch code on cuda"}
            del sd1c, sd2c, tok32
        except Exception as ex_:
            extras["stock_pytorch_b200"] = {"error": repr(ex_)[:200]}

    value = n_trip / (ms_step / 1e3)
    e2e_value = n_trip / (ms_e2e / 1e3)
    peak, hbm_peak, how = measured_peaks()
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    if rank == 0:
        cpu = None if args.no_cpu_baseline else cpu_baseline(args)
        traffic = committed_traffic()
        step_ms_total = ms_step * args.steps

        def sec(kind, name, unit, pk, bound):
            ms, wk, n = prof[kind]
            if n == 0:
                return None
            a = wk / (ms / 1e3) / (1e12 if unit == "TFLOP/s" else 1e9)
            return {"kernel": name, "bound": bound, "achieved": a, "peak": pk, "unit": unit, "frac": a / pk if pk else None,
                    "launches": int(n), "avg_launch_ms": ms / n, "share_of_step": ms / step_ms_total,
                    "traffic": (traffic.get(name) or {}).get("dram_bytes_per_launch")}
        secondary = [x for x in (
            sec(N.PROF_ATTN_TC, "fatc::attention_tc_kernel", "TFLOP/s", peak, "tensor (MUFU.EX2 co-limited: see DESIGN.md 5)"),
            sec(N.PROF_QKV_ATTN, "qkvattn::qkv_attention_kernel", "TFLOP/s", peak, "tensor"),
            sec(N.PROF_ATTN_SELF, "attention_small_kernel", "TFLOP/s", peak, "hbm (QKV re-read)"),
            sec(N.PROF_LAYERNORM, "add_layernorm_kernel", "GB/s", hbm_peak, "hbm")) if x]
        exec_flops = gemm_flops + prof[N.PROF_ATTN_TC][1] + prof[N.PROF_ATTN_SELF][1] + prof[N.PROF_QKV_ATTN][1]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_text(args),
                       "triplets_scored_per_step": n_trip, "chunk_triplets": eng.max_triplets, "chunk_candidates": eng.max_candidates,
                       "l2_note": "per-step working set (gallery tokens 2.0 GB + activations) exceeds the 126 MB L2; no flush needed",
                       "parallelism": (f"{world} ranks, {args.partition}-range partition of the fixed job; weights+gallery replicated; "
                                       "NCCL all-gather of z_t blocks and of (position, score) pairs") if world > 1 else "single GPU",
                       "rank0_plan": plan,
                       "kv_reuse_triplets_per_candidate_load": plan["triplets"] / max(1, plan["candidate_loads"])},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e,
                    "recall_at_10_50": [r10, r50]},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "tc::gemm_tcgen05_kernel", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak if peak else None, "peak_source": how,
                         "traffic": (traffic.get("tc::gemm_tcgen05_kernel") or {}).get("dram_bytes_per_launch"),
                         "traffic_source": traffic.get("source"),
                         "launches": int(gemm_n), "gflop_per_launch": gemm_flops / max(1, gemm_n) / 1e9,
                         "avg_launch_ms": gemm_ms / max(1, gemm_n), "gemm_share_of_step": gemm_ms / step_ms_total,
                         "gemm_plus_fused_qkv_share_of_step": (gemm_ms + prof[N.PROF_QKV_ATTN][0]) / step_ms_total,
                         "executed_tflops_gemm_plus_attention": exec_flops / (step_ms_total / 1e3) / 1e12,
                         "executed_frac_of_peak": exec_flops / (step_ms_total / 1e3) / 1e12 / peak if peak else None,
                         "effective_tflops_at_F_ref": value / world * F_REF_GF / 1e3,
                         "effective_frac_of_peak": value / world * F_REF_GF / 1e3 / peak if peak else None,
                         "secondary": secondary},
            "cpu_baseline": cpu,
            "clocks": sampler.summary(),
            "cross_rank_check": check,
            "extras": extras,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
