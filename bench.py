#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json metric: scored triples/pairs per second at d=100).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): TransE, d=100, |E|=100k, |R|=500, batches of 1024 positives
with 10 corrupted negatives each; region: forward + margin loss + backward (row gradients).

GPU arm.  One STEP = `--launches-per-step` (128) launches of the fused step kernel, each over
`--batches-per-step` (256) such batches (a single 11 264-triple batch is ~14 MB = 2 us of HBM time,
i.e. launch-latency bound; SURVEY.md 8d asks for the steady-state stream, and 20 steps of 128
launches give a timed region of ~1 s).  `value` = scored triples / s with indices resident in HBM,
CUDA events around the K steps, max over ranks; `e2e` = the same through the module API with pinned
host index buffers copied in every launch and the per-batch losses read back every step inside the
timed region.  N > 1: independent replicas, one per GPU (the training path does not shard; DESIGN.md),
value = sum over ranks / max-over-ranks time.  The line also carries
  roofline            dominant kernel vs the measured HBM peak, plus the same kernel at |E| = 500k and 5M
                      (tables far larger than L2) -- DRAM traffic from the ncu captures under profiles/
  regions             BASELINE.md section 4 regions for configs[1..4] on the GPU
  full_train_step     step + global-norm clip + sparse-row optimizer (SURVEY 8f-1); the configs[3]
                      alternating rec / KG loop
  eval                configs[4] shapes: d=128, 5M entities (top-10 and rank counts) and 1M users x 1M items,
                      catalog row-sharded over the N GPUs + ONE NCCL all-gather (top-K) / all-reduce (counts)
  cpu_baseline        (N=1) the reference itself on the host cores, same regions

--impl reference: the reference's own CPU implementation -- the unmodified model classes from
baseline/_ref (baseline/make_ref.py) -- timed on the host cores; each step a bounded sample
(`--ref-batches-per-step` batches) of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "joint-kg-recommender_b200"), os.path.join(ROOT, "baseline")):
    if p not in sys.path:
        sys.path.insert(0, p)

D, N_ENT, N_REL, BATCH, K_NEG = 100, 100_000, 500, 1024, 10
METRIC = "scored (h,r,t) triples/s, TransE d=100 forward + margin loss + backward"
# identical in both arms: what is measured, not how
CONFIG = {"workload": "configs[1]: transe d=100 |E|=100k |R|=500, batches of 1024 positives + 10 corrupted negatives each",
          "region": "forward + marginLoss + backward (row gradients of every gathered row)",
          "units": "a batch counts 1024 * (1 + 10) scored triples",
          "l2": "inputs larger than L2: the index arrays (14 MB / 256 batches, three sets in rotation) and the "
                "1.3 GB of gradient rows per launch stream through the 126 MB L2; the 40 MB entity table of configs[1] is "
                "L2-resident by construction (see roofline.hbm_regime for |E| = 500k / 5M)"}
ROW = 4 * D
FWD_GROUP_BYTES = ((3 + K_NEG) * ROW + (3 + K_NEG) * 4 + (1 + K_NEG) * 4) / (1 + K_NEG)      # 481 B / triple
STEP_GROUP_BYTES = (2 * (3 + K_NEG) * ROW + (3 + K_NEG) * 4 + (1 + K_NEG) * 4) / (1 + K_NEG)  # 954 B / triple
FP32_LANE_OPS = 148 * 128 * 1.965e9


def ncu_traffic(key):
    """DRAM bytes per launch from the committed ncu capture of this kernel at this shape."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            e = json.load(f)[key]
        return e["bytes"], e.get("capture")
    except Exception:
        return None, None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 7 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 7 and r[2].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def add_region_aliases(out):
    """BASELINE.md section 4 asks for the configs[3] / configs[4] regions beside the reference's: the GPU numbers are
    measured by the `joint_train_cfg4` and `eval` legs (whole optimizer steps and top-K passes: MORE work per unit than the
    reference arm's forward + backward / score-matrix regions); list them under `regions` next to the configs[1..2] keys
    so that one dict holds every config.  Pure bookkeeping on already-measured values; never raises."""
    try:
        reg = out.get("regions")
        if reg is None:
            return out
        j, ev = out.get("joint_train_cfg4"), out.get("eval")
        if j:
            reg["cfg4_ktup_rec_step_forward_backward_regularisers_clip_update"] = j["rec_pairs_per_s"]
            reg["cfg4_ktup_kg_step_forward_backward_regularisers_clip_update"] = j["kg_triples_per_s"]
        if ev:
            for key, name in (("kg_top10", "cfg5_transe_evaluateTail_top10_%dq_x_%d_d128"),
                              ("kg_rank_counts", "cfg5_transe_evaluateTail_rank_counts_%dq_x_%d_d128")):
                if key in ev:
                    reg[name % (ev[key]["queries"], ev[key]["catalog_rows"])] = ev[key]["pairs_per_s"]
            if "rec_top10" in ev:
                r = ev["rec_top10"]
                reg["cfg5_tup_soft_evaluate_top10_%du_x_%d_d128" % (r["users_scored"], r["items"])] = r["pairs_per_s"]
    except Exception:
        pass
    return out


def make_indices(torch, gen, n_batches, n_ent=N_ENT, n_rel=N_REL, k_neg=K_NEG):
    """Synthetic positives + corrupt-head/tail negatives (utils/data.py:12-18), int32."""
    n_pos = n_batches * BATCH
    ph = torch.randint(0, n_ent, (n_pos,), generator=gen, dtype=torch.int32)
    pt = torch.randint(0, n_ent, (n_pos,), generator=gen, dtype=torch.int32)
    pr = torch.randint(0, n_rel, (n_pos,), generator=gen, dtype=torch.int32)
    corrupt = torch.randint(0, n_ent, (n_pos * k_neg,), generator=gen, dtype=torch.int32)
    head = torch.rand(n_pos * k_neg, generator=gen) < 0.5
    cfmt = torch.where(head, ~corrupt, corrupt)              # group-compact format: sign bit = head replaced
    return [x.contiguous() for x in (ph, pt, pr, cfmt)]


DUMP_GRAD_SLOTS = 32_768           # gradient rows kept per table: 2 x 32768 x 100 floats = 26 MB


def dump_outputs(out_dir, torch, last, model):
    """What the last launch of the timed region returned to its caller -- per-batch losses, positive and negative
    scores -- and the sparse gradients it left in .grad, as DIR/<name>.npy.  Each gradient is a COO tensor with one
    row per gathered slot (3.1M entity slots at the default shape); a fixed, seeded sample of slots is written: the
    slot positions, the table row each one updates and its gradient row."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    loss, pos, neg = last
    arrays = {"loss_per_batch": loss, "pos_scores": pos, "neg_scores": neg}
    for name in ("ent", "rel"):
        g = getattr(model, name + "_embeddings").weight.grad
        rows, vals = g._indices()[0], g._values()
        pick = torch.randperm(rows.numel(), generator=torch.Generator().manual_seed(2024))[:DUMP_GRAD_SLOTS]
        pick = pick.sort().values
        arrays[name + "_grad_slots"] = pick.double()
        arrays[name + "_grad_rows"] = rows[pick.to(rows.device)].double()
        arrays[name + "_grad_values"] = vals[pick.to(vals.device)]
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


# =============================================================================================================
# reference arm
# =============================================================================================================
def run_reference(args):
    """CPU arm: the unmodified reference classes (baseline/_ref) on a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import ref_arm
    res = ref_arm.time_headline(args.steps, args.warmup, args.ref_batches_per_step)
    out = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "triples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": CONFIG,
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "step_is": "%d reference batches (bounded sample of the workload)" % args.ref_batches_per_step,
    }
    if not args.no_regions:
        out["regions"] = ref_arm.regions(reps=2)
    print(json.dumps(out))


# =============================================================================================================
# GPU arm
# =============================================================================================================
def run_ours(args):
    import torch
    import torch.distributed as dist
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    from kgrec_b200.models.base import device_init
    from kgrec_b200.data import DevicePrefetcher
    from kgrec_b200.optim import SparseRowOptimizer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    json_fd = 1
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its version / debug banner on fd 1 from C, so fd 1 is pointed at
        # stderr for the life of the process and the line is written to a duplicate of the real stdout
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(1234 + rank)
    nb, lps = args.batches_per_step, args.launches_per_step
    n_pos = nb * BATCH
    n_tri = n_pos * (1 + K_NEG)                              # scored triples per launch

    def ev_pair():
        return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timeit(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = ev_pair()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    model = K.TransEModel(False, D, N_ENT, N_REL)
    model.grad_mode = "sparse"
    n_sets = 3                                           # rotate index sets so no launch re-reads its ids from L2
    host_sets = [[x.pin_memory() for x in make_indices(torch, gen, nb)] for _ in range(n_sets)]
    dev_sets = [[x.to(dev) for x in hs] for hs in host_sets]
    loss_host = torch.empty((lps, nb), dtype=torch.float32).pin_memory()

    def launch_device(s):
        ix = dev_sets[s % n_sets]
        model.zero_grad(set_to_none=True)
        return model.loss_step_corrupt(tuple(ix[:3]), ix[3], margin=1.0, batch_pos=BATCH)

    # ---- device-resident timing: K steps of `lps` launches ---------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for s in range(max(args.warmup, 3) * lps):
        launch_device(s)
    launches0 = model.kernel_launches
    barrier()
    t0, t1 = ev_pair()
    step_evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    t0.record()
    step_evs[0].record()
    for k in range(args.steps):
        for s in range(lps):
            last = launch_device(k * lps + s)
        step_evs[k + 1].record()
    t1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, last, model)
    total_ms = max_over_ranks(t0.elapsed_time(t1))
    step_ms = sorted(step_evs[k].elapsed_time(step_evs[k + 1]) for k in range(args.steps))
    launches = model.kernel_launches - launches0
    ms_per_step = total_ms / args.steps
    launch_ms = ms_per_step / lps
    value = world * lps * n_tri / (ms_per_step * 1e-3)

    # ---- end to end through the module API with host buffers ------------------------------------------------
    # ids start in pinned host memory; the package's DevicePrefetcher copies launch i+1 on a side stream while
    # launch i runs; every launch's per-batch losses are copied to the host and each STEP ends with a stream
    # sync (the caller reads the step's losses), so all H2D / D2H traffic is inside the timed region.
    def host_batches(n, base):
        for s in range(n):
            yield host_sets[(base + s) % n_sets]

    def step_e2e(k):
        for i, ix in enumerate(DevicePrefetcher(host_batches(lps, k * lps), dev)):
            model.zero_grad(set_to_none=True)
            loss, _, _ = model.loss_step_corrupt(tuple(ix[:3]), ix[3], margin=1.0, batch_pos=BATCH)
            loss_host[i].copy_(loss.detach(), non_blocking=True)
        torch.cuda.current_stream().synchronize()       # the caller reads the step's losses
        return float(loss_host[0, 0])
    for k in range(max(3, args.warmup)):
        step_e2e(k)
    import gc
    gc.collect()
    gc.disable()                                   # no collector pause inside the timed host loop
    barrier()
    e_evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    e_evs[0].record()
    for k in range(args.steps):
        step_e2e(k)
        e_evs[k + 1].record()
    barrier()
    gc.enable()
    e2e_total = max_over_ranks(e_evs[0].elapsed_time(e_evs[args.steps]))
    e2e_steps = sorted(e_evs[k].elapsed_time(e_evs[k + 1]) for k in range(args.steps))
    e2e_ms = e2e_total / args.steps
    clocks = sampler.stop() if rank == 0 else None
    h2d = lps * sum(x.numel() * x.element_size() for x in host_sets[0])
    e2e = {"value": world * lps * n_tri / (e2e_ms * 1e-3), "unit": "triples/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": lps * nb * 4, "ms_per_step": e2e_ms, "launches_per_step": lps,
           "step_ms_min_median_max": [e2e_steps[0], e2e_steps[len(e2e_steps) // 2], e2e_steps[-1]],
           "pipeline": "DevicePrefetcher: H2D of launch i+1 overlaps launch i; per-batch losses copied back every launch, "
                       "stream sync + host read every step; %d launches timed" % (lps * args.steps)}

    out = {
        "metric": METRIC, "value": value, "unit": "triples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": CONFIG,
        "step_is": "%d launches x %d batches x %d triples; forward + margin loss + sparse-row-gradient backward fused in "
                   "k_group_step_e (COO slot ids written by the same pass), negatives in the group-compact corrupted-id format; "
                   "replicas x%d (the training path does not shard)" % (lps, nb, BATCH * (1 + K_NEG), world),
        "step_ms_min_median_max": [step_ms[0], step_ms[len(step_ms) // 2], step_ms[-1]],
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
    }

    extra = rank == 0 and world == 1 and not args.headline_only      # the single-GPU legs run at N = 1 only
    peak, peak_src = measured_peak()
    # ---- roofline of the dominant kernel (+ the same kernel with tables far larger than L2) -------------------
    step_gbs = n_tri * STEP_GROUP_BYTES / (launch_ms * 1e-3) / 1e9
    traffic, capture = ncu_traffic("k_group_step_e@E100k")
    out["roofline"] = {
        "bound": "hbm", "kernel": "k_group_step_e", "achieved": step_gbs, "peak": peak, "unit": "GB/s",
        "frac": step_gbs / peak, "traffic": traffic, "traffic_source": capture, "peak_source": peak_src,
        "bytes_per_triple": STEP_GROUP_BYTES, "launch_ms": launch_ms,
        "dram_frac": (traffic / (launch_ms * 1e-3) / 1e9 / peak) if traffic else None,
        "note": "achieved = algorithmic bytes (SURVEY 8d fused-group accounting: (3+K) rows read + (3+K) gradient rows written "
                "per 1+K triples) / mean launch time over the timed region (includes the per-batch loss reduction kernel "
                "and the host glue between launches); frac can exceed the DRAM view because configs[1]'s 40 MB table is served "
                "by L2: dram_frac = ncu DRAM bytes / time / peak"}
    if extra:
        hbm = {}
        for n_ent in (500_000, 5_000_000):
            with device_init(dev):
                bm = K.TransEModel(False, D, n_ent, N_REL)
            bm.grad_mode = "sparse"
            g2 = torch.Generator().manual_seed(77)
            sets = [[x.to(dev) for x in make_indices(torch, g2, nb, n_ent=n_ent)] for _ in range(2)]
            cnt = [0]

            def big_launch():
                ix = sets[cnt[0] % 2]
                cnt[0] += 1
                bm.zero_grad(set_to_none=True)
                bm.loss_step_corrupt(tuple(ix[:3]), ix[3], margin=1.0, batch_pos=BATCH)
            ms = timeit(big_launch, reps=10, warm=3)
            gbs = n_tri * STEP_GROUP_BYTES / (ms * 1e-3) / 1e9
            key = "k_group_step_e@E%s" % ("500k" if n_ent == 500_000 else "5M")
            tr, cap = ncu_traffic(key)
            hbm[key] = {"entities": n_ent, "table_MB": n_ent * ROW / 1e6, "launch_ms": ms, "triples_per_s": n_tri / (ms * 1e-3),
                        "achieved": gbs, "frac": gbs / peak, "traffic": tr, "traffic_source": cap,
                        "dram_frac": (tr / (ms * 1e-3) / 1e9 / peak) if tr else None}
            del bm, sets
        out["roofline"]["hbm_regime"] = hbm

    # ---- regions of BASELINE.md section 4 on the GPU (rank 0) -------------------------------------------------------
    if extra:
        reg = {}
        ix = dev_sets[0]
        ms = timeit(lambda: model.rank_loss_corrupt(tuple(ix[:3]), ix[3], margin=1.0, batch_pos=BATCH))
        reg["cfg2_transe_forward"] = n_tri / (ms * 1e-3)
        reg["cfg2_transe_forward_backward"] = n_tri / (launch_ms * 1e-3)
        nq = 4096
        q = torch.arange(nq, device=dev) % N_ENT
        qr = torch.arange(nq, device=dev) % N_REL
        ms = timeit(lambda: model.topk("tail", q, qr, k=10), reps=3)
        reg["cfg2_transe_evaluateTail_top10_4096q_x_100k"] = nq * N_ENT / (ms * 1e-3)
        ms = timeit(lambda: model.evaluateTail(q[:512], qr[:512]), reps=3)
        reg["cfg2_transe_evaluateTail_full_matrix_512q_x_100k"] = 512 * N_ENT / (ms * 1e-3)
        # configs[2]: TUP d=100 P=20 ST-Gumbel 50k x 50k
        torch.manual_seed(13)
        with device_init(dev):
            tm = K.TransUPModel(False, D, 50_000, 50_000, 20, True)
        tm.grad_mode = "sparse"
        tg = torch.Generator().manual_seed(5)
        tu, ti, tn = (torch.randint(0, 50_000, (n_pos,), generator=tg, dtype=torch.int32).to(dev) for _ in range(3))
        ms = timeit(lambda: tm.rank_loss((tu, ti), (tu, tn), target=-1.0, batch_pos=BATCH))
        reg["cfg3_tup_gumbel_forward"] = 2 * n_pos / (ms * 1e-3)

        def tup_step():
            tm.zero_grad(set_to_none=True)
            tm.loss_step((tu, ti), (tu, tn), target=-1.0, batch_pos=BATCH)
        tup_ms = timeit(tup_step)
        reg["cfg3_tup_gumbel_forward_backward"] = 2 * n_pos / (tup_ms * 1e-3)
        # the whole training step through the optimizer: row-factored ST-Gumbel step vs the pair kernel
        gopt = SparseRowOptimizer(tm, optimizer_type="Adagrad", lr=0.005, clip=5.0)

        def tup_gumbel_full():
            gopt.step_pairs((tu, ti), (tu, tn), target=-1.0, batch_pos=BATCH, reg=True)
        gum_rows_ms = timeit(tup_gumbel_full)
        os.environ["KGREC_REC_ROWS"] = "0"
        gum_pairs_ms = timeit(tup_gumbel_full)
        os.environ.pop("KGREC_REC_ROWS")
        del gopt
        qu = torch.arange(4096, device=dev) % 50_000
        gcat = tm.gumbel_catalog()                    # augmented item rows, built once per table state
        ms = timeit(lambda: tm.topk_items(qu, k=10, soft_catalog=gcat), reps=3)
        reg["cfg3_tup_gumbel_evaluate_top10_4096u_x_50k"] = 4096 * 50_000 / (ms * 1e-3)
        del gcat
        tm.use_st_gumbel = False
        soft_cat = tm.soft_catalog()
        qu4 = torch.arange(4096, device=dev) % 50_000
        ms = timeit(lambda: tm.topk_items(qu4, k=10, soft_catalog=soft_cat), reps=3)
        reg["cfg3_tup_soft_evaluate_top10_4096u_x_50k"] = 4096 * 50_000 / (ms * 1e-3)
        # the same tables trained with soft preferences through the optimizer: row-factored step vs the pair kernel
        topt = SparseRowOptimizer(tm, optimizer_type="Adagrad", lr=0.005, clip=5.0)

        def tup_soft_step():
            topt.step_pairs((tu, ti), (tu, tn), target=-1.0, batch_pos=BATCH, reg=True)
        soft_rows_ms = timeit(tup_soft_step)
        os.environ["KGREC_REC_ROWS"] = "0"
        soft_pairs_ms = timeit(tup_soft_step)
        os.environ.pop("KGREC_REC_ROWS")
        tables_finite = all(bool(torch.isfinite(v).all()) for v in tm._weights().values())   # after ~30 optimizer steps of both kinds
        del tm, soft_cat, topt
        out["regions"] = reg
        out["train_rec"] = {"tup_st_gumbel": {"ms": tup_ms, "pairs_per_s": 2 * n_pos / (tup_ms * 1e-3), "fma_per_pair": 14000,
                                              "frac_of_fp32_bound": 2 * n_pos / (tup_ms * 1e-3) * 14000 / FP32_LANE_OPS},
                            "tup_st_gumbel_full_step": {"what": "configs[2]: forward + BPR + backward + regularisers + clip + sparse-row Adagrad, "
                                                                "ST-Gumbel, L2, 50k users x 50k items, %d positives + 1 negative each" % n_pos,
                                                        "row_factored_ms": gum_rows_ms, "pair_kernel_ms": gum_pairs_ms,
                                                        "pairs_per_s": 2 * n_pos / (gum_rows_ms * 1e-3)},
                            "tables_finite_after_training": tables_finite,
                            "tup_soft_full_step": {"what": "forward + BPR + backward + regularisers + clip + sparse-row Adagrad, 50k users x 50k items, "
                                                           "%d positives + 1 negative each" % n_pos,
                                                   "row_factored_ms": soft_rows_ms, "pair_kernel_ms": soft_pairs_ms,
                                                   "pairs_per_s": 2 * n_pos / (soft_rows_ms * 1e-3)}}

    # ---- complete training steps: fused step + global-norm clip + sparse-row optimizer --------------------------------
    if extra:
        omodel = K.TransEModel(False, D, N_ENT, N_REL)
        opt = SparseRowOptimizer(omodel, optimizer_type="Adagrad", lr=0.01, clip=5.0)
        cnt = [0]

        def full_step():
            ix = dev_sets[cnt[0] % n_sets]
            cnt[0] += 1
            opt.step_corrupt(tuple(ix[:3]), ix[3], margin=1.0, batch_pos=BATCH)
        opt_ms = timeit(full_step, reps=20, warm=3)

        def full_step_reg():
            ix = dev_sets[cnt[0] % n_sets]
            cnt[0] += 1
            opt.step_corrupt(tuple(ix[:3]), ix[3], margin=1.0, batch_pos=BATCH, reg=True)
        reg_ms = timeit(full_step_reg, reps=20, warm=3)
        from kgrec_b200.sampling import TripleNegativeSampler
        kn = torch.stack([dev_sets[0][0], dev_sets[0][1], dev_sets[0][2]], dim=1).long().cpu()
        smp = TripleNegativeSampler(N_ENT, N_REL, kn, device=dev)

        def loop_step():
            ix = dev_sets[cnt[0] % n_sets]
            cnt[0] += 1
            opt.step_corrupt(tuple(ix[:3]), smp.sample(tuple(ix[:3]), K_NEG, seed=cnt[0]), margin=1.0, batch_pos=BATCH)
        loop_ms = timeit(loop_step, reps=20, warm=3)
        out["full_train_step"] = {
            "what": "k_group_step_e (dense accumulate) + k_rows_mark + k_rows_sqnorm (clip_grad_norm 5) + k_rows_update (sparse-row "
                    "Adagrad on the touched rows), %d batches per step (kgrec_b200.optim.SparseRowOptimizer)" % nb,
            "ms": opt_ms, "triples_per_s": n_tri / (opt_ms * 1e-3),
            "with_fused_regularisers_ms": reg_ms,
            "with_device_negative_sampling_ms": loop_ms,
            "with_device_negative_sampling_triples_per_s": n_tri / (loop_ms * 1e-3)}
        del omodel, opt, smp

        # TransR (configs[1] shapes, d x d projection per relation): the relation-run step kernel through the optimizer
        with device_init(dev):
            rmodel = K.TransRModel(False, D, N_ENT, N_REL)
        ropt = SparseRowOptimizer(rmodel, optimizer_type="Adagrad", lr=0.01, clip=5.0)
        nb_r = min(nb, 32)
        rix = [x[: nb_r * BATCH * (K_NEG if i == 3 else 1)] for i, x in enumerate(dev_sets[0])]

        def transr_step():
            ropt.step_corrupt(tuple(rix[:3]), rix[3], margin=1.0, batch_pos=BATCH)
        tr_ms = timeit(transr_step, reps=5, warm=2)
        n_grp = nb_r * BATCH
        fma_grp = 3 * (2 + K_NEG) * D * D                # Y = V M^T, dM += G^T V, dV = G M over the group's 2 + K rows
        out["train_transr"] = {
            "what": "TransR d=%d, %d relations: counting sort by relation + k_run_step_r (M_r, M_r^T resident per run, packed-FMA "
                    "register-tiled GEMMs) + clip + sparse-row Adagrad; %d batches of 1024 positives + %d negatives per step" % (D, N_REL, nb_r, K_NEG),
            "ms": tr_ms, "triples_per_s": n_grp * (1 + K_NEG) / (tr_ms * 1e-3), "fma_per_group": fma_grp,
            "frac_of_fp32_bound": n_grp / (tr_ms * 1e-3) * fma_grp / FP32_LANE_OPS}
        del rmodel, ropt

        # configs[3]: KTUP joint training, ml1m-scale rec (6040 x 3706) + 500k entities, R = P = 20, joint_ratio 0.5:
        # 5 rec steps then 5 KG steps per 10 (knowledgable_recommendation.py:209,320), each step = `nb` batches of 1024
        import numpy as np
        n_user, n_item, n_ent4, n_rel4 = 6040, 3706, 500_000, 20
        ents = np.random.RandomState(0).permutation(n_ent4)[:n_item]
        new_map = {i: (int(ents[i]) if i % 10 < 7 else -1, i) for i in range(n_item)}
        with device_init(dev):
            jm = K.jTransUPModel(False, D, n_user, n_item, n_ent4, n_rel4, {i: i for i in range(n_item)}, new_map, False, False)
        jopt = SparseRowOptimizer(jm, optimizer_type="Adagrad", lr=0.005, clip=5.0)
        jg = torch.Generator().manual_seed(6)
        ju = torch.randint(0, n_user, (n_pos,), generator=jg, dtype=torch.int32).to(dev)
        jpi, jni = (torch.randint(0, n_item, (n_pos,), generator=jg, dtype=torch.int32).to(dev) for _ in range(2))
        jk = [x.to(dev) for x in make_indices(torch, jg, nb, n_ent=n_ent4, n_rel=n_rel4, k_neg=1)]

        def rec_step():
            jopt.step_pairs((ju, jpi), (ju, jni), target=-1.0, batch_pos=BATCH, reg=True)

        def kg_step():
            jopt.step_corrupt(tuple(jk[:3]), jk[3], margin=1.0, batch_pos=BATCH, reg=True, grad_loss=1.0)

        def joint_cycle():
            for _ in range(5):
                rec_step()
            for _ in range(5):
                kg_step()
        rec_ms, kg_ms = timeit(rec_step, reps=5), timeit(kg_step, reps=5)
        os.environ["KGREC_REC_ROWS"] = "0"           # A/B: the pair (tile) kernel instead of the row-factored soft step
        rec_pairs_ms = timeit(rec_step, reps=5)
        os.environ.pop("KGREC_REC_ROWS")
        cyc_ms = timeit(joint_cycle, reps=3, warm=1)
        units = 5 * 2 * n_pos + 5 * 2 * n_pos            # scored pairs + scored triples per 10-step cycle
        out["joint_train_cfg4"] = {
            "what": "jtransup, joint_ratio 0.5: 5 rec steps (tile kernel + orthogonalLoss + clip + sparse-row Adagrad) then 5 KG steps "
                    "(TransH step kernel with fused regularisers + clip + update) per cycle; %d batches of 1024 positives + 1 negative per step; "
                    "6040 users x 3706 items, 500k entities, R = P = 20" % nb,
            "rec_step_ms": rec_ms, "rec_step_pair_kernel_ms": rec_pairs_ms, "kg_step_ms": kg_ms, "cycle_ms": cyc_ms, "scored_pairs_plus_triples_per_s": units / (cyc_ms * 1e-3),
            "rec_pairs_per_s": 2 * n_pos / (rec_ms * 1e-3), "kg_triples_per_s": 2 * n_pos / (kg_ms * 1e-3)}
        del jm, jopt

    # ---- single-batch latency (the shape every unchanged driver step has) --------------------------------------------
    if extra:
        small = [x[:BATCH * (1 if i < 3 else K_NEG)].contiguous() for i, x in enumerate(dev_sets[0])]

        def one_batch():
            model.zero_grad(set_to_none=True)
            model.loss_step_corrupt(tuple(small[:3]), small[3], margin=1.0)
        out["single_batch_latency_us"] = timeit(one_batch, reps=50, warm=5) * 1e3
        gs = model.graphed_loss_step(BATCH, K_NEG, margin=1.0)
        for buf, src in ((gs.h, small[0]), (gs.t, small[1]), (gs.r, small[2]), (gs.corrupt, small[3])):
            buf.copy_(src)
        out["single_batch_latency_graph_us"] = timeit(gs.replay, reps=200, warm=10) * 1e3
        out["single_batch_note"] = ("one 1024 pos + 10 neg/pos batch, forward + margin loss + backward: module API call vs the same two "
                                    "kernels replayed from a CUDA graph over static id buffers (TransEModel.graphed_loss_step)")

    # ---- full-catalog evaluation at configs[4] shapes, catalog row-sharded over the N GPUs ----------------------------
    if not args.no_eval:
        d5 = 128
        ev = {}
        torch.manual_seed(7)                                  # the same tables on every rank
        with device_init(dev):
            torch.cuda.manual_seed(7)
            emodel = K.TransEModel(False, d5, args.eval_entities, N_REL)
        n_cat = args.eval_entities
        lo, hi = KE.shard_bounds(n_cat, world, rank)
        shard = emodel.ent_embeddings.weight.detach()[lo:hi]
        nq = args.eval_queries
        qg = torch.Generator().manual_seed(99)
        qh = torch.randint(0, n_cat, (nq,), generator=qg).to(dev)
        qr = torch.randint(0, N_REL, (nq,), generator=qg).to(dev)
        gold = torch.randint(0, n_cat, (nq,), generator=qg).to(dev)

        def topk_pass():
            keys = emodel.topk("tail", qh, qr, k=10, catalog=shard, id_base=lo)
            return KE.sharded_topk(keys) if world > 1 else keys

        gs = emodel.gold_scores("tail", qh, qr, gold)

        def rank_pass():
            cnt = emodel.rank_counts("tail", qh, qr, gold, gold_scores=gs, catalog=shard, id_base=lo)
            return KE.sharded_rank_counts(cnt) if world > 1 else cnt
        for name, fn in (("kg_top10", topk_pass), ("kg_rank_counts", rank_pass)):
            for _ in range(2):
                fn()
            barrier()
            a0, a1 = ev_pair()
            a0.record()
            for _ in range(3):
                fn()
            a1.record()
            barrier()
            ems = max_over_ranks(a0.elapsed_time(a1)) / 3
            bound = FP32_LANE_OPS / (2 * d5) * world
            ev[name] = {"pairs_per_s": nq * n_cat / (ems * 1e-3), "ms": ems, "queries": nq, "catalog_rows": n_cat, "d": d5,
                        "collective": ("1 NCCL all-gather of [nq,10] uint64 keys" if name == "kg_top10" else "1 NCCL all-reduce of [nq] int32 counts")
                        if world > 1 else "none (1 GPU)",
                        "frac_of_fp32_bound": nq * n_cat / (ems * 1e-3) / bound}
        del emodel, shard
        # rec side: 1M users x 1M items, TUP soft preferences (the shipped transup.sh setting), top-10
        with device_init(dev):
            torch.cuda.manual_seed(11)
            rmodel = K.TransUPModel(False, d5, args.eval_users, args.eval_items, 20, False)
        ilo, ihi = KE.shard_bounds(args.eval_items, world, rank)
        soft_cat = rmodel.soft_catalog(rmodel.item_embeddings.weight.detach()[ilo:ihi])
        nu = args.eval_rec_queries
        qu = torch.randint(0, args.eval_users, (nu,), generator=qg).to(dev)

        def rec_pass():
            keys = rmodel.topk_items(qu, k=10, soft_catalog=soft_cat, id_base=ilo)
            return KE.sharded_topk(keys) if world > 1 else keys
        for _ in range(2):
            rec_pass()
        barrier()
        a0, a1 = ev_pair()
        a0.record()
        for _ in range(3):
            rec_pass()
        a1.record()
        barrier()
        rms = max_over_ranks(a0.elapsed_time(a1)) / 3
        ev["rec_top10"] = {"pairs_per_s": nu * args.eval_items / (rms * 1e-3), "ms": rms, "users_scored": nu, "users": args.eval_users,
                           "items": args.eval_items, "d": d5, "model": "TUP soft P=20",
                           "note": "augmented item rows of the shard built once (soft_catalog), user rows per call"}
        ev["sharding"] = "catalog rows / %d GPUs (strong scaling: total work fixed)" % world
        out["eval"] = ev
        del rmodel, soft_cat

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import ref_arm
        cb = ref_arm.time_headline(steps=1000, warmup=1, batches_per_step=1, budget_s=10.0)
        out["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if extra and not args.no_regions:
            out["cpu_baseline"]["regions"] = ref_arm.regions(reps=1)
    if rank == 0:
        add_region_aliases(out)
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batches-per-step", type=int, default=256, help="batches of 1024 positives per kernel launch")
    ap.add_argument("--launches-per-step", type=int, default=128)
    ap.add_argument("--ref-batches-per-step", type=int, default=4)
    ap.add_argument("--eval-queries", type=int, default=8192)
    ap.add_argument("--eval-entities", type=int, default=5_000_000)
    ap.add_argument("--eval-users", type=int, default=1_000_000)
    ap.add_argument("--eval-items", type=int, default=1_000_000)
    ap.add_argument("--eval-rec-queries", type=int, default=16384)
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-regions", action="store_true")
    ap.add_argument("--headline-only", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed launch computed (losses, scores, a seeded sample of the gradient rows) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
