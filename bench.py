#!/usr/bin/env python
"""Contract benchmark of the B200 path.

    python bench.py --gpus N --steps K --warmup W                # images/sec, BASELINE.json configs[1] (N=1) / [2] (N>1)
    torchrun --nproc-per-node N ... bench.py --gpus N ...        # one rank per GPU over NCCL
    python bench.py --impl reference ...                         # CPU arm: the oracle port of the reference path
    python bench.py --workload refiner [--gpus N]                # configs[4]: ProtoRefiner-only sweep, bank cell-sharded over N GPUs
    python bench.py --workload train [--gpus N] [--all-trainable]   # configs[3]: fine-tune step, gradient all-reduce overlapped
    python bench.py ... --dump-outputs DIR                       # also write the last timed step's outputs as DIR/<name>.npy

One step = one pass of the hot path over one batch of synthetic input:
  infer,   N = 1 : batch 256 four-view panoramas (1024 views), fp16 operands, + head + refine            (configs[1])
  infer,   N > 1 : 256 samples per rank, one packed all-gather of the per-rank head outputs, retrieval over a bank whose
                   geocells are sharded across the ranks (second small all-gather of the per-candidate partials)   (configs[2])
  refiner        : B = 8192 queries (the same on every rank), P = 1M prototypes, D = 768, bank cell-sharded   (configs[4])
  train          : 128 four-view samples per rank, forward + backward + AdamW, NCCL gradient averaging        (configs[3])
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the benchmark leaves the source tree as it found it (it may be read-only)

FLOP_PER_VIEW = 381.92e9          # SURVEY.md §8 / BASELINE.md §2 (un-padded, 2*MAC)
GEMM_FLOP_PER_VIEW = 87.12e9 + 29.04e9 + 232.33e9 + 0.69e9
ATTN_FLOP_PER_VIEW = 32.73e9
NUM_CELLS, NUM_PROTOS, TOPK, NUM_CAND = 1000, 100_000, 5, 50
REFINER_T, REFINER_MAX_KM = 1.6, 1000.0
METRIC = "four-view 336x336 images/sec (ViT-L/14 + geocell head + ProtoRefiner)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, f"/tmp/pg_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


class Dist:
    """Process-group plumbing shared by the workloads (one rank per GPU, NCCL)."""

    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        assert self.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"

    def timed(self, fn, steps, warmup):
        """W untimed steps, then exactly K steps between barrier + synchronize on both sides, CUDA events on the launch
        stream.  Returns (max over ranks of the ms, per-rank ms list, last result)."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = None
        for _ in range(steps):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()
        mine = torch.tensor([e0.elapsed_time(e1)], device=self.dev, dtype=torch.float64)
        per_rank = [mine.item()]
        if self.world > 1:
            allms = torch.empty(self.world, device=self.dev, dtype=torch.float64)
            self.dist.all_gather_into_tensor(allms, mine)
            per_rank = [float(x) for x in allms.tolist()]
        return max(per_rank), per_rank, r

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def host_outputs(name, value, out=None):
    """Host copies of the tensors in `value` (a tensor or a namedtuple of them, nested; None is skipped), keyed `name`
    or `name_<field>`."""
    out = {} if out is None else out
    if torch.is_tensor(value):
        out[name] = value.detach().cpu().clone()
    elif hasattr(value, "_fields"):
        for f in value._fields:
            host_outputs(f"{name}_{f}", getattr(value, f), out)
    return out


def dump_outputs(directory, arrays):
    """--dump-outputs: every array as <directory>/<name>.npy, float64 kept, other floats as float32, integers (indices)
    as float64, which holds them exactly."""
    os.makedirs(directory, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.numpy()
        a = a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in "iub" else np.float32)
        total += a.nbytes
        assert total <= 64 << 20, "--dump-outputs: more than 64 MB of outputs"
        np.save(os.path.join(directory, name + ".npy"), a)


def read_profile():
    """Per-launch device times recorded by the library between pg_profile_begin/end: {family: (ms, launches)}."""
    import ctypes as C
    from pigeon_b200 import _lib
    lib = _lib.load()
    n = lib.pg_profile_end()
    names = (C.c_char_p * n)()
    ms = (C.c_float * n)()
    counts = (C.c_int32 * n)()
    lib.pg_profile_read(names, ms, counts, n)
    return {names[i].decode(): (float(ms[i]), int(counts[i])) for i in range(n)}


# ================================================================================================ workload: infer
def build_models(device, seed=0, fold_layernorm=True, shard_cells=False):
    from pigeon_b200 import CLIPVisionTower, ProtoRefiner, SuperGuessr, VitDims, synthetic
    dims = VitDims()
    torch.manual_seed(1000 + seed)   # same geocell head on every rank (nn.Linear's default init uses the global RNG)
    tower = CLIPVisionTower(dims)
    tower.load_state_dict(synthetic.random_vit_state_dict(dims, seed=seed))
    tower.max_views_per_pass = 1024
    tower.fold_layernorm = fold_layernorm
    cells = synthetic.synthetic_geocells(NUM_CELLS, 0)
    model = SuperGuessr(tower, panorama=True, freeze_base=True, num_candidates=NUM_CAND, geocells=cells).to(device).eval()
    bank = synthetic.synthetic_bank(NUM_CELLS, NUM_PROTOS, dims.hidden, seed=2, members_mean=0.0, empty_cells=5)
    refiner = ProtoRefiner(topk=TOPK, max_refinement=REFINER_MAX_KM, temperature=REFINER_T, protos=bank, device=device,
                           shard_cells=shard_cells).eval()
    return model, refiner, dims, cells, bank


def parity_check(model, refiner, px_dev, labels, labels_clf, full, rank, with_oracle):
    """The timed pass runs 1024 views at once (M = 590 848 GEMM rows, 40 960 attention jobs): check ITS outputs.
      (1) a stride sample of the batch recomputed in a 16-view pass must reproduce the big pass bit for bit;
      (2) the first two images against the fp32 CPU oracle: embedding rel-L2 <= 1e-3, top-1 geocell identical."""
    from pigeon_b200 import evaluation
    ll_full, cell_full, out_full = full
    pooled_full = model.last_pooled.clone()               # view mean of the big pass (the small pass below overwrites it)
    B = px_dev.shape[0]
    lo = rank * B if ll_full.shape[0] > B else 0          # this rank's rows of the gathered outputs
    idx = torch.tensor(sorted({0, B // 3, (2 * B) // 3, B - 1}), device=px_dev.device)
    small = evaluation.predict_batch(model, None, dict(pixel_values=px_dev[idx], labels=labels[idx], labels_clf=labels_clf[idx]),
                                     gather=False)[2]
    res = {"small_pass_views": int(4 * idx.numel()),
           "embedding_bit_equal": bool(torch.equal(small.embedding, out_full.embedding[idx])),
           "top_candidates_equal": bool(torch.equal(small.top5_geocells.indices, out_full.top5_geocells.indices[idx]))}
    # refining this rank's own samples alone must give its rows of the (gathered, possibly cell-sharded) result
    from pigeon_b200 import ProtoRefiner
    solo = ProtoRefiner(topk=TOPK, max_refinement=REFINER_MAX_KM, temperature=REFINER_T, protos=refiner.protos,
                        device=px_dev.device).eval()
    _, ll_solo, cell_solo = solo(pooled_full, initial_preds=out_full.preds_LLH,
                                 candidate_cells=out_full.top5_geocells.indices, candidate_probs=out_full.top5_geocells.values)
    res["refined_rows_equal_local_refine"] = bool(torch.equal(ll_solo, ll_full[lo:lo + B]) and
                                                  torch.equal(cell_solo, cell_full[lo:lo + B]))
    if with_oracle:
        from oracle import head as ohead, vit as ovit
        from pigeon_b200 import synthetic
        from pigeon_b200.vit_engine import VitDims
        dims = VitDims()
        sd = synthetic.random_vit_state_dict(dims, seed=0)
        n_img = 2
        px = px_dev[:n_img].float().cpu().reshape(n_img * 4, 3, dims.image_size, dims.image_size)
        emb = ovit.clip_embedding(sd, px, patch=dims.patch_size, heads=dims.heads, layers=dims.layers, eps=dims.ln_eps)
        h = ohead.head_forward(emb.reshape(n_img, 4, -1), model.cell_layer.weight.detach().cpu(),
                               model.cell_layer.bias.detach().cpu(), model.lla_geocells.detach().cpu(), NUM_CAND, True)
        ours = out_full.embedding[:n_img].float().cpu().reshape(n_img * 4, -1)
        res["oracle_images"] = n_img
        res["oracle_embedding_rel_l2"] = float((ours.double() - emb.double()).norm() / emb.double().norm())
        res["oracle_top1_equal"] = bool(torch.equal(h.topk_idx[:, 0].cpu(), out_full.top5_geocells.indices[:n_img, 0].cpu()))
    res["ok"] = bool(res["embedding_bit_equal"] and res["top_candidates_equal"] and res["refined_rows_equal_local_refine"]
                     and res.get("oracle_embedding_rel_l2", 0.0) <= 1e-3 and res.get("oracle_top1_equal", True))
    return res


def run_infer(args):
    from pigeon_b200 import _lib, evaluation, synthetic
    D = Dist(args)
    world, rank, dev = D.world, D.rank, D.dev
    peaks = load_peaks()
    B = args.batch
    shard = world > 1 and not args.replicated_bank
    model, refiner, dims, cells, bank = build_models(dev, fold_layernorm=not args.no_ln_fold, shard_cells=shard)
    g = torch.Generator().manual_seed(1 + rank)
    # synthetic panoramas, fp16, (B, 12, 336, 336): view index fastest inside a sample (dataset_preprocessing.py:199-200)
    px_host = torch.randn(B, 12, dims.image_size, dims.image_size, generator=g, dtype=torch.float32).half().pin_memory()
    px_dev = px_host.to(dev)
    labels = torch.from_numpy(synthetic.synthetic_geocells(B, 7 + rank)).to(dev)
    labels_clf = (torch.arange(B) % NUM_CELLS).to(dev)

    def step_device():
        return evaluation.predict_batch(model, refiner, dict(pixel_values=px_dev, labels=labels, labels_clf=labels_clf))

    def step_e2e():
        ll, cell, out = evaluation.predict_batch(model, refiner, dict(pixel_values=px_host, labels=labels, labels_clf=labels_clf))
        return ll.cpu(), cell.cpu(), out.loss.cpu()          # device -> host read of the step's result

    sampler = ClockSampler(D.local)
    if rank == 0:
        sampler.start()
    ms, ms_by_rank, res = D.timed(step_device, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:      # the refiner's predictions and SuperGuessr's ModelOutput
        dump_outputs(args.dump_outputs, host_outputs("refined_preds_LLH", res[0]) |
                     host_outputs("refined_preds_geocell", res[1]) | host_outputs("model", res[2]))
    e2e_steps = max(2, min(args.steps, 5))
    ms_e2e, e2e_by_rank, _ = D.timed(step_e2e, e2e_steps, 1)

    # per-kernel-family device time of ONE step (CUDA events recorded by the library on the launch stream).
    # Every rank runs it (the step contains the all-gathers); only rank 0 reports.
    lib = _lib.load()
    lib.pg_profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    full = step_device()
    e1.record()
    torch.cuda.synchronize()
    fam = read_profile()
    total_ms = e0.elapsed_time(e1)

    check = parity_check(model, refiner, px_dev, labels, labels_clf, full, rank, with_oracle=(rank == 0 and not args.no_oracle_check))
    if world > 1:       # every rank's check must hold
        flag = torch.tensor([1 if check["ok"] else 0], device=dev)
        D.dist.all_reduce(flag, op=D.dist.ReduceOp.MIN)
        check["ok_all_ranks"] = bool(flag.item())

    images = B * world
    out = {
        "metric": METRIC, "value": images * args.steps / (ms / 1e3), "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp16",
        "data": "synthetic (randn panoramas, random-init ViT-L/14-336, 1000 synthetic geocells, 100k synthetic prototypes)",
        "config": {"workload": f"batch={B}/GPU four-view synthetic panoramas ({4 * B} views), ViT-L/14-336 embed + "
                               f"geocell head (C={NUM_CELLS}, top-{NUM_CAND}) + ProtoRefiner (P={NUM_PROTOS}, topk={TOPK}); "
                               "BASELINE.json configs[1]" + ("" if world == 1 else " per rank = configs[2] sharded"),
                   "global_batch": images, "views_per_gpu": 4 * B, "parallelism": f"dp{world}",
                   "l2": "inputs larger than L2 (0.69 GB pixels + >2 GB activations per step); no explicit flush",
                   "collective": "none" if world == 1 else
                                 ("2 packed all_gather_into_tensor (NCCL) per step: per-rank head outputs, then the per-candidate "
                                  "partials of the cell-sharded bank" if shard else
                                  "1 all_gather_into_tensor (NCCL) of per-rank head outputs per step, replicated bank"),
                   "layernorm": "kernels" if args.no_ln_fold else "folded into the GEMM epilogues"},
        "ms_per_step_by_rank": [m / args.steps for m in ms_by_rank],
        "e2e": {"value": images * e2e_steps / (ms_e2e / 1e3), "unit": "images/s",
                "h2d_bytes_per_step": px_host.numel() * 2, "d2h_bytes_per_step": B * world * (8 + 8) + 4,
                "ms_per_step_by_rank": [m / e2e_steps for m in e2e_by_rank], "steps": e2e_steps,
                "note": "SuperGuessr.forward + ProtoRefiner.forward with pinned HOST fp16 pixels, results read back"},
        "parity_check": check,
        "clocks": clocks,
        "tflops_per_gpu": FLOP_PER_VIEW * 4 * B * args.steps / (ms / 1e3) / 1e12,
    }
    views = 4 * B
    gemm = {k: v for k, v in fam.items() if k.startswith("gemm")}
    gemm_ms, gemm_n = sum(v[0] for v in gemm.values()), sum(v[1] for v in gemm.values())
    attn_ms = fam.get("attention", (0.0, 0))[0]
    ach = GEMM_FLOP_PER_VIEW * views / (gemm_ms / 1e3) / 1e12
    traffic, traffic_note = None, None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        t = json.load(open(tp))
        traffic, traffic_note = t.get("gemm_dram_bytes_per_launch"), t.get("how")
    out["roofline"] = {"kernel": "gemm2_f16_kernel (tcgen05 GEMM, all projection/MLP launches of one step)", "bound": "tensor",
                       "achieved": ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                       "frac": ach / peaks["tflops_sustained"], "traffic": traffic, "traffic_note": traffic_note,
                       "peak_source": peaks["source"] + ", sustained bf16 cuBLAS figure (kernel timed inside a long step)",
                       "launches": gemm_n, "avg_launch_ms": gemm_ms / max(gemm_n, 1), "share_of_step": gemm_ms / total_ms}
    a_ach = ATTN_FLOP_PER_VIEW * views / (attn_ms / 1e3) / 1e12 if attn_ms else 0.0
    attn_kernel = {None: "attention_fold_kernel", "fold": "attention_fold_kernel", "pair": "attention_pair_kernel",
                   "split": "attention_split_kernel"}.get(os.environ.get("PG_ATTN_VARIANT"), "attention_kernel (first generation)")
    out["roofline_attention"] = {"kernel": attn_kernel + " (tcgen05 QK^T / PV, softmax in between)", "bound": "tensor",
                                 "achieved": a_ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                                 "frac": a_ach / peaks["tflops_sustained"], "share_of_step": attn_ms / total_ms}
    out["kernel_ms_per_step"] = {"gemm_ms": round(gemm_ms, 3), "attention_ms": round(attn_ms, 3),
                                 "layernorm_ms": round(fam.get("layernorm", (0.0, 0))[0], 3),
                                 "other_ms": round(sum(v[0] for k, v in fam.items() if not k.startswith("gemm")
                                                       and k not in ("attention", "layernorm")), 3),
                                 "total_ms": round(total_ms, 3)}
    out["family_ms_per_step"] = {k: round(v[0], 3) for k, v in sorted(fam.items(), key=lambda kv: -kv[1][0])}
    out["gpu_launches"] = sum(v[1] for v in fam.values()) * args.steps     # counted by the library's launch hooks, per step
    out["launches_by_family_per_step"] = {k: v[1] for k, v in fam.items()}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(sample_images=args.cpu_sample)
    if rank == 0:
        print(json.dumps(out))
    D.close()


# ================================================================================================ workload: refiner
def run_refiner(args):
    """BASELINE.json configs[4]: ProtoRefiner-only, P = 1M prototypes, D = 768, C = 2076 geocells, B = 8192 queries with
    `topk` distinct candidate cells each.  N GPUs: strong scaling — every rank holds the same queries and the geocells with
    cell % N == rank (bank bytes per GPU / N), scans them, one packed all-gather of the (B, topk, 3) partials, merge by owner,
    final stage on every rank."""
    from pigeon_b200 import ProtoRefiner, _lib, bank as bank_mod
    D = Dist(args)
    world, rank, dev = D.world, D.rank, D.dev
    peaks = load_peaks()
    C, P, dim, B, k = 2076, 1_000_000, args.refiner_dim, 8192, args.refiner_topk
    rng = np.random.default_rng(0)
    sizes = rng.multinomial(P, np.ones(C) / C)
    cell_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    own = (np.arange(C) % world) == rank
    # the shard is generated on the device cell by cell from per-cell seeds, so every rank count sees the same bank
    my_sizes = np.where(own, sizes, 0)
    my_off = np.concatenate([[0], np.cumsum(my_sizes)]).astype(np.int64)
    Pm = int(my_off[-1])
    emb = torch.empty((max(Pm, 1), dim), dtype=torch.float32, device=dev)
    ll = torch.empty((max(Pm, 1), 2), dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev)
    for c in np.nonzero(own)[0]:
        if sizes[c] == 0:
            continue
        gen.manual_seed(1000 + int(c))
        emb[my_off[c]:my_off[c + 1]] = torch.randn(int(sizes[c]), dim, generator=gen, device=dev) * 0.3
        ll[my_off[c]:my_off[c + 1]] = torch.rand(int(sizes[c]), 2, generator=gen, device=dev) * 90
    arrays = dict(cell_off=my_off, proto_emb=emb[:Pm], proto_lnglat=ll[:Pm], proto_count=torch.ones(Pm, dtype=torch.int32),
                  member_off=torch.arange(Pm + 1), member_idx=torch.zeros(Pm, dtype=torch.int64),
                  data_emb=torch.zeros(1, dim), data_lnglat=torch.zeros(1, 2))
    refiner = ProtoRefiner(topk=k, max_refinement=REFINER_MAX_KM, temperature=REFINER_T, protos=dict(cell_off=my_off),
                           device=dev).eval()
    from pigeon_b200 import ops
    refiner._bank = ops.DeviceBank(dev, **arrays)          # pre-sharded bank, built on the device
    ops.refiner_set_schedule(args.refiner_schedule)
    refiner._bank_world = world
    rq = np.random.default_rng(3)
    cand = np.stack([rq.choice(C, size=k, replace=False) for _ in range(B)]).astype(np.int64)
    probs = -np.sort(-rq.dirichlet(np.ones(k), size=B), axis=1).astype(np.float32)
    gq = torch.Generator().manual_seed(11)
    q_host = (torch.randn(B, dim, generator=gq) * 0.3).pin_memory()
    init_host = (torch.rand(B, 2, generator=gq, dtype=torch.float64) * 90).pin_memory()
    cand_host, probs_host = torch.from_numpy(cand).pin_memory(), torch.from_numpy(probs).pin_memory()
    q, init, candt, probst = q_host.to(dev), init_host.to(dev), cand_host.to(dev), probs_host.to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def step_device():
        flush.zero_()                                       # the 0.4 GB shard at N = 8 would otherwise sit in the 126 MB L2 partly
        return refiner(q, initial_preds=init, candidate_cells=candt, candidate_probs=probst)

    def step_e2e():
        flush.zero_()
        _, ll_, cell_ = refiner(q_host.to(dev, non_blocking=True), initial_preds=init_host.to(dev, non_blocking=True),
                                candidate_cells=cand_host.to(dev, non_blocking=True),
                                candidate_probs=probs_host.to(dev, non_blocking=True))
        return ll_.cpu(), cell_.cpu()

    # the flush is inside the timed region: measure it alone and subtract
    def only_flush():
        flush.zero_()
    sampler = ClockSampler(D.local)
    if rank == 0:
        sampler.start()
    ms_f, _, _ = D.timed(only_flush, args.steps, 2)
    ms, ms_by_rank, res = D.timed(step_device, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:      # ProtoRefiner's (loss, preds_LLH, preds_geocell)
        dump_outputs(args.dump_outputs, host_outputs("loss", res[0]) | host_outputs("preds_LLH", res[1]) |
                     host_outputs("preds_geocell", res[2]))
    ms_e2e, e2e_by_rank, _ = D.timed(step_e2e, args.steps, 1)
    ms, ms_e2e = ms - ms_f, ms_e2e - ms_f
    lib = _lib.load()
    lib.pg_profile_begin()
    step_device()
    torch.cuda.synchronize()
    fam = read_profile()
    scan_ms = fam.get("refiner_scan", (0.0, 0))[0] + fam.get("refiner_scan_finish", (0.0, 0))[0]
    touched = np.unique(cand)
    mine = touched[(touched % world) == rank]
    alg_bytes = float(sizes[mine].sum()) * dim * 4 + B * dim * 4 + B * k * 12 + B * 32     # SURVEY.md 8d, per rank
    pair_elems = float(sizes[cand][(cand % world) == rank].sum()) * dim
    # result check against the replicated single-GPU answer is tools/refiner_shard_check.py (needs the whole bank on one GPU);
    # here: all ranks must agree bit for bit
    _, ll_, cell_ = res
    agree = True
    if world > 1:
        ref_ll, ref_cell = ll_.clone(), cell_.clone()
        D.dist.broadcast(ref_ll, 0); D.dist.broadcast(ref_cell, 0)
        flag = torch.tensor([1 if (torch.equal(ref_ll, ll_) and torch.equal(ref_cell, cell_)) else 0], device=dev)
        D.dist.all_reduce(flag, op=D.dist.ReduceOp.MIN)
        agree = bool(flag.item())
    out = {
        "metric": "refined queries/sec (ProtoRefiner-only sweep, BASELINE.json configs[4])",
        "value": B * args.steps / (ms / 1e3), "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (randn * 0.3 prototypes and queries, multinomial cell sizes, k distinct uniform candidate cells)",
        "config": {"workload": f"ProtoRefiner-only: P={P} prototypes, D={dim}, C={C} geocells, B={B} queries, topk={k}",
                   "parallelism": f"cells sharded over {world} GPU(s) (cell % N), queries replicated",
                   "bank_bytes_per_gpu": Pm * dim * 4,
                   "l2": "256 MB flush between steps (timed alone and subtracted)",
                   "collective": "none" if world == 1 else "1 packed all_gather_into_tensor (NCCL) of (B, topk, 3) fp32 partials per step"},
        "ms_per_step_by_rank": [m / args.steps for m in ms_by_rank],
        "e2e": {"value": B * args.steps / (ms_e2e / 1e3), "unit": "queries/s",
                "h2d_bytes_per_step": B * dim * 4 + B * 16 + B * k * 12, "d2h_bytes_per_step": B * 16},
        "roofline": {"kernel": ("slab_scan_kernel + tile_finish_kernel" if args.refiner_schedule in (0, 4) else
                                "tile_scan_kernel + tile_finish_kernel" if args.refiner_schedule == 3 else
                                "cell_major_scan_kernel" if args.refiner_schedule == 2 else "scan_kernel") + " (rank 0's shard)",
                     "bound": "hbm",
                     "achieved": alg_bytes / (scan_ms / 1e3) / 1e9 if scan_ms else None, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": (alg_bytes / (scan_ms / 1e3) / 1e9 / peaks["hbm_gbs"]) if scan_ms else None, "traffic": None,
                     "algorithmic_bytes": alg_bytes, "scan_ms": scan_ms, "fp32_fma_tflops": 2 * pair_elems / (scan_ms / 1e3) / 1e12 if scan_ms else None,
                     "peak_source": peaks["source"]},
        "family_ms_per_step": {kk: round(v[0], 4) for kk, v in sorted(fam.items(), key=lambda kv: -kv[1][0])},
        "gpu_launches": sum(v[1] for v in fam.values()) * args.steps,
        "parity_check": {"all_ranks_agree_bit_for_bit": agree}, "clocks": clocks,
    }
    if rank == 0:
        print(json.dumps(out))
    D.close()


# ================================================================================================ workload: train
def run_train(args):
    """BASELINE.json configs[3]: fine-tune step, ViT-L/14-336 + geocell head, 128 four-view samples per rank (1024 over 8 GPUs),
    bf16 tensor-core operands in the backward, haversine-smoothed CE, AdamW lr 2e-5, gradient averaging over NCCL."""
    from pigeon_b200 import CLIPVisionTower, SuperGuessr, VitDims, _lib, synthetic
    from pigeon_b200.training import AdamW
    D = Dist(args)
    world, rank, dev = D.world, D.rank, D.dev
    dims = VitDims()
    tower = CLIPVisionTower(dims)
    tower.load_state_dict(synthetic.random_vit_state_dict(dims, seed=0), strict=True)
    sg = SuperGuessr(tower, panorama=True, should_smooth_labels=True, num_candidates=5,
                     geocells=synthetic.synthetic_geocells(NUM_CELLS, 0)).to(dev)
    if not args.all_trainable:                      # reference freeze policy, models/super_guessr.py:159-160
        for p in sg.base_model.vision_model.encoder.layers[:-1].parameters():
            p.requires_grad = False
    sg.max_train_views = args.chunk_views
    sg.train()
    n_train = sum(p.numel() for p in sg.parameters() if p.requires_grad)
    opt = AdamW(sg.parameters(), lr=2e-5)
    B = args.train_batch
    torch.manual_seed(1234 + rank)
    px_host = torch.randn(B, 12, 336, 336).half().pin_memory()
    px = px_host.to(dev)
    labels = torch.tensor(synthetic.synthetic_geocells(B, 5 + rank))
    labels_clf = torch.randint(0, NUM_CELLS, (B,))

    def step_with(pixels):
        out = sg(pixel_values=pixels, labels=labels, labels_clf=labels_clf)
        sg.backward(out.loss)
        opt.step()
        opt.zero_grad()
        return out.loss

    sampler = ClockSampler(D.local)
    if rank == 0:
        sampler.start()
    ms, ms_by_rank, loss = D.timed(lambda: step_with(px), args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:      # the step's loss and a fixed sample of every parameter the optimizer updated
        params = {}
        for n, p in sg.named_parameters():
            if p.requires_grad:
                pick = torch.randperm(p.numel(), generator=torch.Generator().manual_seed(0))[:16384].sort().values
                params[n] = p.detach().reshape(-1)[pick.to(dev)].cpu()
        dump_outputs(args.dump_outputs, {"loss": loss.detach().cpu()} | params)
    ms_e2e, _, _ = D.timed(lambda: step_with(px_host.to(dev, non_blocking=True)).cpu(), max(1, min(args.steps, 2)), 1)
    lib = _lib.load()
    lib.pg_profile_begin()
    step_with(px)
    torch.cuda.synchronize()
    fam = read_profile()
    out = {
        "metric": "fine-tune samples/sec (four-view 336x336, ViT-L/14 + geocell head, forward + backward + AdamW)",
        "value": world * B * args.steps / (ms / 1e3), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16 forward / bf16 backward operands, fp32 accumulation and master weights", "data": "synthetic",
        "config": {"workload": f"fine-tune step, {B} four-view samples per GPU ({4 * B} views), "
                               f"{'all parameters' if args.all_trainable else 'reference freeze policy'} trainable "
                               f"({n_train / 1e6:.1f} M), chunks of {args.chunk_views} views; BASELINE.json configs[3] "
                               f"({world} x {B} = {world * B} samples)",
                   "parallelism": f"dp{world}", "grad_allreduce_bytes_per_step": 4 * n_train,
                   "collective": "none" if world == 1 else "NCCL all-reduce of the flat fp32 gradient, per-layer buckets on a side "
                                                           "stream overlapped with the backward of the last chunk"},
        "ms_per_step_by_rank": [m / args.steps for m in ms_by_rank],
        "e2e": {"value": world * B * max(1, min(args.steps, 2)) / (ms_e2e / 1e3), "unit": "samples/s",
                "h2d_bytes_per_step": px_host.numel() * 2, "d2h_bytes_per_step": 4},
        "loss": float(loss), "max_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30,
        "family_ms_per_step": {kk: round(v[0], 3) for kk, v in sorted(fam.items(), key=lambda kv: -kv[1][0])[:24]},
        "gpu_launches": sum(v[1] for v in fam.values()) * args.steps, "clocks": clocks,
    }
    if rank == 0:
        print(json.dumps(out))
    D.close()


# ================================================================================================ CPU arm
def cpu_port_images(n_images: int, threads: int):
    """The oracle (CPU port of the reference path) on `n_images` four-view images of the SAME configuration as the GPU arm
    (ViT-L/14-336, 1000 geocells, 100k-prototype bank, top-5 of 50 candidates); returns seconds."""
    from oracle import head as ohead, refiner as oref, vit as ovit
    from pigeon_b200 import synthetic
    from pigeon_b200.vit_engine import VitDims
    torch.set_num_threads(threads)
    dims = VitDims()
    sd = synthetic.random_vit_state_dict(dims, seed=0)
    cells = torch.from_numpy(synthetic.synthetic_geocells(NUM_CELLS, 0))
    lin = torch.nn.Linear(dims.hidden, NUM_CELLS)
    bank = _cpu_bank(dims.hidden)
    px = torch.randn(n_images * 4, 3, dims.image_size, dims.image_size, generator=torch.Generator().manual_seed(1))
    t0 = time.perf_counter()
    emb = ovit.clip_embedding(sd, px, patch=dims.patch_size, heads=dims.heads, layers=dims.layers, eps=dims.ln_eps)
    h = ohead.head_forward(emb.reshape(n_images, 4, -1), lin.weight.detach(), lin.bias.detach(), cells, NUM_CAND, True)
    oref.refiner_forward(bank, emb.reshape(n_images, 4, -1), h.pred_LLH, h.topk_idx, h.topk_val, TOPK, REFINER_T, REFINER_MAX_KM)
    return time.perf_counter() - t0


_CPU_BANK = None


def _cpu_bank(dim):
    global _CPU_BANK
    if _CPU_BANK is None:
        from pigeon_b200 import synthetic
        _CPU_BANK = synthetic.synthetic_bank(NUM_CELLS, NUM_PROTOS, dim, seed=2, empty_cells=5)
    return _CPU_BANK


def usable_cpus() -> int:
    """Host cores this process may really use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


_BEST_THREADS = None


def best_threads() -> int:
    """Thread count that maximises fp32 GEMM throughput of the oracle's dominant op on this host (a box that
    advertises more logical CPUs than it schedules runs slower with all of them); tried: powers of two up to the
    usable core count."""
    global _BEST_THREADS
    if _BEST_THREADS is None:
        n = usable_cpus()
        cands = sorted({c for c in (4, 8, 16, 32, 64, 128, 256, n) if c <= n} | {n})
        a, b = torch.randn(2308, 1024), torch.randn(1024, 4096)
        best, best_t = n, float("inf")
        for c in cands:
            torch.set_num_threads(c)
            a @ b
            t0 = time.perf_counter()
            for _ in range(3):
                a @ b
            dt = time.perf_counter() - t0
            if dt < best_t * 0.95:
                best, best_t = c, dt
        _BEST_THREADS = best
    return _BEST_THREADS


def cpu_baseline(sample_images: int):
    threads = best_threads()
    cpu_port_images(1, threads)                       # warm-up (thread pools, allocator, bank)
    sec = cpu_port_images(sample_images, threads)
    return {"value": sample_images / sec, "unit": "images/s", "cores": threads, "kind": "port",
            "sample": f"{sample_images} four-view images ({4 * sample_images} views) through the fp32 CPU oracle "
                      f"(ViT-L/14-336 + head + refiner over the same 100k-prototype bank), {sec:.1f} s, torch {torch.__version__} "
                      f"with {threads} threads (best of the thread counts tried; {usable_cpus()} usable logical CPUs)"}


def run_reference(args):
    """CPU arm: the oracle port of the reference path (the reference itself is Python under /root/reference and cannot travel to
    the GPU box).  Same model, geocells, bank size and candidate counts as the GPU arm; one step = ONE four-view image, a
    bounded sample of the 256-image batch (the per-image cost of the fp32 CPU path does not depend on the batch size)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = best_threads()
    for _ in range(min(args.warmup, 1)):
        cpu_port_images(1, threads)
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_port_images(1, threads)
    sec = time.perf_counter() - t0
    v = steps / sec
    sample = (f"{steps} steps x 1 four-view image (4 views) through the fp32 CPU oracle, {threads} threads "
              f"(best of the thread counts tried; {usable_cpus()} usable logical CPUs)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC,
        "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1),
        "ms_per_step": sec / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": "ViT-L/14-336 embed + geocell head (C=1000, top-50) + ProtoRefiner (P=100000, topk=5) on host "
                               "cores: the GPU arm's model, geocells and bank; each step is a bounded sample (1 four-view image) "
                               "of the 256-image batch of BASELINE.json configs[1]",
                   "same_config": "model / head / bank / candidate counts identical to the GPU arm; batch per step 1 instead of "
                                  "256 (bounded sample)"},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="infer", choices=["infer", "refiner", "train"])
    ap.add_argument("--batch", type=int, default=256, help="infer: four-view samples per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=4, help="four-view images in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-oracle-check", action="store_true", help="skip the 2-image CPU-oracle comparison of parity_check")
    ap.add_argument("--no-ln-fold", action="store_true", help="A/B: run the LayerNorm kernels instead of the folded epilogues")
    ap.add_argument("--replicated-bank", action="store_true", help="infer, N > 1: every rank holds the whole bank (A/B)")
    ap.add_argument("--refiner-topk", type=int, default=5)
    ap.add_argument("--refiner-schedule", type=int, default=0, choices=[0, 1, 2, 3, 4],
                    help="refiner scan: 0 automatic (slab scan at this shape), 1 query-major, 2 cell-major (round-1/2 kernel), 3 tile scan, 4 slab scan")
    ap.add_argument("--refiner-dim", type=int, default=768)
    ap.add_argument("--train-batch", type=int, default=128, help="train: four-view samples per GPU per step")
    ap.add_argument("--chunk-views", type=int, default=64)
    ap.add_argument("--all-trainable", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "refiner":
        run_refiner(args)
    elif args.workload == "train":
        run_train(args)
    else:
        run_infer(args)


if __name__ == "__main__":
    main()
