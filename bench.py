#!/usr/bin/env python
"""bench.py — masks/sec of the PSALM inference hot path (PSALM.eval_seg) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): COCO-panoptic prompt with 134 class names, 1024x1024 image,
100 queries, Swin-B + Phi-1.5, bf16 storage / fp32 accumulate, synthetic data and random-init weights
of that architecture (no checkpoint or dataset is reachable offline).  One step = eval_seg on one
batch of B images per GPU; masks/sec = images/sec x 100.  Default B = 4 (BASELINE.json configs[3] shards
32 images over 8 GPUs = 4 per GPU; configs[1] does not fix a batch size): the library GEMMs of the Phi
prefill run at M = 4 x 920 tokens instead of 920 and the step is 27 % cheaper per image than at B = 1
(measured: B = 1 / 2 / 4 / 8 -> 12.2 K / 15.0 K / 16.7 K / 16.9 K masks/s; `--batch 1` reproduces the
single-image latency of the reference's eval scripts, 8.2 ms).

  value : inputs (normalised image, sequence plan) already resident in HBM, device-timed (CUDA events),
          CUDA-graph replay of the network + task heads, includes the post-processing (and its one small D2H copy).
  batch1: the same arm at one image per step (the reference's eval scripts run batch 1).
  e2e   : the same metric through the public API call `PSALM.eval_seg(...)` with HOST (pinned) inputs: the
          uint8 image batch is uploaded on a copy stream (upload of step k+1 overlaps compute of step k) and
          normalised on the device; the results (panoptic id maps, class / score records, semantic arg-max) are
          read back, and at N > 1 the per-step all_gather of every rank's predictions over NVLink is inside too.
  roofline : the MSDeformAttn sampling kernel, timed with CUDA events around each of its launches
          inside K eager steps; algorithmic bytes per launch are stated in DESIGN.md; `traffic` is the DRAM
          traffic of one launch at this batch from the committed ncu capture (profiles/msda_traffic.json).
  roofline_extra : the other hot kernels, each against the roofline that bounds it (HBM or tensor).
  cpu_baseline : the CPU oracle port of the reference (oracle/psalm_oracle.py, validated bit-exact
          against the reference here) on the box's host cores, one image (rank 0, N=1 only).
  parity : the timed bf16 graph path (image 0 of the timed batch) and the fp32-storage path against that same
          oracle pass (same bf16-rounded weights): mask-logit errors, class arg-max agreement, task outputs.
  accuracy : PQ / mIoU / pixel agreement of the GPU outputs scored against the oracle's on held inputs
          (`--acc-images` per rank, accumulators all_reduced over ranks; oracle/accuracy.py).
  --impl reference : times that CPU port as the reference arm (the reference is Python and cannot
          travel to the box; its CUDA op has no CPU build — see DESIGN.md).
  --dump-outputs DIR : after the timed steps of the value arm, writes what its last step returned (rank 0) as
          DIR/<name>.npy, for an output-by-output comparison of two builds on the same (seeded) inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the bench leaves the source tree as it found it (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOAD = "coco-panoptic 1024x1024, 134 class names, 100 queries, Swin-B + Phi-1.5"
N_CLASSES, IMG = 134, 1024


def env_int(name, default):
    return int(os.environ.get(name, default))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


MSDA_KERNEL = "msda_encoder_fused_kernel"   # the L1-gather kernel (auto); the TMA-tile kernel (impl 3) is slower, DESIGN.md


def msda_traffic(B, dtype):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the MSDeformAttn kernel at the bench batch, from
    the committed `ncu --set full` capture of this command (profiles/; ncu cannot run inside a timed bench)."""
    p = os.path.join(ROOT, "profiles", "msda_traffic.json")
    if os.path.exists(p):
        d = json.load(open(p))
        e = d.get("%s_b%d" % (dtype, B))
        if e:
            return {"traffic": e["dram_bytes"], "traffic_source": e["source"]}
    return {"traffic": None, "traffic_source": "no ncu capture committed for this (dtype, batch)"}


def kernel_roofline(name, B, T_seq, esz):
    """Algorithmic bytes / flops per launch of the other hot kernels (DESIGN.md section 4) -> function us -> dict."""
    hbm, _ = peaks()
    tf = tensor_peak()

    def hbm_bound(nbytes):
        return lambda us: {"bound": "hbm", "algorithmic_bytes_per_launch": nbytes, "achieved": nbytes / us / 1e3,
                           "unit": "GB/s", "peak": hbm, "frac": nbytes / us / 1e3 / hbm}

    def tensor_bound(flops):
        return lambda us: {"bound": "tensor", "algorithmic_flops_per_launch": flops, "achieved": flops / us / 1e6,
                           "unit": "TFLOP/s", "peak": tf, "frac": flops / us / 1e6 / tf}
    if name.startswith("masked_cross_attention_"):
        hw = int(name.rsplit("_", 1)[1])
        return hbm_bound(B * (2 * hw * 256 * esz + 100 * hw // 8 + 2 * 100 * 256 * esz))
    if name == "mask_projection":
        return hbm_bound(B * (65536 * 256 * esz + 100 * 256 * esz + 100 * 65536 * esz))
    if name == "causal_attention":   # a contraction: QK^T + PV over the causal half, 32 heads x head_dim 64
        return tensor_bound(B * 32 * 2 * 2 * (T_seq * (T_seq + 1) // 2) * 64)
    if name.startswith("window_attention_stage"):
        st = int(name[-1])
        return hbm_bound(B * (65536 >> (2 * st)) * 4 * (128 << st) * esz)
    return None


def tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))
    return 1590.0


def msda_algorithmic_bytes(B, S=21504, M=8, D=32, L=3, P=4, e_val=2, e_ow=2):
    """Fused-kernel boundary (DESIGN.md): value read + raw offsets/logits read + output write."""
    return B * (e_val * S * M * D + e_ow * S * M * L * P * 3 + e_val * S * M * D)


# ------------------------------------------------------------------------------------------------
PIXEL_MEAN = (123.675, 116.28, 103.53)   # datasets_mapper/coco_panoptic_mapper.py:118-119
PIXEL_STD = (58.395, 57.12, 57.375)


def bench_inputs(batch, seed):
    """The bench request: synth_inputs' prompt + a uint8 RGB image per sample (what exists before the mapper's
    normalisation) and the float image the reference's eval_seg receives, (u8 - mean) / std computed on the host
    in fp32 exactly like the mapper (coco_panoptic_mapper.py:161)."""
    from psalm_b200 import synth
    inp = synth.synth_inputs(batch=batch, height=IMG, width=IMG, task="panoptic", n_classes=N_CLASSES, seed=seed)
    mean = torch.tensor(PIXEL_MEAN).view(1, 3, 1, 1)
    std = torch.tensor(PIXEL_STD).view(1, 3, 1, 1)
    # uint8 pixels with the statistics the mapper's normalisation expects: the N(0, 1) synthetic image, de-normalised,
    # rounded and clamped to [0, 255]
    u8 = (inp["images"] * std + mean).round().clamp(0, 255).to(torch.uint8)
    inp["images_u8"] = u8
    inp["images"] = (u8 - mean) / std
    return inp


def bench_weights(cfg, dtype):
    """CPU-generated (bit-reproducible on every box) weights, rounded to the storage type: the GPU model and the
    CPU oracle legs consume exactly the same values."""
    from psalm_b200 import synth
    sd = synth.synth_state_dict(cfg, seed=0)
    if dtype != torch.float32:
        sd = {k: (v.to(dtype).float() if v.is_floating_point() else v) for k, v in sd.items()}
    return sd


def oracle_eval(sd, inp, b, threads, relaxed=False, intermediates=True):
    """CPU oracle (port of the reference path) on sample b of `inp`; returns (seconds, results, intermediates)."""
    from oracle import psalm_oracle as O
    torch.set_num_threads(threads)
    sl = slice(b, b + 1)
    with torch.no_grad():
        t0 = time.perf_counter()
        out = O.eval_seg(sd, inp["input_ids"][sl], inp["attention_mask"][sl], inp["images"][sl], inp["seg_info"][sl],
                         class_name_ids=inp["class_name_ids"][sl], cls_indices=inp["cls_indices"][sl],
                         class_name_embedding_indices=inp["class_name_embedding_indices"][sl],
                         is_thing_list=inp["is_thing_list"], task="panoptic", return_intermediates=intermediates,
                         obj_thr=0.0 if relaxed else 0.8, ovl_thr=0.0 if relaxed else 0.8)
        dt = time.perf_counter() - t0
    return (dt,) + (tuple(out) if intermediates else (out, None))


def cpu_threads():
    # all host cores the port can use productively: measured on the 128-core box, 16-32 threads are fastest
    # (9.1 s / image), 64 threads 15.5 s, 128 threads 198 s (oversubscribed small ops)
    return min(32, os.cpu_count())


def run_reference(args, rank, world):
    if rank != 0:
        return
    from psalm_b200.layout import PsalmConfig
    K, W = args.steps, args.warmup
    t0 = time.perf_counter()
    threads = cpu_threads()
    sd = bench_weights(PsalmConfig(), torch.float32)
    inp = bench_inputs(1, 1)
    times = [oracle_eval(sd, inp, 0, threads, intermediates=False)[0] for _ in range(W + K)]
    timed = times[W:]
    sec = sum(timed) / len(timed)
    val = 100.0 / sec
    line = {"impl": "reference", "metric": "masks/sec", "value": val, "unit": "masks/s", "n_gpus": args.gpus,
            "steps": len(timed), "warmup": W, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": args.batch, "images_per_step": 1,
                       "note": "bounded sample: each step is ONE image of the batch (masks/s is per image); "
                       "CPU port of the reference path "
                       "(oracle/psalm_oracle.py, bit-exact vs the reference in the build container); "
                       "Swin evaluated once (the reference evaluates it twice)"},
            "cpu_baseline": {"value": val, "unit": "masks/s", "cores": threads, "kind": "port",
                             "sample": "%d x one 1024^2 panoptic image, fp32" % len(timed)},
            "e2e": {"value": val, "unit": "masks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def timed_device_steps(step, K, W, barrier):
    """(milliseconds of K timed steps after W warm-up steps, what the last timed step returned)"""
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(K):
        last = step()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    return e0.elapsed_time(e1), last


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(results, image_hw, n_queries, out_dir, seed=0):
    """Write what one step returned (PSALM.post_process: per image sem_seg [C,H,W], instances, panoptic_seg) to
    out_dir/<name>.npy.  Every shape depends only on the batch B, the class count C and the query count Q, never on
    the values, so that two builds run with the same arguments write arrays of the same shapes:
      pixel_yx [N,2]: a fixed, seeded sample of N pixels, N chosen to keep the files under DUMP_BYTES;
      panoptic_seg [B,N]: segment id at each sampled pixel;
      panoptic_segments [B,Q,3]: row k = (id, isthing, category_id) of segment id k + 1, -1 where there is none;
      sem_seg [B,C,N];
      instances [B,Q,3]: (score, pred_class, query_index) of each kept instance, then -1 rows;
      instance_masks [B,Q,N]: the masks of those instances at the sampled pixels, then zero rows."""
    H, W = image_hw
    B, C, Q = len(results), results[0]["sem_seg"].shape[0], n_queries
    n = min(H * W, (DUMP_BYTES - 4 * 10 ** 6) // (4 * B * (1 + C + Q)))
    pix = torch.from_numpy(np.sort(np.random.default_rng(seed).choice(H * W, n, replace=False)))
    dev_pix = pix.to(results[0]["sem_seg"].device)
    segments = np.full((B, Q, 3), -1.0)
    inst = np.full((B, Q, 3), -1.0)
    inst_masks = np.zeros((B, Q, n), dtype=np.float32)
    for b, r in enumerate(results):
        for s in r["panoptic_seg"][1]:                 # ids are 1 .. number of segments <= Q
            segments[b, s["id"] - 1] = (s["id"], s["isthing"], s["category_id"])
        i = r["instances"]
        k = len(i.scores)                              # <= Q: the top-k of the task heads keeps at most Q
        inst[b, :k] = torch.stack([i.scores.float(), i.pred_classes.float(), i.query_index.float()], 1).cpu().numpy()
        inst_masks[b, :k] = i.pred_masks.flatten(1)[:, dev_pix].float().cpu().numpy()
    arrays = {
        "pixel_yx": np.stack([pix.numpy() // W, pix.numpy() % W], 1).astype(np.float64),
        "panoptic_seg": torch.stack([r["panoptic_seg"][0].flatten()[dev_pix] for r in results]).float().cpu().numpy(),
        "panoptic_segments": segments,
        "sem_seg": torch.stack([r["sem_seg"].flatten(1)[:, dev_pix] for r in results]).float().cpu().numpy(),
        "instances": inst,
        "instance_masks": inst_masks,
    }
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from psalm_b200 import dist as PD
    from psalm_b200 import kernels
    from psalm_b200.layout import PsalmConfig
    from psalm_b200.psalm import PSALM
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    K, W, B = args.steps, max(args.warmup, 3), args.batch
    cfg = PsalmConfig()
    dtype = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}[args.dtype]
    wall0 = time.perf_counter()
    sd = bench_weights(cfg, dtype)                       # CPU, storage-rounded: the oracle legs use the same values
    model = PSALM(sd, cfg, dtype, dev, "panoptic", use_cuda_graph=not args.no_graph)
    inp = bench_inputs(B, 1 + rank)
    kw = {k: inp[k] for k in ("class_name_ids", "cls_indices", "class_name_embedding_indices", "is_thing_list")}
    images_u8_h = inp["images_u8"].pin_memory()
    model.is_thing_list = inp["is_thing_list"]

    def barrier():
        if world > 1:
            dist.barrier()

    # ---------------- device-resident arm (value) ----------------
    images_d = inp["images"].to(dev)
    plan_d = model.make_plan(inp["input_ids"], inp["attention_mask"], (IMG, IMG), inp["class_name_ids"],
                             inp["cls_indices"], inp["class_name_embedding_indices"]).to(dev)

    def step_device():
        out = model.forward_core(images_d, plan_d) if args.no_graph else model.forward_core_graphed(images_d, plan_d)
        return model.post_process(out, (IMG, IMG), inp["seg_info"])

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_total, last = timed_device_steps(step_device, K, W, barrier)
    if args.dump_outputs and rank == 0:
        dump_outputs(last, (IMG, IMG), model.num_queries, args.dump_outputs)
    del last
    # outputs of the timed configuration (graph replay at batch B), kept for the parity / accuracy checks below
    out_timed = None
    if not args.no_graph:
        g_out = model.forward_core_graphed(images_d, plan_d)
        out_timed = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in g_out.items() if k != "post"}

    # single-image latency of the same build (the reference's eval scripts run batch 1, panoptic_segmentation.py:57)
    b1 = None
    if B != 1 and not args.no_batch1:
        img1, plan1 = images_d[:1].contiguous(), model.make_plan(
            inp["input_ids"][:1], inp["attention_mask"][:1], (IMG, IMG), inp["class_name_ids"][:1],
            inp["cls_indices"][:1], inp["class_name_embedding_indices"][:1]).to(dev)

        def step_b1():
            out = model.forward_core(img1, plan1) if args.no_graph else model.forward_core_graphed(img1, plan1)
            return model.post_process(out, (IMG, IMG), inp["seg_info"][:1])
        ms1 = PD.max_over_ranks([timed_device_steps(step_b1, K, W, barrier)[0]], dev)[0]
        b1 = {"value": K * world * 100.0 / (ms1 / 1e3), "unit": "masks/s", "ms_per_image": ms1 / K, "batch_per_gpu": 1}

    # the reference's real eval flow (coco_panoptic_mapper.py:148-162): a 640 x 480 image resized to 1024 x 768, padded to
    # 1024^2 with a padding mask, outputs at the original size - the composed fused task-head kernel (crop + resize)
    mflow = None
    if not args.no_graph and not args.no_batch1:
        pmask = torch.zeros(IMG, IMG, dtype=torch.bool)
        pmask[768:, :] = True
        seg_m = [dict(padding_mask=pmask, height=480, width=640) for _ in range(B)]
        fused_m, boxes_m = model._fused_applies((IMG, IMG), seg_m)

        def step_mapper():
            out = model.forward_core_graphed(images_d, plan_d, fuse_post=fused_m)
            return model.post_process(out, (IMG, IMG), seg_m, boxes_m)
        msm = PD.max_over_ranks([timed_device_steps(step_mapper, K, W, barrier)[0]], dev)[0]
        mflow = {"value": K * B * world * 100.0 / (msm / 1e3), "unit": "masks/s", "ms_per_step": msm / K,
                 "fused_task_heads": bool(fused_m), "geometry": "1024x768 valid region of the padded 1024^2 input -> 480x640 outputs"}

    # roofline leg: the same K steps launched eagerly (a CUDA graph cannot carry timing events), with
    # CUDA events on the launch stream around every hot-kernel launch; also counts our launches per step
    def step_eager():
        # eager launches are CPU bound (~30 ms of Python per image vs ~6 ms of GPU work): park the GPU on a
        # ~40 ms spin first so that every kernel of the step is already queued when it runs and the event
        # pairs below measure device time, not launch gaps
        torch.cuda._sleep(80_000_000)
        out = model.forward_core(images_d, plan_d)
        return model.post_process(out, (IMG, IMG), inp["seg_info"])
    overlap_keep = model.overlap_branches
    model.overlap_branches = False     # per-kernel rooflines: every kernel timed alone, not under the other branch
    step_eager()
    kernels.PROFILE_EVENTS = {}
    l0 = kernels.launches()
    for _ in range(K):
        step_eager()
    torch.cuda.synchronize()
    launches = kernels.launches() - l0
    ev = kernels.PROFILE_EVENTS
    kernels.PROFILE_EVENTS = None
    model.overlap_branches = overlap_keep
    msda_us = [a.elapsed_time(b) * 1e3 for a, b in ev.get("msda", [])]
    esz_ = 4 if dtype == torch.float32 else 2
    T_seq = int(plan_d.T)
    extra = []
    for name, pairs in sorted(ev.items()):
        if name == "msda":
            continue
        us = sum(a.elapsed_time(b) for a, b in pairs) * 1e3 / len(pairs)
        rf = kernel_roofline(name, B, T_seq, esz_)
        if rf is None:
            continue
        extra.append(dict(kernel=name, avg_us=us, launches_timed=len(pairs), **rf(us)))
    clocks = sampler.stop()

    # ---------------- end-to-end arm (host buffers through the public API) ----------------
    # per step: uint8 image batch uploaded from pinned memory on the copy stream (the upload of step k+1 overlaps the
    # compute of step k), normalisation on the device, eval_seg, results read back to the host, and (N > 1) the
    # all_gather of every rank's predictions - all inside the timed region
    # Pipelined through the public async API: batch k+1 is submitted (lane (k+1) % 2) before batch k is finished, and
    # the finish work of k (host merge of the panoptic rule, id maps, packing, all_gather, read-back into pinned
    # buffers) runs on a side stream under the device work of k+1.  Every batch is fully read back; the clock
    # stops after the last one.
    post_stream = torch.cuda.Stream(device=dev)
    pins = {}

    def to_pinned(name, t):
        buf = pins.get(name)
        if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
            buf = pins[name] = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        buf.copy_(t, non_blocking=True)
        return buf

    def submit(k, staged):
        return model.eval_seg_async(input_ids=inp["input_ids"], attention_mask=inp["attention_mask"], images=staged,
                                    seg_info=inp["seg_info"], lane=k % 2, **kw)

    def finish(pending):
        with torch.cuda.stream(post_stream):
            res = pending.result()
            meta, maps = PD.pack_predictions(res, model.num_queries)
            gmeta, gmaps = PD.gather_predictions(meta, maps)      # NCCL all_gather over NVLink (no-op at N = 1)
            host = [to_pinned("meta", gmeta), to_pinned("maps", gmaps)]
            sem = torch.stack([r["sem_seg"].argmax(0).to(torch.uint8) for r in res])
            host.append(to_pinned("sem", sem))
        post_stream.synchronize()
        return host

    def run_e2e(n):
        host = None
        pend = submit(0, model.stage_images(images_u8_h))
        for k in range(n):
            nxt = submit(k + 1, model.stage_images(images_u8_h)) if k + 1 < n else None
            host = finish(pend)
            pend = nxt
        return host

    def run_e2e_sync(n):     # the blocking call, one batch at a time (what round 1 reported as e2e)
        host = None
        nxt = model.stage_images(images_u8_h)
        for k in range(n):
            cur = nxt
            if k + 1 < n:
                nxt = model.stage_images(images_u8_h)
            res = model.eval_seg(input_ids=inp["input_ids"], attention_mask=inp["attention_mask"], images=cur,
                                 seg_info=inp["seg_info"], **kw)
            meta, maps = PD.pack_predictions(res, model.num_queries)
            gmeta, gmaps = PD.gather_predictions(meta, maps)
            host = [to_pinned("meta", gmeta), to_pinned("maps", gmaps),
                    to_pinned("sem", torch.stack([r["sem_seg"].argmax(0).to(torch.uint8) for r in res]))]
            torch.cuda.synchronize()
        return host

    def timed_wall(fn):
        fn(3)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        host = fn(K)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        return host, dt

    host, e2e_sync_s = timed_wall(run_e2e_sync)
    host, e2e_s = timed_wall(run_e2e)
    h2d = images_u8_h.numel() * images_u8_h.element_size()
    d2h = sum(t.numel() * t.element_size() for t in host)
    nvlink = 0 if world == 1 else (host[0].numel() * 4 + host[1].numel() * 4)
    ms_total, e2e_ms, e2e_sync_ms = PD.max_over_ranks([ms_total, e2e_s * 1e3, e2e_sync_s * 1e3], dev)

    # ---------------- parity + accuracy vs the CPU oracle (checker only; outside every timed region) -------------
    parity_line = accuracy_line = cpu_line = None
    if not args.no_oracle and out_timed is not None:
        from oracle import accuracy, parity
        threads = cpu_threads() if world == 1 else max(4, min(32, os.cpu_count() // world))
        acc = accuracy.Accumulator(N_CLASSES)
        # panoptic thresholds 0.0 / 0.0 in BOTH arms for the task-output comparison: the reference's hard-coded
        # 0.8 / 0.8 (llava_phi.py:331-332) leaves no segment on random weights (oracle/accuracy.py)
        model.object_mask_threshold = model.overlap_threshold = 0.0
        res_relaxed = model.eval_seg(input_ids=inp["input_ids"], attention_mask=inp["attention_mask"],
                                     images=images_d, seg_info=inp["seg_info"], **kw)
        H4, W4 = out_timed["mask_size"]
        it0 = None
        n_acc = args.acc_images if args.acc_images > 0 else max(2, 16 // world)    # 16 images over the ranks by default
        cur_inp, cur_res, cur_masks = inp, res_relaxed, out_timed["pred_masks"]
        for n in range(n_acc):
            b = n % B
            if n > 0 and b == 0:   # a further batch of held images, through the timed graph path
                fresh = bench_inputs(B, 1000 + 17 * rank + n)
                cur_inp = dict(inp, images=fresh["images"], images_u8=fresh["images_u8"])      # same prompt, new images
                cur_res = model.eval_seg(input_ids=cur_inp["input_ids"], attention_mask=cur_inp["attention_mask"],
                                         images=cur_inp["images"].to(dev), seg_info=cur_inp["seg_info"], **kw)
                cur_res = [dict(panoptic_seg=(r["panoptic_seg"][0].clone(), r["panoptic_seg"][1]), sem_arg=r["sem_seg"].argmax(0).cpu())
                           for r in cur_res]
                cur_masks = model.forward_core_graphed(cur_inp["images"].to(dev), plan_d)["pred_masks"].clone()
            dt, ores, it = oracle_eval(sd, cur_inp, b, threads, relaxed=True)
            if n == 0:
                it0 = it
                cpu_line = {"value": 100.0 / dt, "unit": "masks/s", "cores": threads, "kind": "port",
                            "sample": "one 1024^2 panoptic image, fp32, single pass, no warm-up"}
                one = {k: (v[:1] if torch.is_tensor(v) else v) for k, v in out_timed.items()}
                parity_line = {"bf16_graph_path": dict(parity.final_metrics(one, it),
                                                       **parity.result_metrics(res_relaxed[:1], ores, "panoptic")),
                               "bf16_stages_teacher_forced_l2rel": parity.forced_stage_errors(model, it, inp["images"][:1]),
                               "bf16_decoder_layers_teacher_forced": parity.forced_layer_errors(model, it),
                               "oracle_decoder_sensitivity_to_bf16_inputs": parity.predictor_sensitivity(sd, it, torch.bfloat16),
                               "note": "image 0 of the timed batch vs the CPU oracle on the same bf16-rounded weights; task "
                                       "outputs compared at panoptic thresholds 0.0 / 0.0 in both arms; teacher-forced = every "
                                       "stage / decoder layer fed the oracle's inputs; sensitivity = the ORACLE's decoder "
                                       "re-run on its own inputs rounded to bf16 (the masked attention thresholds mask "
                                       "logits: a discontinuity of the reference itself)"}
            r, o = cur_res[b], ores[0]
            acc.add_panoptic(r["panoptic_seg"][0].cpu().numpy(), r["panoptic_seg"][1], o["panoptic_seg"][0].numpy(),
                             o["panoptic_seg"][1])
            sem_arg = r["sem_arg"] if "sem_arg" in r else r["sem_seg"].argmax(0).cpu()
            acc.add_semantic(sem_arg.numpy(), o["sem_seg"].argmax(0).numpy())
            up = torch.nn.functional.interpolate(cur_masks[b].float().view(1, -1, H4, W4), size=(IMG, IMG),
                                                 mode="bilinear", align_corners=False)[0]
            acc.add_masks((up > 0).cpu(), it["mask_pred"][0] > 0)
            acc.add_image()
            del up
        model.object_mask_threshold, model.overlap_threshold = cfg.mask.object_mask_threshold, cfg.mask.overlap_threshold
        acc.load(*PD.reduce_sum(acc.tensors(), dev))
        accuracy_line = dict(acc.report(), reference="CPU oracle outputs on the same held inputs and weights",
                             thresholds="object 0.0 / overlap 0.0 in both arms")
        # fp32 storage path (the north-star tolerance) on the same weights and image, rank 0 at N = 1
        if rank == 0 and world == 1 and not args.no_fp32_parity:
            del model, res_relaxed
            torch.cuda.empty_cache()
            m32 = PSALM(sd, cfg, torch.float32, dev, "panoptic")
            p1 = m32.make_plan(inp["input_ids"][:1], inp["attention_mask"][:1], (IMG, IMG), inp["class_name_ids"][:1],
                               inp["cls_indices"][:1], inp["class_name_embedding_indices"][:1]).to(dev)
            parity_line["fp32_path"] = parity.final_metrics(m32.forward_core(images_d[:1].contiguous(), p1), it0)
            del m32
    if rank != 0:
        return
    images_total = K * B * world
    value = images_total * 100.0 / (ms_total / 1e3)
    e2e_value = images_total * 100.0 / (e2e_ms / 1e3)
    hbm, peak_src = peaks()
    esz = 4 if dtype == torch.float32 else 2
    alg = msda_algorithmic_bytes(B, e_val=esz, e_ow=esz)
    avg_us = sum(msda_us) / max(1, len(msda_us))
    achieved = alg / avg_us / 1e3 if avg_us > 0 else 0.0
    line = {"metric": "masks/sec", "value": value, "unit": "masks/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "images_per_step": B * world, "parallelism": "dp%d" % world,
                       "l2": "inputs larger than L2 (3.2 GB of weights are streamed every step)",
                       "timed": "Swin (once) + projector + Phi prefill + pixel decoder + masked decoder + post-processing",
                       "cuda_graph": not args.no_graph,
                       "weights": "synthetic, generated on the CPU (bit-reproducible), rounded to the storage type",
                       "e2e_input": "uint8 [B,3,1024,1024] from pinned host memory, normalised on the device; upload of "
                                    "step k+1 overlaps compute of step k; results + (N>1) prediction all_gather inside"},
            "e2e": {"value": e2e_value, "unit": "masks/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / K, "nvlink_gather_bytes_per_step": int(nvlink),
                    "api": "PSALM.eval_seg_async, two lanes: batch k is finished (host merge, gather, read-back to pinned "
                           "memory) under the device work of batch k+1",
                    "blocking_call": {"value": images_total * 100.0 / (e2e_sync_ms / 1e3), "ms_per_step": e2e_sync_ms / K,
                                      "api": "PSALM.eval_seg, one batch at a time"}},
            "gpu_launches": int(launches), "gpu_launches_per_step": int(launches // K),
            "clocks": clocks,
            "roofline": dict({"kernel": MSDA_KERNEL, "bound": "hbm", "achieved": achieved, "peak": hbm,
                              "unit": "GB/s", "frac": achieved / hbm, "peak_source": peak_src,
                              "avg_us": avg_us, "launches_timed": len(msda_us), "algorithmic_bytes_per_launch": alg,
                              "timed_in": "K eager steps of the same workload, CUDA events on the launch stream"},
                             **msda_traffic(B, args.dtype)),
            "roofline_extra": extra,
            "wall_s": time.perf_counter() - wall0}
    if b1 is not None:
        line["batch1"] = b1
    if mflow is not None:
        line["mapper_flow"] = mflow
    if parity_line is not None:
        line["parity"] = parity_line
    if accuracy_line is not None:
        line["accuracy"] = accuracy_line
    if cpu_line is not None and world == 1:
        line["cpu_baseline"] = cpu_line
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4, help="images per GPU per step (1 = single-image latency)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f16", "f32"])
    ap.add_argument("--no-oracle", action="store_true", help="skip the CPU-oracle legs (cpu_baseline, parity, accuracy)")
    ap.add_argument("--no-fp32-parity", action="store_true", help="skip the fp32-storage parity pass (N = 1)")
    ap.add_argument("--no-batch1", action="store_true", help="skip the single-image latency measurement")
    ap.add_argument("--acc-images", type=int, default=0,
                    help="held images per rank scored against the oracle (0 = 16 images divided over the ranks, at least 2)")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
