#!/usr/bin/env python
"""bench.py — story-turns/sec of the SEED-Story interleaved inference hot path on B200 (contract in the task brief).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config story|sink|sdxl] [--stories-per-gpu S]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

--config story (default; BASELINE.json configs[1], and configs[2] when launched on N GPUs): a *step* is one 10-turn
synthetic StoryStream-shaped story per GPU: start image 448x448, 64-token caption, each turn = 64 greedy text tokens +
forced <img>, 64 image queries, </img>, EOS, then one SDXL 1024x1024 image (Euler, 50 steps, CFG 7.5, seed 42) decoded
by the VAE; window of 8 images.  Stories are independent, so N GPUs run N stories data-parallel with no data-path
collective ("scaling": "weak").
--config sink  (configs[3]): 25-turn stories in LIVE multimodal attention-sink mode (paged KV kept across turns, sink
retention at every eviction); --stories-per-gpu 4 runs four stories per GPU with their MLLM decode steps batched over
the paged KV cache (continuous batching; a step is then 4 stories, `value` still counts story-turns).
--config sdxl  (configs[4]): a step is one SDXL de-tokenizer image (30 Euler steps, CFG, VAE decode) per GPU from a
256x4096 image-feature tensor; metric = images/s.

  value : metric with the inputs already on the device, results left on the device
  e2e   : the same steps through the reference-facing API (src.* drop-ins) from HOST buffers: pinned inputs copied H2D
          inside the timed region, every turn's token ids and 1024x1024 uint8 image copied D2H (bounded to --e2e-steps,
          default 6, of the same steps so that the default run stays within minutes)
  roofline            : the dominant kernel family (tcgen05 GEMM / implicit-GEMM conv of the UNet): every launch type of
                        one UNet step timed live as 10 back-to-back launches in a CUDA graph (CUDA events), weighted by
                        its count; peak = BURST bf16 (kernels timed in isolation)
  roofline_whole_step : all algorithmic flops of a UNet CFG step (GEMM + conv + attention) / its graph-replay time,
                        against the SUSTAINED bf16 peak (timed inside a long step)
  roofline_decode     : weight + KV bytes of one Llama decode step / its graph-replay time, against the HBM peak
  gpu_eager_baseline  : the oracle (torch restatement of the reference path) in fp16 eager PyTorch on the same GPU
                        (cuBLAS / cuDNN / SDPA, unmerged LoRA, python greedy loop with .item(), fp32 VAE, zero-image ViT
                        per turn): the "reference fp16 GPU path" of BASELINE.md section 3, as a bounded sample
  cpu_baseline        : the oracle in fp32 on the host cores, bounded sample (see cpu_reference_step)
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "seed-story_b200"), os.path.join(ROOT, "seed-story_b200", "shims")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

TURNS = 10
DENOISE_STEPS = 50
N_TEXT, N_RUN = 64, 67                 # free text tokens; <img> + 64 queries + </img> + EOS
TOKENS_PER_TURN = N_TEXT + N_RUN       # 131 decoded positions per turn in the reference's token-by-token loop
MEAN_PROMPT = 716                      # mean prompt length over the 10 turns (131 + 130 (t-1), window 8)
METRICS = dict(story="story-turns/sec (text+image) at 10-turn seq", sink="story-turns/sec (text+image) at 25-turn seq, live attention sink",
               sdxl="SDXL 1024^2 img/s")


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows, self.stop_flag, self.index = [], False, index
        self.t = None

    def start(self):
        def run():
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            while not self.stop_flag:
                try:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                    self.rows.append([c.strip() for c in out.stdout.strip().split(",")])
                except Exception:
                    pass
                time.sleep(0.5)
        self.t = threading.Thread(target=run, daemon=True)
        self.t.start()

    def stop(self):
        self.stop_flag = True
        if self.t:
            self.t.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None, reasons=reasons, samples=len(sm))


def synthetic_story(s, vocab_text=32000):
    """seed 1000+s: uniform-random uint8 448x448x3 image through the CLIP transform, 64 caption ids in [3, 32000)."""
    g = torch.Generator().manual_seed(1000 + s)
    img = torch.randint(0, 256, (3, 448, 448), generator=g, dtype=torch.uint8).float() / 255.0
    mean = torch.tensor([0.48145466, 0.4578275, 0.40821073]).view(3, 1, 1)
    std = torch.tensor([0.26862954, 0.26130258, 0.27577711]).view(3, 1, 1)
    img = ((img - mean) / std).half().unsqueeze(0)
    cap = torch.randint(3, vocab_text, (64,), generator=g).tolist()
    return img, cap


def ev():
    return torch.cuda.Event(enable_timing=True)


DUMP_BYTES = 60 * 10 ** 6     # payload bound of --dump-outputs (the .npy headers stay far inside 64 MB)


def dump_outputs(outdir, last):
    """--dump-outputs: what the last timed step returned to its caller, as float32 .npy files in `outdir`.
      generate_ids.npy [n, L]    every turn's generated ids (stories in order, then turns), padded with -1
      has_img_output.npy [n]     1 where the turn produced an image
      images.npy [m, K]          the m uint8 1024x1024x3 images, flattened; all of each image when they fit the bound,
                                 else the same K positions of each (torch.randperm, seed 0), listed in image_index.npy
    The bench inputs and weights are seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    turns = last.get("turns", [])
    images = last.get("images", [o["image"] for o in turns if o["image"] is not None])
    arrays = {}
    if turns:
        width = max(len(o["generate_ids"]) for o in turns)
        ids = np.full((len(turns), width), -1, np.float32)
        for r, o in enumerate(turns):
            ids[r, :len(o["generate_ids"])] = o["generate_ids"]
        arrays["generate_ids"] = ids
        arrays["has_img_output"] = np.array([o["has_img_output"] for o in turns], np.float32)
    if images:
        numel = images[0].numel()
        room = (DUMP_BYTES - sum(a.nbytes for a in arrays.values())) // 4
        flat = [im.reshape(-1) for im in images]
        if numel * len(images) <= room:
            arrays["images"] = torch.stack(flat).float().cpu().numpy()
        else:
            k = room // (len(images) + 1)
            idx = torch.randperm(numel, generator=torch.Generator().manual_seed(0))[:k].sort().values
            idx_dev = idx.to(images[0].device)
            arrays["images"] = torch.stack([f[idx_dev] for f in flat]).float().cpu().numpy()
            arrays["image_index"] = idx.float().numpy()      # exact: numel < 2^24
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from seedstory import _capi, ops, story
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    ops.require_device()
    pipe = story.StoryPipeline(device=dev, cfg=story.FULL, num_inference_steps=args.denoise_steps, verbose=(rank == 0))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(n):
        if world == 1:
            return n
        t = torch.tensor([n], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    n_steps_total = args.warmup + args.steps
    host_img = torch.empty((1024, 1024, 3), dtype=torch.uint8).pin_memory()
    counters = dict(h2d=0, d2h=0)
    last = {}      # what the last timed step returned, kept for --dump-outputs

    def keep(i):
        return args.dump_outputs is not None and i == n_steps_total - 1

    if args.config in ("story", "sink"):
        turns, sink, spg = args.turns, args.config == "sink", max(1, args.stories_per_gpu)
        # step i of this rank = stories i*spg .. i*spg+spg-1 (spg > 1: their MLLM decode steps are batched, configs[3])
        inputs = [synthetic_story(rank * 1000 + i) for i in range(n_steps_total * spg)]
        dev_inputs = [(im.to(dev), cap) for im, cap in inputs]
        pinned = [(im.pin_memory(), cap) for im, cap in inputs]

        def run(ims, caps, **kw):
            if spg == 1:
                return [pipe.run_story(ims[0], caps[0], turns, sink=sink, **kw)]
            return pipe.run_stories(ims, caps, turns, sink=sink, **kw)

        def step_dev(i):
            grp = dev_inputs[i * spg:(i + 1) * spg]
            outs = run([g[0] for g in grp], [g[1] for g in grp], return_images=keep(i))
            if keep(i):
                last["turns"] = [o for st in outs for o in st]
            return sum(1 for st in outs for o in st if o["has_img_output"])   # a story ends early if a turn emits no image

        def step_e2e(i):
            ims, caps = [], []
            for im_host, cap in pinned[i * spg:(i + 1) * spg]:
                ims.append(im_host.to(dev, non_blocking=True))
                cap_dev = torch.tensor(cap, dtype=torch.int32).pin_memory().to(dev, non_blocking=True)   # ids travel too
                counters["h2d"] += im_host.numel() * 2 + cap_dev.numel() * 4
                caps.append(cap)
            n = 0
            for st in run(ims, caps, return_images=True):
                for o in st:
                    if not o["has_img_output"]:
                        continue
                    n += 1
                    host_img.copy_(o["image"], non_blocking=True)
                    counters["d2h"] += host_img.numel() + len(o["generate_ids"]) * 8
            torch.cuda.current_stream().synchronize()
            return n
        unit = "story-turns/s"
    else:   # sdxl standalone: one image per step from a [1, 256, 4096] image-feature tensor (what the MLLM hands over)
        g = torch.Generator().manual_seed(77 + rank)
        feats = [(torch.randn(1, 256, 4096, generator=g) * 0.5).half() for _ in range(n_steps_total)]
        dev_feats = [f.to(dev) for f in feats]
        pinned_feats = [f.pin_memory() for f in feats]

        def sdxl_image(feat):
            return pipe.adapter.generate(image_embeds=feat, num_inference_steps=args.denoise_steps, height=1024, width=1024,
                                         output_type="pt", input_image_size=448)[0]

        def step_dev(i):
            img = sdxl_image(dev_feats[i])
            if keep(i):
                last["images"] = [img]
            return 1

        def step_e2e(i):
            f = pinned_feats[i].to(dev, non_blocking=True)
            counters["h2d"] += f.numel() * 2
            host_img.copy_(sdxl_image(f), non_blocking=True)
            counters["d2h"] += host_img.numel()
            torch.cuda.current_stream().synchronize()
            return 1
        unit = "img/s"

    # ---- value: device-resident inputs -----------------------------------------------------------
    for i in range(args.warmup):
        step_dev(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    c0 = _capi.launch_count()
    e0, e1 = ev(), ev()
    n_units = 0
    e0.record()
    for i in range(args.warmup, n_steps_total):
        n_units += step_dev(i)
    e1.record()
    barrier()
    launches = _capi.launch_count() - c0
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    value = sum_over_ranks(n_units) / (ms * 1e-3)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()

    # ---- e2e: host buffers, H2D + D2H inside the timed region --------------------------------------
    # (same steps, same inputs; bounded to args.e2e_steps of them so the whole default run stays within minutes)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    step_e2e(args.warmup)   # warm the path (pinned allocations)
    counters["h2d"] = counters["d2h"] = 0
    n_units_e2e = 0
    barrier()
    e0.record()
    for i in range(args.warmup, args.warmup + e2e_steps):
        n_units_e2e += step_e2e(i)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = sum_over_ranks(n_units_e2e) / (ms_e2e * 1e-3)

    extra = {}
    if rank == 0:
        peaks = load_peaks()
        extra.update(measure_rooflines(pipe, dev, peaks, args))
        if world == 1:
            if not args.no_eager_baseline:
                try:
                    extra["gpu_eager_baseline"] = gpu_eager_baseline(dev, args)
                except Exception as e:   # a baseline must never take the bench line down
                    import traceback
                    traceback.print_exc()
                    extra["gpu_eager_baseline"] = dict(error=repr(e)[:300])
            if not args.no_cpu_baseline:
                extra["cpu_baseline"] = cpu_baseline(args)
    if rank == 0:
        if args.config == "sdxl":
            workload = (f"configs[4]: SDXL de-tokenizer standalone, one 1024^2 image per step per GPU from a 256x4096 image-"
                        f"feature tensor: ResamplerXLV2 + zero-image ViT branch (cached) + {args.denoise_steps} Euler steps CFG 7.5 "
                        f"(UNet batch 2) + VAE decode")
        elif args.config == "sink":
            workload = (f"configs[3]: {max(1, args.stories_per_gpu)} stor{'y' if args.stories_per_gpu <= 1 else 'ies'} per GPU "
                        f"(MLLM decode steps batched over the paged KV cache), {args.turns}-turn stories in LIVE attention-sink mode "
                        f"(paged KV kept across turns, sink retention at each eviction, window 8), SDXL {args.denoise_steps} steps")
        else:
            workload = ("configs[1]: 10-turn interleaved story, batch=1 per GPU, fp16, 448^2 start image, 64-token caption, "
                        f"64 text tokens + 66-token image run per turn, SDXL 1024^2 {args.denoise_steps} Euler steps CFG 7.5, "
                        "window 8" + ("; at N GPUs = configs[2] (N stories data-parallel, one image per GPU)" if world > 1 else ""))
        line = dict(metric=METRICS[args.config], value=round(value, 4), unit=unit, n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=round(ms / args.steps, 2), higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype="f16", data="synthetic",
                    config=dict(workload=workload, turns_per_step=(args.turns if args.config != "sdxl" else None),
                                units_counted=int(n_units), stories_per_gpu=max(1, args.stories_per_gpu),
                                parallelism=f"dp{world} (independent replicas, no data-path collective)",
                                timing="operands (13.2 GB Llama weights per decode step, 5.1 GB UNet) exceed the 126 MB L2; no flush needed",
                                weights="seeded random, real shapes (no checkpoints offline)",
                                schedule="EOS and <img> suppressed in the 64 free text slots (SuppressTokens semantics), <img> "
                                         "forced at slot 64, EOS after </img>"),
                    e2e=dict(value=round(e2e_value, 4), unit=unit, h2d_bytes_per_step=counters["h2d"] // e2e_steps,
                             d2h_bytes_per_step=counters["d2h"] // e2e_steps, steps=e2e_steps,
                             ms_per_step=round(ms_e2e / e2e_steps, 2)),
                    gpu_launches=int(launches), clocks=clocks)
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def measure_rooflines(pipe, dev, peaks, args):
    """Live CUDA-event measurements of the dominant kernels on this GPU (rank 0, after the timed regions)."""
    from seedstory import ops
    out = {}
    ue = pipe.unet.engine()
    if ue._graph is None:
        return out
    # one eager UNet forward records every tcgen05 GEMM / conv / attention launch together with a closure that re-issues
    # it on the same buffers; each distinct GEMM/conv launch type is then timed as 10 back-to-back launches inside a
    # CUDA graph (CUDA events on the launching stream, no host gaps, programmatic-dependent-launch overlap as in the
    # real step), and the per-launch times are weighted by how often the type occurs in the step
    ops.RECORD = []
    torch.cuda.synchronize()
    ue.forward()
    torch.cuda.synchronize()
    rec = ops.RECORD
    ops.RECORD = None
    types = {}
    for name, fl, fn in rec:
        if name.startswith("fmha"):
            continue
        t = types.setdefault(name, [0, fl, fn])
        t[0] += 1
    g0, g1 = ev(), ev()
    side = torch.cuda.Stream()
    tc_ms = 0.0
    per_type = []
    for name, (cnt, fl, fn) in types.items():
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(10):
                fn()
        gr.replay()
        torch.cuda.synchronize()
        g0.record()
        for _ in range(3):
            gr.replay()
        g1.record()
        torch.cuda.synchronize()
        us = g0.elapsed_time(g1) / 30 * 1e3
        tc_ms += cnt * us * 1e-3
        per_type.append((cnt * us, name, cnt, round(us, 2), round(fl / us / 1e6, 1)))
        del gr
    per_type.sort(reverse=True)
    tc_fl = sum(f for (n, f, _) in rec if not n.startswith("fmha"))
    attn_fl = sum(f for (n, f, _) in rec if n.startswith("fmha"))
    g0.record()
    for _ in range(10):
        ue._graph.replay()
    g1.record()
    torch.cuda.synchronize()
    fwd_ms = g0.elapsed_time(g1) / 10
    ach = tc_fl / (tc_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    tf = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if os.path.exists(tf):
        try:
            with open(tf) as f:
                t = json.load(f)
            traffic, traffic_src = t.get("dram_bytes_per_launch"), t.get("source")
        except Exception:
            pass
    out["roofline"] = dict(
        bound="tensor", kernel="gemm_tc_pair_kernel / gemm_tc_persist_kernel (tcgen05 GEMM + implicit-GEMM conv3x3 of the SDXL UNet)",
        achieved=round(ach, 1), peak=peaks["tf_burst"], unit="TFLOP/s", frac=round(ach / peaks["tf_burst"], 4),
        traffic=traffic, traffic_source=traffic_src,
        peak_source=peaks["src"] + ", burst bf16 (each launch type timed in isolation)",
        method="per launch type: 10 back-to-back launches in a CUDA graph, CUDA events; weighted by count in the step",
        top_types=[dict(launch=n, count=c, us=u, tflops=t) for (_, n, c, u, t) in per_type[:6]],
        launches_per_unet_step=len(rec), algorithmic_tflop=round(tc_fl / 1e12, 3),
        share_of_unet_step=round(tc_ms / fwd_ms, 3))
    whole = (tc_fl + attn_fl) / (fwd_ms * 1e-3) / 1e12
    out["roofline_whole_step"] = dict(
        bound="tensor", kernel="one UNet CFG step (batch 2, 128^2 latents): all launches of the captured CUDA graph",
        achieved=round(whole, 1), peak=peaks["tf_sustained"], unit="TFLOP/s", frac=round(whole / peaks["tf_sustained"], 4),
        algorithmic_tflop=round((tc_fl + attn_fl) / 1e12, 3), attention_tflop=round(attn_fl / 1e12, 3),
        ms=round(fwd_ms, 3), peak_source=peaks["src"] + ", sustained bf16 (timed inside a long step)")
    # ---- Llama decode step at the mean context of the workload (HBM-bound: weights + KV streamed once per step)
    eng = pipe.agent.llm.engine()
    c = eng.cfg
    ctx = MEAN_PROMPT + N_TEXT
    emb = (torch.randn(ctx, c.hidden, device=dev) * 0.02).half()
    eng.reset_sequence(0)
    eng.forward_chunk(0, emb, list(range(ctx)), want_logits=False)
    eng.begin_decode([5], [ctx])
    eng.decode_step(1)
    torch.cuda.synchronize()
    state = [t.clone() for t in (eng.cur_ids, eng.tok_pos, eng.tok_slot, eng.seq_lens, eng.n_out, eng.done)]
    reps = 20
    g0.record()
    for _ in range(reps):
        eng.decode_step(1)
    g1.record()
    torch.cuda.synchronize()
    dec_ms = g0.elapsed_time(g1) / reps
    for t, sv in zip((eng.cur_ids, eng.tok_pos, eng.tok_slot, eng.seq_lens, eng.n_out, eng.done), state):
        t.copy_(sv)
    eng.reset_sequence(0)
    wbytes = sum(t.numel() * 2 for L in eng.w["layers"] for k, t in L.items()) + eng.w["lm_head"].numel() * 2 \
        + eng.w["norm"].numel() * 2
    mean_ctx = ctx + reps / 2
    kvbytes = c.layers * 2 * c.heads * c.head_dim * 2 * (mean_ctx + 1)
    gbs = (wbytes + kvbytes) / (dec_ms * 1e-3) / 1e9
    out["roofline_decode"] = dict(
        bound="hbm", kernel="one Llama-2-7B decode step (CUDA graph: skinny GEMMs + paged split-KV attention), batch 1",
        achieved=round(gbs, 1), peak=peaks["hbm"], unit="GB/s", frac=round(gbs / peaks["hbm"], 4),
        algorithmic_bytes=int(wbytes + kvbytes), context=int(mean_ctx), ms=round(dec_ms, 4), peak_source=peaks["src"])
    # ---- SDXL de-tokenizer alone (the img/s half of the metric)
    feat = (torch.randn(1, 256, 4096, device=dev) * 0.5).half()

    def one():
        return pipe.adapter.generate(image_embeds=feat, num_inference_steps=args.denoise_steps, height=1024, width=1024,
                                     output_type="pt", input_image_size=448)
    one()
    g0.record()
    for _ in range(2):
        one()
    g1.record()
    torch.cuda.synchronize()
    img_ms = g0.elapsed_time(g1) / 2
    out["sdxl_img_per_s"] = dict(value=round(1e3 / img_ms, 4), unit="img/s", denoise_steps=args.denoise_steps,
                                 ms_per_image=round(img_ms, 1), note="one GPU, batch 1 (UNet batch 2 = CFG), incl. VAE decode")
    return out


# ------------------------------------------------------------------------------------------------
# "reference fp16 GPU path": the oracle in eager fp16 PyTorch on the same GPU (bounded sample)
# ------------------------------------------------------------------------------------------------
def gpu_eager_baseline(dev, args):
    from oracle import llama_oracle as LO
    from oracle import sdxl_oracle as SO
    from oracle import vision_oracle as VO
    from seedstory import story, synthetic
    torch.cuda.empty_cache()

    def timed(fn, n):
        fn()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n * 1e-3

    old_te, old_rope, old_att = SO.timestep_embedding, LO.rope_tables, LO.attend_bottom_right
    try:
        with torch.no_grad():
            SO.timestep_embedding = lambda t, dim, max_period=10000: old_te(t.cpu(), dim, max_period).to(dev)
            cfg = SO.SDXL_UNET_CONFIG
            sd = {k: v.to(torch.float16) for k, v in synthetic.random_unet_state_dict(cfg, seed=1, device=dev).items()}
            x = torch.randn(2, 4, 128, 128, device=dev).half()
            ctx = torch.randn(2, 64, 2048, device=dev).half()
            pooled = torch.randn(2, 1280, device=dev).half()
            tid = torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]] * 2, device=dev).half()
            t_unet = timed(lambda: SO.unet_forward(sd, cfg, x, torch.tensor([981.0, 981.0], device=dev), ctx, pooled, tid), 3)
            del sd
            vcfg = dict(synthetic.SDXL_VAE_CONFIG)
            vsd = {k: v.float() for k, v in synthetic.random_vae_decoder_state_dict(vcfg, seed=2, device=dev).items()}
            lat = torch.randn(1, 4, 128, 128, device=dev) * 0.2
            t_vae = timed(lambda: SO.vae_decode(vsd, vcfg, lat), 2)      # fp32 upcast, as diffusers does (force_upcast)
            del vsd
            torch.cuda.empty_cache()
            # Llama-2-7B + unmerged LoRA, fp16 on the device
            g = torch.Generator(device=dev).manual_seed(1)
            p = LO.LlamaParams(4096, 11008, 32, 32, 32066, lora_r=16)
            rn = lambda *s: (torch.randn(*s, generator=g, device=dev) * 0.02).half()
            p.embed, p.norm, p.lm_head = rn(32066, 4096), torch.ones(4096, device=dev).half(), rn(32066, 4096)
            for _ in range(32):
                Ld = {}
                for name, (o, i) in {"q_proj": (4096, 4096), "k_proj": (4096, 4096), "v_proj": (4096, 4096), "o_proj": (4096, 4096),
                                     "gate_proj": (11008, 4096), "up_proj": (11008, 4096), "down_proj": (4096, 11008)}.items():
                    Ld[name], Ld[name + ".lora_A"], Ld[name + ".lora_B"] = rn(o, i), rn(16, i), rn(o, 16)
                Ld["input_layernorm"] = torch.ones(4096, device=dev).half()
                Ld["post_attention_layernorm"] = torch.ones(4096, device=dev).half()
                p.layers.append(Ld)
            LO.rope_tables = lambda d, n, base=10000.0: tuple(t.to(dev) for t in old_rope(d, n, base))

            def attend(q, k, v):
                tq, tk = q.shape[-2], k.shape[-2]
                qi = torch.arange(tq, device=q.device).unsqueeze(1)
                kj = torch.arange(tk, device=q.device).unsqueeze(0)
                return torch.nn.functional.scaled_dot_product_attention(q, k, v, attn_mask=(kj <= qi + (tk - tq)))
            LO.attend_bottom_right = attend
            L = MEAN_PROMPT
            emb = (torch.randn(1, L, 4096, device=dev) * 0.02).half()
            pos = torch.arange(L, device=dev).unsqueeze(0)
            t_pre = timed(lambda: LO.model_forward(p, emb, pos, None), 2)
            _, _, kv = LO.model_forward(p, emb, pos, None)

            def step():
                lg, _, _ = LO.model_forward(p, emb[:, :1], torch.tensor([[L]], device=dev), kv)
                return int(lg[0, -1].argmax().item())         # the reference syncs every token (generation.py:22)
            t_dec = timed(step, 5)
            del p, kv
            torch.cuda.empty_cache()
            # zero-image ViT the reference recomputes every turn (adapter_modules.py:406-414)
            from src.models.qwen_visual import VisionTransformerWithAttnPool
            with torch.device(dev):
                vit = VisionTransformerWithAttnPool(**story.FULL["vit"])
            vsd = {k: v.detach().half().to(dev) for k, v in vit.state_dict().items()}   # (sincos tables are built on the host)
            del vit
            z = torch.zeros(1, 3, 448, 448, device=dev).half()
            vc = story.FULL["vit"]
            t_vit = timed(lambda: VO.vit_forward(vsd, z, vc["heads"], vc["layers"], vc["patch_size"]), 2)
            del vsd
    finally:
        SO.timestep_embedding, LO.rope_tables, LO.attend_bottom_right = old_te, old_rope, old_att
        torch.cuda.empty_cache()
    turn = TOKENS_PER_TURN * t_dec + t_pre + args.denoise_steps * t_unet + t_vae + t_vit
    return dict(value=round(1.0 / turn, 4), unit="story-turns/s", kind="oracle restatement of the reference path, eager fp16 PyTorch on this GPU",
                sample=f"UNet CFG step {t_unet * 1e3:.1f} ms x {args.denoise_steps}; decode step (32 layers, unmerged LoRA r=16, python loop "
                       f"with .item(), ctx {L}) {t_dec * 1e3:.2f} ms x {TOKENS_PER_TURN}; re-prefill {L} tokens {t_pre * 1e3:.1f} ms; fp32 VAE decode "
                       f"{t_vae * 1e3:.1f} ms; zero-image ViT-G {t_vit * 1e3:.1f} ms; resamplers / scheduler glue left out (favours the baseline)",
                turn_s=round(turn, 4))


# ------------------------------------------------------------------------------------------------
# CPU: the oracle (fp32 torch restatement of the reference path) on the host cores
# ------------------------------------------------------------------------------------------------
def usable_threads():
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def pick_threads():
    """torch's CPU GEMMs stop scaling (and collapse when oversubscribed) beyond a few dozen threads: take the thread
    count that maximises a 4096^3 fp32 matmul among {8,16,32,48,64,96,128} <= usable threads."""
    limit = usable_threads()
    a = torch.randn(4096, 4096)
    best, best_t = 0.0, 1
    for th in (8, 16, 32, 48, 64, 96, 128):
        if th > limit and th != 8:
            break
        torch.set_num_threads(th)
        a @ a
        t0 = time.time()
        a @ a
        r = 1.0 / (time.time() - t0)
        if r > best * 1.05:
            best, best_t = r, th
    torch.set_num_threads(best_t)
    return best_t, limit, round(best * 2 * 4096 ** 3 / 1e12, 2)


class CpuReference:
    """Full-size fp32 oracle pieces for the bounded CPU sample.  One *reference step* =
         1 decoded token through 32 decoder-layer passes (+ final norm + lm_head) at the mean context, and
         1 full-resolution (128^2 latents) batch-1 UNet forward (a CFG step is two of them).
    Host memory is bounded by cycling 4 distinct fp32 layer weight sets (3.2 GB, far beyond any L3) over the 32 layer
    passes; every pass does the full arithmetic.  A turn = 131 decoded tokens + 50 CFG steps (= 100 batch-1 forwards)
    + one re-prefill + fp32 VAE decode + zero-image ViT (each of the last three measured once, in `setup`)."""

    def __init__(self, args):
        from oracle import llama_oracle as LO
        from oracle import sdxl_oracle as SO
        from seedstory import synthetic
        self.LO, self.SO, self.args = LO, SO, args
        self.threads, self.limit, self.gemm_tf = pick_threads()
        self.p4 = LO.LlamaParams.random(4096, 11008, 32, 4, 32066, lora_r=16, seed=1)
        self.p32 = LO.LlamaParams(4096, 11008, 32, 32, 32066, eps=self.p4.eps, lora_r=16, scaling=self.p4.scaling)
        self.p32.embed, self.p32.norm, self.p32.lm_head = self.p4.embed, self.p4.norm, self.p4.lm_head
        self.p32.layers = [self.p4.layers[i % 4] for i in range(32)]
        self.ucfg = dict(SO.SDXL_UNET_CONFIG)
        self.usd = synthetic.random_unet_state_dict(self.ucfg, seed=1234)
        self.ctx = MEAN_PROMPT + N_TEXT
        self.once = {}

    def setup(self):
        """Stages measured once (not per step): re-prefill of the mean prompt, KV cache for the decode sample."""
        LO = self.LO
        with torch.no_grad():
            emb = torch.randn(1, MEAN_PROMPT, 4096) * 0.02
            t0 = time.time()
            _, _, kv = LO.model_forward(self.p32, emb, torch.arange(MEAN_PROMPT).unsqueeze(0), None)
            self.once["prefill_s"] = time.time() - t0
            # pad the cache to the mean decode context with copies (content is irrelevant for timing)
            extra = self.ctx - MEAN_PROMPT
            self.kv = [(torch.cat([k, k[:, :, :extra]], 2), torch.cat([v, v[:, :, :extra]], 2)) for (k, v) in kv]

    def step(self):
        LO, SO = self.LO, self.SO
        with torch.no_grad():
            t0 = time.time()
            LO.model_forward(self.p32, torch.randn(1, 1, 4096) * 0.02, torch.tensor([[self.ctx]]), self.kv)
            t_tok = time.time() - t0
            t0 = time.time()
            SO.unet_forward(self.usd, self.ucfg, torch.randn(1, 4, 128, 128), torch.tensor([981.0]), torch.randn(1, 64, 2048),
                            torch.randn(1, 1280), torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]]))
            t_unet = time.time() - t0
        return t_tok, t_unet

    def turn_seconds(self, t_tok, t_unet):
        return TOKENS_PER_TURN * t_tok + 2 * self.args.denoise_steps * t_unet + self.once.get("prefill_s", 0.0)

    def describe(self, t_tok, t_unet):
        return (f"oracle fp32 on {self.threads} threads ({self.limit} usable, {os.cpu_count()} present; 4096^3 matmul {self.gemm_tf} TFLOP/s): "
                f"per step 1 decoded token x 32 decoder-layer passes + lm_head at ctx {self.ctx} ({t_tok * 1e3:.0f} ms) and 1 full-resolution "
                f"batch-1 UNet forward ({t_unet:.2f} s); turn = {TOKENS_PER_TURN} tokens + {2 * self.args.denoise_steps} UNet forwards + re-prefill of "
                f"{MEAN_PROMPT} tokens ({self.once.get('prefill_s', 0.0):.1f} s, measured once); fp32 VAE and zero-image ViT left out (favours CPU)")


def cpu_baseline(args):
    t_all = time.time()
    ref = CpuReference(args)
    ref.setup()
    t_tok, t_unet = ref.step()
    turn = ref.turn_seconds(t_tok, t_unet)
    return dict(value=round(1.0 / turn, 6), unit="story-turns/s", cores=ref.threads, kind="port",
                sample=ref.describe(t_tok, t_unet) + f"; sample wall {time.time() - t_all:.0f} s")


def run_reference(args):
    """Reference arm: the reference's CPU path = the oracle port on this box's host cores.  Every step REALLY runs the
    bounded sample described in CpuReference (ms_per_step is its measured wall time, so steps x ms_per_step fits the
    run); `value` converts the mean per-step timings into story-turns/s with the fixed turn composition."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_start = time.time()
    ref = CpuReference(args)
    ref.setup()
    for _ in range(args.warmup):
        ref.step()
    toks, unets = [], []
    t0 = time.time()
    for _ in range(args.steps):
        a, b = ref.step()
        toks.append(a)
        unets.append(b)
    wall = time.time() - t0
    t_tok, t_unet = sum(toks) / len(toks), sum(unets) / len(unets)
    if args.config == "sdxl":
        v = 1.0 / (2 * args.denoise_steps * t_unet)
        unit = "img/s"
    else:
        v = 1.0 / ref.turn_seconds(t_tok, t_unet)
        unit = "story-turns/s"
    base = dict(value=round(v, 6), unit=unit, cores=ref.threads, kind="port", sample=ref.describe(t_tok, t_unet))
    line = dict(metric=METRICS[args.config], value=round(v, 6), unit=unit, n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=round(wall / args.steps * 1e3, 1), higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=dict(workload="same workload as our arm; CPU fp32 oracle port of the reference path (transformers 4.34 / diffusers / "
                                     "peft / xformers are not installable offline, so `oracle/` stands in for them); each step is the bounded "
                                     "sample in cpu_baseline.sample, really executed; value = 1 / (fixed turn composition x measured per-op times)",
                            turns_per_step=args.turns),
                cpu_baseline=base,
                e2e=dict(value=round(v, 6), unit=unit, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                note=f"whole run {time.time() - t_start:.0f} s on the host; timed region {wall:.0f} s")
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="story", choices=["story", "sink", "sdxl"])
    ap.add_argument("--turns", type=int, default=None)
    ap.add_argument("--denoise-steps", type=int, default=None)
    ap.add_argument("--stories-per-gpu", type=int, default=1, help="stories per step per GPU; > 1 batches their MLLM decode "
                    "steps over the paged KV cache (BASELINE configs[3] uses 4)")
    ap.add_argument("--e2e-steps", type=int, default=6, help="steps of the host-buffer (e2e) leg, <= --steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last "
                    "timed step returned (rank 0) as DIR/<name>.npy, float32, under 64 MB in all (see dump_outputs)")
    args = ap.parse_args()
    if args.turns is None:
        args.turns = 25 if args.config == "sink" else TURNS
    if args.denoise_steps is None:
        args.denoise_steps = 30 if args.config == "sdxl" else DENOISE_STEPS
    if args.impl == "reference":
        if args.dump_outputs is not None:
            ap.error("--dump-outputs: the reference arm times oracle pieces and returns no story outputs")
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
