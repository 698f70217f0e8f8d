#!/usr/bin/env python
"""VQACL train-step throughput on B200 (BASELINE.json metric: train samples/s, VL-T5 base, 36 RoIs).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic batch of configs[1]: VLT5VQA.train_step (forward with the SI
prototype update/retrieval) + loss.backward() + clip_grad_norm_(5) + HF AdamW, B = 320 per GPU, 36 x 2048 RoI features,
20 question tokens, 5 target tokens, dropout 0.1, task id 3 (SURVEY.md §8d). N > 1 is launched with torchrun, one rank
per GPU, weak scaling, gradients averaged over NCCL from inside backward.

  value : whole-job samples/s with the batch resident in HBM, CUDA-event timed, max over ranks
  e2e   : the same through the public API with the batch in PINNED HOST memory (H2D inside the timed region) and a
          device->host read of the loss every step
  roofline : the step's algorithmic tensor FLOPs (37.79 GFLOP/sample, SURVEY.md §8d) / step time vs the measured
          sustained bf16 peak (MEASURED_PEAKS.json), plus per-GEMM-shape figures timed in isolation (burst peak)
  cpu_baseline : the fp32 oracle (oracle/vlt5_oracle.py, a port of the reference's PyTorch path) on the host cores,
          configs[0] (B = 8), rank 0 only
`--impl reference` times that CPU path alone (the reference is pure PyTorch and cannot be imported here — SURVEY.md H3 —
so the oracle port is the reference arm).

`--dump-outputs DIR` writes what the last timed step returned to its caller, as DIR/<name>.npy (float32, or float64 for
integers): train mode the loss, the prototype-retrieval indices, the encoder attention mask, the logits and encoder hidden
states of a fixed seeded sample of batch rows, the SI prototype banks, and a fixed seeded sample of every parameter after
the optimizer step; decode mode the generated token ids. Inputs, weights and dropout seeds depend only on the arguments,
so two builds can be compared output for output (weight gradients accumulate with fp32 atomics, so the comparison needs
a tolerance, not bit equality).
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
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

FLOP_PER_SAMPLE_STEP = 37.79e9          # SURVEY.md §8(d): forward 12.634 GFLOP x 3 minus the unneeded VisEmbed dX (T = 5, S = 56)
METRIC = "VQACL train samples/s (VL-T5 base, 36 RoIs)"
DUMP_ROWS = 16                          # --dump-outputs: batch rows kept of the [B, ...] float outputs (logits alone are 206 MB)
DUMP_PARAM_ELEMS = 1024                 # --dump-outputs: elements kept of every parameter
DUMP_LIMIT = 64 << 20


def dump_rows(B):
    """The fixed, seeded sample of batch rows --dump-outputs keeps."""
    import torch
    return torch.randperm(B, generator=torch.Generator().manual_seed(0))[:min(B, DUMP_ROWS)].sort().values


def write_dump(out_dir, arrays):
    """arrays: name -> tensor; written as out_dir/<name>.npy, integers as float64 (exact), floats as float32."""
    import numpy as np
    import torch
    host = {}
    for name, t in arrays.items():
        t = t.detach().cpu()
        host[name] = (t.double() if not t.is_floating_point() or t.dtype == torch.float64 else t.float()).numpy()
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def step_flops(N=36, L=20, T=5, d=768, f=3072, V=32200, F=2048, Le=12, Ld=12):
    """Algorithmic tensor FLOPs of one train step per sample (SURVEY.md §8d formulas; 37.79e9 at the configs[1] shape)."""
    S, S2 = L + N, L + N + 2
    fwd = (N * 2 * (F + 5) * d + Le * (8 * S * d * d + 4 * S * S * d + 4 * S * d * f)
           + Ld * (8 * T * d * d + 4 * T * T * d + 4 * T * d * d + 4 * S2 * d * d + 4 * T * S2 * d + 4 * T * d * f) + 2 * T * d * V)
    return 3 * fwd - N * 2 * F * d


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), hbm=d["hbm_gbs"],
                    source="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference(steps, warmup, B=8):
    """configs[0]: the fp32 oracle port of the reference path on all host cores; one full step = forward + backward +
    clip_grad_norm_(5) + HF AdamW, dropout 0, task 0 (SURVEY.md §8d)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vlt5_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = O.VLT5Config(dropout_rate=0.0)
    model = O.VLT5VQA(cfg).init_weights_like_reference(66666)
    model.train()
    opt = O.HFAdamW(list(model.named_parameters()))
    times = []
    for i in range(warmup + steps):
        batch = O.synthetic_batch(B, seed=1234 + i, task_id=0)
        t0 = time.perf_counter()
        O.full_train_step(model, opt, batch, 0, 0.5, 0.3)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tot = sum(times)
    return dict(value=B * len(times) / tot, unit="samples/s", cores=cores, kind="port",
                sample=f"{len(times)} full fp32 train steps of configs[0] (B={B}, 36 RoIs, L=20, T=5) after {warmup} warm-up, "
                       f"torch {torch.__version__} CPU, {cores} threads", ms_per_step=1e3 * tot / len(times)), B


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)      # one step = one B = 8 train step (~0.4 s on 16 cores)
    cb, B = cpu_reference(steps, warm)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "samples/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"VL-T5 base VQACL train step on host CPU (oracle port of the reference), batch {B}, 36 RoIs x 2048, "
                                   "20 question tokens, 5 target tokens, SI prototype bank"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def gemm_shape_rooflines(eng, pk, B):
    """The dominant tcgen05 GEMM shapes of the step timed in isolation (CUDA events, 20 launches each)."""
    import ctypes
    import torch
    from vqacl_b200._lib import check, cur_stream, ptr
    L = eng.L
    out = []
    M = B * 56
    shapes = [("enc qkv fwd", M, 2304, 768, 0, 0, 0), ("enc ffn wi fwd (+relu)", M, 3072, 768, 0, 0, 1),
              ("enc ffn wo fwd (+residual)", M, 768, 3072, 0, 0, 2), ("enc ffn dX (B mn-major)", M, 3072, 768, 0, 1, 0),
              ("enc ffn dW (split-K)", 3072, 768, M, 1, 1, 3)]
    for name, m, n, k, amn, bmn, epi in shapes:
        A = torch.randn((k, m) if amn else (m, k), device=eng.device).bfloat16()
        Bm = torch.randn((k, n) if bmn else (n, k), device=eng.device).bfloat16()
        C = torch.zeros(m, n, device=eng.device, dtype=torch.float32 if epi in (2, 3) else torch.bfloat16)
        R = torch.zeros(m, n, device=eng.device) if epi == 2 else None
        splits = 1
        if epi == 3:
            tiles = ((m + 127) // 128) * ((n + 255) // 256)
            splits = max(1, min((2 * 148) // tiles, ((k + 63) // 64) // 8))

        def call():
            check(L.vqacl_gemm_bf16(ptr(A), A.stride(0), amn, ptr(Bm), Bm.stride(0), bmn, ptr(C), C.stride(0), ptr(R),
                                    R.stride(0) if R is not None else 0, m, n, k, epi, ctypes.c_float(1.0), splits, 0, cur_stream()))
        for _ in range(3):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(20):
            call()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / 20
        tf = 2.0 * m * n * k / us / 1e6
        out.append({"kernel": f"gemm_bf16_tcgen05 {name}", "M": m, "N": n, "K": k, "us": round(us, 2), "achieved": round(tf, 1),
                    "peak": pk["burst"], "unit": "TFLOP/s", "frac": round(tf / pk["burst"], 4)})
    return out


def run_native(args):
    import torch
    import torch.distributed as dist
    import vqacl_b200 as V
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vlt5_oracle as O                       # synthetic_batch generator + the cpu_baseline leg only

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()

    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:      # N = 1 only (contract): at N > 1 torchrun pins OMP to one thread and
        cpu_base, _ = cpu_reference(24, 1)           # the other ranks would sit in a barrier; the driver times the CPU arm itself
        torch.set_num_threads(max(1, (os.cpu_count() or 8) // max(1, world)))
    if world > 1:
        dist.barrier()

    B, task = args.batch, 3
    cfg = V.VLT5Config(vocab_size=32200, dropout_rate=args.dropout)
    torch.manual_seed(66666)                      # param.py:58 default seed; identical weights on every rank
    model = V.VLT5VQA(cfg)
    model.encoder.visual_embedding.feat_embedding[0].weight.data.normal_(0, 1)      # H14: visual layers stay N(0,1)
    model.encoder.visual_embedding.absolute_vis_pos_embedding[0].weight.data.normal_(0, 1)
    model.encoder.visual_embedding.img_order_embedding.weight.data.normal_(0, 1)
    model = model.to(dev)
    model.train()
    if os.environ.get("VQACL_COMM_SMS"):
        model.comm_sms = int(os.environ["VQACL_COMM_SMS"])
    opt = V.FusedAdamW(model, lr=1e-4, eps=1e-6, weight_decay=0.01, overlap_with_next_forward=not args.no_overlap_optimizer,
                       shard_state=False if os.environ.get("VQACL_NO_SHARD") == "1" else None)
    sched = V.get_constant_schedule_with_warmup(opt, 10)

    # a small pool of distinct batches: pinned host copies (e2e) and device-resident copies (value)
    pool = 4
    host, devb = [], []
    for i in range(pool):
        b = O.synthetic_batch(B, seed=1234 + rank * 1000 + i, task_id=task, rehearsal=(i % 2 == 1), n_boxes=args.boxes)
        hb = {k: v.pin_memory() for k, v in b.items()}
        host.append(hb)
        devb.append({k: v.to(dev) for k, v in b.items()})
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())

    dumped = {}
    rows = dump_rows(B).to(dev) if args.dump_outputs else None

    def step(batch, read_loss, keep=False):
        r = model.train_step(batch, task, 0.5, 0.3)
        if keep:
            # device copies taken as train_step returns: the returned tensors are views of workspaces later kernels reuse
            dumped.update(loss=r["loss"].detach().clone(), max_idx_Q=r["max_idx_Q"].clone(), max_idx_V=r["max_idx_V"].clone(),
                          encoder_attention_mask=r["encoder_attention_mask"].clone(), sample_rows=rows,
                          logits_sample=r["logits"].index_select(0, rows),
                          encoder_hidden_states_sample=r["encoder_hidden_states"].index_select(0, rows))
        r["loss"].backward()
        opt.step(max_grad_norm=5.0)
        sched.step()
        opt.zero_grad()
        if read_loss:
            return r["loss"].item()
        return None

    prefetcher = {}

    def timed(batches, steps, warmup, read_loss, prefetch=False, keep_last=False):
        if prefetch:
            prefetcher["p"] = V.BatchPrefetcher(None, dev)
            prefetcher["p"].loader = [batches[i % pool] for i in range(max(warmup, 4))]
            for b in prefetcher["p"]:          # warm-up through the same path: staging buffers get allocated here
                step(b, read_loss)
        else:
            for i in range(warmup):
                step(batches[i % pool], read_loss)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = model._engine.launch_count()
        e0.record()
        if prefetch:
            # the public input path: pinned host batches -> BatchPrefetcher (H2D of batch i+1 on a side stream during step i)
            prefetcher["p"].loader = (batches[i % pool] for i in range(steps))
            for b in prefetcher["p"]:
                step(b, read_loss)
        else:
            for i in range(steps):
                step(batches[i % pool], read_loss, keep=keep_last and i == steps - 1)
        model.param_sync()          # an overlapped optimizer tail of the last step belongs to the timed region
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, model._engine.launch_count() - l0

    warm = max(3, args.warmup)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms, launches = timed(devb, args.steps, warm, False, keep_last=bool(args.dump_outputs))
    ck = clocks.stop() if rank == 0 else None
    if args.dump_outputs:
        g = torch.Generator().manual_seed(0)
        params = [v.detach().reshape(-1)[torch.randint(0, v.numel(), (min(v.numel(), DUMP_PARAM_ELEMS),), generator=g).to(v.device)]
                  for v in model.state_dict().values() if v.is_floating_point()]
        dumped.update(Q_prototype=model.Q_prototype, V_prototype=model.V_prototype, params_sample=torch.cat([p.float() for p in params]))
        if rank == 0:
            write_dump(args.dump_outputs, dumped)
    ms_e2e, _ = timed(host, args.steps, 2, True, prefetch=True)
    # the literal drop-in call: pinned CPU batch straight into train_step, whose own .to(device) copies it on the compute stream
    ms_dropin, _ = timed(host, args.steps, 2, True, prefetch=False)
    value = world * B * args.steps / (ms / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)
    e2e_dropin = world * B * args.steps / (ms_dropin / 1e3)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_step_dram_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_step")
    if rank == 0:
        flop = FLOP_PER_SAMPLE_STEP if args.boxes == 36 else step_flops(N=args.boxes)
        tf = value / world * flop / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"configs[1]: VL-T5 base (T5-base geometry, random init, vocab 32200) VQACL train step, batch {B} per GPU, "
                                   f"{args.boxes} RoIs x 2048-d + boxes, 20 question tokens, 5 target tokens, SS encoder + SI prototype bank "
                                   f"(10 question types + 80 object classes), dropout {args.dropout}, task id {task}, "
                                   "fwd + bwd + clip_grad_norm_(5) + HF AdamW",
                       "global_batch": B * world,
                       "parallelism": f"dp{world}" + (" (gradients reduce-scattered, optimizer state sharded, bf16 weights all-gathered)"
                                                       if getattr(opt, "shard", False) else ""),
                       "l2": "per-step working set (activations ~6 GB, weights+optimizer 3.6 GB) >> 126 MB L2; 4 distinct batches rotate"},
            "e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps, "path": "pinned host batch -> vqacl_b200.BatchPrefetcher -> VLT5VQA.train_step",
                    "dropin_value": e2e_dropin, "dropin_ms_per_step": ms_dropin / args.steps,
                    "dropin_path": "pinned host batch -> VLT5VQA.train_step (the reference's call, vqa_model.py:20-27; H2D on the compute stream)"},
            "gpu_launches": int(launches),
            "clocks": ck,
            "roofline": {"bound": "tensor", "achieved": round(tf, 1), "peak": pk["sustained"], "unit": "TFLOP/s",
                         "frac": round(tf / pk["sustained"], 4), "traffic": traffic,
                         "traffic_note": "DRAM bytes read + written by all kernels of one step (ncu dram__bytes_read/write.sum over a step window, "
                                         "profiles/r02_step_dram_traffic.json); null until captured",
                         "kernel": f"whole train step: algorithmic {flop / 1e9:.2f} GFLOP/sample (98.7% in gemm_bf16_tcgen05 launches) / step time, per GPU",
                         "peak_source": pk["source"] + " sustained bf16 (kernel timed inside a long step)"},
        }
        if not args.no_kernel_roofline:
            line["roofline_kernels"] = gemm_shape_rooflines(model._engine, pk, B)
        if cpu_base is not None:
            line["cpu_baseline"] = {k: cpu_base[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_decode(args):
    """configs[4]: eval-only greedy answer generation (VLT5VQA.test_step, vqa_model.py:68-121), batch 512 per GPU, <= 20
    tokens, frozen prototype banks; every rank decodes its own shard (no data-path collective)."""
    import torch
    import torch.distributed as dist
    import vqacl_b200 as V
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vlt5_oracle as O                       # synthetic_batch generator only
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    B = args.batch if args.batch != 320 else 512
    cfg = V.VLT5Config(vocab_size=32200, dropout_rate=0.0)
    torch.manual_seed(66666)
    model = V.VLT5VQA(cfg)
    for mod in (model.encoder.visual_embedding.feat_embedding[0], model.encoder.visual_embedding.absolute_vis_pos_embedding[0],
                model.encoder.visual_embedding.img_order_embedding):
        mod.weight.data.normal_(0, 1)
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(9)
    model.Q_prototype, model.V_prototype = torch.randn(10, 768, generator=g), torch.randn(80, 768, generator=g)
    pool = 3
    host = [{k: v.pin_memory() for k, v in O.synthetic_batch(B, seed=77 + rank * 100 + i).items()} for i in range(pool)]
    devb = [{k: v.to(dev) for k, v in b.items()} for b in host]
    h2d = sum(host[0][k].numel() * host[0][k].element_size() for k in ("vis_feats", "boxes", "input_ids"))

    dumped = {}

    def timed(batches, steps, warmup, to_host, keep_last=False):
        ntok = 0
        for i in range(warmup):
            model.test_step(batches[i % pool])
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = model._engine.launch_count()
        e0.record()
        for i in range(steps):
            t = model.test_step(batches[i % pool])["token_ids"]
            if keep_last and i == steps - 1:
                dumped["token_ids"] = t.clone()
            ntok += t.shape[1] - 1
            if to_host:
                t = t.cpu()                        # the answers leave the device (tokenizer.batch_decode runs on the host)
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = tt.item()
        return ms, model._engine.launch_count() - l0, ntok

    warm = max(3, args.warmup)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms, launches, ntok = timed(devb, args.steps, warm, False, keep_last=bool(args.dump_outputs))
    ck = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, dumped)
    ms_e2e, _, _ = timed(host, args.steps, 2, True)
    if rank == 0:
        c = cfg
        dec_w = c.num_decoder_layers * (6 * c.d_model * c.d_model + 2 * c.d_model * c.d_ff) * 2 + c.vocab_size * c.d_model * 2
        kv = B * 58 * c.num_decoder_layers * 2 * c.d_model * 2
        per_tok = dec_w + kv                                   # bf16 decoder + LM-head weights + the cross-attention K/V of 12 layers
        gbs = per_tok * ntok / (ms / 1e3) / 1e9
        line = {"metric": "VQACL eval greedy-decode samples/s (VL-T5 base, 36 RoIs, max_length 20)", "value": world * B * args.steps / (ms / 1e3),
                "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"configs[4]: eval-only greedy answer generation, batch {B} per GPU, 12+12 layers, vocab 32200, random init "
                                       f"(no EOS: all {ntok // max(1, args.steps)} decode steps run), frozen SI prototype banks",
                           "global_batch": B * world,
                           "parallelism": f"dp{world} (independent replicas: evaluation has no exchange step)",
                           "l2": f"{pool} distinct batches rotate; K/V + weights per token step {per_tok / 1e6:.0f} MB > 126 MB L2"},
                "e2e": {"value": world * B * args.steps / (ms_e2e / 1e3), "unit": "samples/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": B * 20 * 8, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "clocks": ck,
                "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": pk["hbm"], "unit": "GB/s", "frac": round(gbs / pk["hbm"], 4),
                             "traffic": None, "kernel": "decode token steps: bytes that must stream per step (bf16 decoder + tied LM-head weights "
                             f"{dec_w / 1e6:.0f} MB + cross-attention K/V {kv / 1e6:.0f} MB) x steps / whole generate time (encoder included in the time)",
                             "peak_source": pk["source"]}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--batch", type=int, default=320)
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--boxes", type=int, default=36,
                    help="visual tokens per sample (36 = configs[1]; 16 = NExT-QA; 64 / 128 = the configs[3] longer-visual-sequence sweep)")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--mode", default="train", choices=["train", "decode"],
                    help="train: configs[1] train step (the BASELINE.json metric); decode: configs[4] greedy evaluation, batch 512")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-roofline", action="store_true")
    ap.add_argument("--no-overlap-optimizer", action="store_true",
                    help="run clip+AdamW on the main stream instead of overlapping it with the next step's forward")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the native implementation")
        # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every host core (set before torch is imported)
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
        os.environ.pop("MKL_NUM_THREADS", None)
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr",
               "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.mode == "decode":
        run_decode(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
