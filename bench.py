"""Headline benchmark: GGNN role-graph stage, images/sec forward+backward (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --steps K --warmup W     # CPU arm: the UNMODIFIED reference (baseline/_ref)

Workload (BASELINE.json configs[2]/[3]): one training step of the GGNN stage at global batch 6144, D=2048,
504 verbs / 190 roles / 2001 labels / 6 roles, synthetic backbone features and labels, random-init weights:
verb path + predicted-verb noun path + gt-verb noun path forward, the three losses, backward of
verb_loss + nouns_loss (sr.py:63-79), gradient all-reduce when N > 1, clip_grad_norm_(1) + Adamax (sr.py:80-83).
The batch is sharded over the N GPUs (strong scaling, as BASELINE.json states it).  Prints ONE JSON line.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_IMAGE_FWD_BWD = 6.547e9   # BASELINE.md section 3 (algorithmic, aggregate-then-project)
# dram__bytes_read.sum + dram__bytes_write.sum of one noun-path launch (M = 36864) from the `ncu --set full` captures
# summarised under profiles/ (r01_ncu_full_gru_kernels.md); None = not captured yet
NCU_TRAFFIC_BYTES = {"gemm_gru_zr_ab": 1.067e9 + 0.434e9, "gemm_gru_h_ab": 1.001e9 + 0.559e9}   # profiles/r01_ncu_full_final.md
METRIC = "ggnn_images_per_sec_fwd_bwd"
UNIT = "images/s"
D = 2048


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"bf16_sustained": d.get("bf16_tflops_sustained", 1396.2), "bf16_burst": d.get("bf16_tflops", 1658.8),
                "hbm_gbs": d.get("hbm_gbs", 6550.4), "source": "measured"}
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # samples under load = the upper half (the sampler also sees the idle edges of the region)
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm
def oracle_setup(B, seed=1234):
    import torch
    from oracle import ggnn_oracle as O
    from situation_recognition_b200.imsitu_encoder import imsitu_encoder
    from situation_recognition_b200.synthetic import make_batch, make_train_json
    enc = imsitu_encoder(make_train_json(seed=0), verbose=False)
    params = O.init_params(enc.get_num_verbs(), enc.get_num_roles(), enc.get_num_labels(), D, seed=0)
    batch = make_batch(enc, B, D, seed=seed)
    tables = O.build_tables(enc.roles_per_verb, enc.verb_list, enc.role_list)
    return O, enc, params, batch, tables


def oracle_step(O, enc, params, batch, tables):
    fv, fn, gt_verb, gt_nouns = batch
    t, c = tables
    return O.train_step_grads(params, fv, fn, gt_verb, gt_nouns, t, c, enc.get_num_labels())


REF_SAMPLE = 64      # images per CPU step: a fixed, bounded sample of the 6144-image step (same at every N)


def reference_runner(sample):
    """(callable running ONE CPU training step on `sample` images, kind, description).

    kind "reference": the unmodified reference classes from the git-ignored copy baseline/_ref (FCGGNN.forward +
    verb_loss + nouns_loss + backward + clip_grad_norm_ + Adamax, sr.py:63-83, backbones replaced by Identity so the
    input is the [B, 2048] feature matrix).  kind "port": the oracle restatement, when no reference copy travelled."""
    import torch
    from oracle import ref_harness
    from situation_recognition_b200.synthetic import make_batch, make_train_json
    if ref_harness.available():
        st = ref_harness.ReferenceStep(make_train_json(seed=0), D=D, seed=0)
        _, fn, gt_verb, gt_nouns = make_batch(st.encoder, sample, D, seed=1234)
        return (lambda: st(fn, gt_verb, gt_nouns)), "reference", \
            "unmodified reference (baseline/_ref: FCGGNN.forward + losses + backward + clip + Adamax, sr.py:63-83, fp32)"
    O, enc, params, batch, tables = oracle_setup(sample)
    return (lambda: oracle_step(O, enc, params, batch, tables)), "port", \
        "oracle port of the reference arithmetic (no baseline/_ref copy on this box), fwd+bwd, fp32"


def cpu_baseline(steps=8):
    """The reference's CPU implementation of the step, timed on this host's cores on a bounded sample (~10-30 s).

    Runs `bench.py --impl reference` in a child process with the GPU hidden: the unmodified reference moves its index
    tensors to CUDA whenever `torch.cuda.is_available()` (model.py:118-119,148-149), so its CPU path only runs in a
    process that sees no GPU."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS"):
        env.pop(k, None)
    try:
        res = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps),
                              "--warmup", "1"], env=env, capture_output=True, text=True, timeout=600)
        lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
        cb = json.loads(lines[-1])["cpu_baseline"]
        cb["sample"] = "%d steps after 1 warm-up; %s" % (steps, cb["sample"])
        return cb
    except Exception as e:   # the GPU measurement above must not be lost to a CPU-leg failure
        return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable",
                "sample": "cpu leg failed: %s" % (str(e)[:200],)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # The unmodified reference sends its role-index / mask tensors to CUDA whenever a GPU is visible
    # (model.py:118-119,148-149): its CPU path -- the arm this flag times -- needs a process that sees none.
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    import torch
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core, the same count at every N
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    steps, warmup = args.steps, args.warmup
    run, kind, what = reference_runner(REF_SAMPLE)
    for _ in range(warmup):
        run()
    t0 = time.time()
    for _ in range(steps):
        run()
    dt = (time.time() - t0) / max(1, steps)
    value = REF_SAMPLE / dt
    cb = {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
          "sample": "each step = %d images (fixed bounded sample of the 6144-image step): %s; os.cpu_count()=%s"
                    % (REF_SAMPLE, what, os.cpu_count())}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "ggnn_stage_fwd_bwd (BASELINE.json configs[2]; sharded = configs[3])",
                       "global_batch": args.batch, "sample_batch": REF_SAMPLE, "D": D,
                       "verbs": 504, "roles": 190, "labels": 2001, "max_roles": 6, "T": 4,
                       "step": "zero_grad+fwd(verb,pred-noun,gt-noun)+3 losses+bwd+clip+adamax"},
            "cpu_baseline": cb,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
DUMP_SAMPLE = 1 << 18      # elements --dump-outputs keeps of a larger tensor: 40 tensors of at most 1 MB


def dump_outputs(out_dir, losses, model):
    """What the last timed step computed, as float32 DIR/<name>.npy: `losses` (verb, nouns, gt-nouns loss) and, for
    every trainable tensor, `param.<name>` (the weights after the optimizer step) and `grad.<name>` (rank 0's gradient
    buffer).  A tensor of more than DUMP_SAMPLE elements is reduced to a fixed, seeded sample of that many flat
    elements, in index order."""
    import numpy as np
    import torch
    arrays = {"losses": losses}
    for name, p in model.named_parameters():
        if p.requires_grad:
            arrays["param." + name] = p
            arrays["grad." + name] = p.grad
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    import situation_recognition_b200 as S
    from situation_recognition_b200 import _lib, parallel
    from situation_recognition_b200.synthetic import make_batch, make_train_json

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the GGNN stage (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # The bench prints exactly ONE line on stdout.  NCCL_DEBUG stays as the caller set it (the driver counts the
    # communicator's ranks in NCCL's INFO lines): everything that is written to fd 1 while the bench runs -- NCCL's banner
    # and INFO lines included -- is redirected to stderr, and the result line goes to the saved stdout at the end.
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    enc = S.imsitu_encoder(make_train_json(seed=0), verbose=False)
    torch.manual_seed(0)
    model = S.FCGGNN(enc, D, backbone=None, precision="bf16").to(dev)
    model.train()
    if args.cta_group:
        model._engine_for(dev).set_cta_group(args.cta_group)
    if args.no_compact_rows:
        model._engine_for(dev).set_compact_rows(False)
    flat = parallel.attach(model, flat_params=True)
    # One GPU: kernels are launched eagerly (with the verb path overlapped on a side stream the GPU never waits for the
    # host at B=6144: graph replay 31.89 ms vs eager 31.87 ms).  Sharded runs replay the whole step (NCCL collectives
    # included) from one CUDA graph: at 8 x 768 images the host needs most of the step time to queue the launches.
    # --graph / --no-graph override.
    use_graph = (args.graph or world > 1) and not args.no_graph
    # sr.py:80-83,472-473 as one fused kernel; sharded over the ranks when N > 1 (reduce-scatter of the gradient, clip +
    # Adamax on 1/N of the parameters, all-gather of the parameters) unless --replicated-optimizer
    sharded = world > 1 and not args.replicated_optimizer
    opt = parallel.FlatAdamax(flat, lr=0.002, max_norm=1.0, group=dist.group.WORLD if sharded else None)
    params = [p for p in model.parameters() if p.requires_grad]
    # --dump-outputs: the last timed step starts again from the seeded initial weights and optimizer state.  The steps
    # before it are as many as the pre-heat's time allows, and atomic / split-K reduce-add sums have no fixed order, so
    # the state they leave differs from run to run; the state they start from does not.  The copies back (~0.5 GB) fall
    # inside the timed window, once.
    dump_state = None
    if args.dump_outputs:
        dump_state = [(t, t.clone()) for t in (flat.flat_param, opt.exp_avg, opt.exp_inf, opt.scratch)]

    def restore_dump_state():
        for t, saved in dump_state:
            t.copy_(saved)
        flat.version += 1                                       # the packed bf16 weights are stale

    Bg = args.batch
    lo, hi = parallel.shard_range(Bg, rank, world)
    Bl = hi - lo
    fv, fn, gt_verb, gt_nouns = make_batch(enc, Bg, D, seed=1234)
    host = [x[lo:hi].contiguous().pin_memory() for x in (fv, fn, gt_verb, gt_nouns)]
    resident = [x.to(dev, non_blocking=True) for x in host]
    h2d_bytes = sum(x.numel() * x.element_size() for x in host)

    model.global_batch = Bg        # the sharded verb loss divides by the global batch without an extra all-reduce

    def step(inputs):
        a, b, v, n = inputs
        model._counts_cache = None      # a real loop sees new labels every step: count (and all-reduce) them every step
        flat.zero()
        pred_verb, pred_nouns, gt_pred_nouns = model(a, v, img_nouns=b)
        vl = model.verb_loss(pred_verb, v)
        nl = model.nouns_loss(pred_nouns, n)
        gl = model.nouns_loss(gt_pred_nouns, n)                # logged, never back-propagated (sr.py:70,76)
        (vl + nl).backward()
        if not sharded:
            flat.all_reduce()
        opt.step()                                              # clip_grad_norm_(1) + Adamax (sr.py:81-82)
        return torch.stack([vl.detach(), nl.detach(), gl.detach()])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k, before_last=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        for i in range(k):
            if i == k - 1 and before_last is not None:
                before_last()
            out = fn()
        timed.host_issue_ms = (time.perf_counter() - t0) * 1e3   # host time to QUEUE the k steps (no sync inside)
        timed.last_out = out
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    gstep = None
    if use_graph:
        # the whole step (no host sync inside) is captured once into a CUDA graph and replayed
        from situation_recognition_b200.graph import GraphedTrainStep
        gstep = GraphedTrainStep(model, opt, flat, Bl).capture(resident)
        run_resident = lambda: gstep(*gstep.static_in)
    else:
        run_resident = lambda: step(resident)
    for _ in range(max(3, args.warmup)):
        run_resident()
    if dump_state is not None:
        # the dropout seed counter exists from the first step on and advances by one per step
        dump_state += [(t, t.clone()) for t in model._seed_state.values()]
    # pre-heat: the same step, back to back for >= args.preheat seconds, so that the timed region starts in the
    # sustained clock / power state at every N (a 0.1 s window after an idle GPU runs at boost clocks)
    t_probe = timed(run_resident, 2) / 2
    n_heat = int(max(0.0, args.preheat) * 1e3 / max(t_probe, 1e-3)) + 1 if args.preheat > 0 else 0
    t_heat0 = time.perf_counter()
    for i in range(n_heat):
        run_resident()
        if (i & 15) == 15:
            torch.cuda.current_stream().synchronize()        # keep the launch queue bounded
    torch.cuda.synchronize()
    preheat_s = time.perf_counter() - t_heat0
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = lib.srg_launch_count()
    total_ms = timed(run_resident, args.steps, restore_dump_state if dump_state is not None else None)
    host_issue_ms = timed.host_issue_ms / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, timed.last_out, model)
    launches = (lib.srg_launch_count() - n0)
    if use_graph:
        launches = gstep.launches * args.steps
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = total_ms / args.steps
    value = Bg / ms_per_step * 1e3

    # ---- dominant kernel, timed live with CUDA events on the launching stream (second pass, same steps)
    kinds = 32
    ms_k = (ctypes.c_double * kinds)()
    fl_k = (ctypes.c_double * kinds)()
    ct_k = (ctypes.c_longlong * kinds)()
    barrier()
    model.overlap_streams = False     # per-kernel event timing needs the kernels one after the other on one stream
    lib.srg_profile_begin()
    for _ in range(args.steps):
        step(resident)
    _lib.check(lib.srg_profile_end(kinds, ms_k, fl_k, ct_k))
    model.overlap_streams = True
    peaks = load_peaks()
    per_kind = []
    for k in range(kinds):
        if ct_k[k] > 0:
            per_kind.append({"kernel": lib.srg_profile_kind_name(k).decode(), "launches_per_step": ct_k[k] / args.steps,
                             "ms_per_step": ms_k[k] / args.steps,
                             "tflops": fl_k[k] / max(ms_k[k], 1e-9) / 1e9})
    per_kind.sort(key=lambda d: -d["ms_per_step"])
    top = per_kind[0]
    gemm_ms = sum(d["ms_per_step"] for d in per_kind)
    executed_flops_per_step = sum(fl_k[k] for k in range(kinds)) / args.steps * world   # all ranks
    roofline = {"bound": "tensor", "kernel": top["kernel"], "achieved": top["tflops"], "peak": peaks["bf16_sustained"],
                "unit": "TFLOP/s", "frac": top["tflops"] / peaks["bf16_sustained"],
                "achieved_note": "FLOPs the kernel executed (2*M*N*K with the device-resident row count of the compact "
                                 "role-node layout: real role nodes + one shared pad row) / CUDA-event time of its "
                                 "launches inside a step; the step_* fields below use the algorithmic 6.547 GFLOP/image",
                "traffic": NCU_TRAFFIC_BYTES.get(top["kernel"]) if Bl == 6144 else None,
                "traffic_note": "bytes of one noun-path launch of this kernel, ncu --set full, profiles/",
                "peak_source": peaks["source"] + " (sustained bf16; burst %.1f)" % peaks["bf16_burst"],
                "peak_burst": peaks["bf16_burst"], "frac_burst": top["tflops"] / peaks["bf16_burst"],
                "step_frac_burst": value * FLOP_PER_IMAGE_FWD_BWD / 1e12 / world / peaks["bf16_burst"],
                "launch_ms": top["ms_per_step"] / top["launches_per_step"],
                "share_of_step": top["ms_per_step"] / ms_per_step,
                # per-GPU figures (the whole-job value divided by the number of GPUs)
                "step_tflops_algorithmic": value * FLOP_PER_IMAGE_FWD_BWD / 1e12 / world,
                "step_frac": value * FLOP_PER_IMAGE_FWD_BWD / 1e12 / world / peaks["bf16_sustained"],
                # the neighbour projection W_p is folded into the gate weights (P_x = W_x W_p), so fewer FLOPs are
                # executed than the algorithmic (aggregate-then-project) count the fraction above is quoted on
                "step_tflops_executed": executed_flops_per_step / (ms_per_step * 1e-3) / 1e12 / world,
                "step_frac_executed": executed_flops_per_step / (ms_per_step * 1e-3) / 1e12 / world
                / peaks["bf16_sustained"],
                "gemm_share_of_step": gemm_ms / ms_per_step, "kernels": per_kind[:8]}

    # ---- end to end through the public API with HOST buffers (pinned), H2D + D2H inside the timed region
    losses_host = torch.empty(3, dtype=torch.float32).pin_memory()

    # The step's inputs start in pinned host memory.  Their H2D copy runs on a copy stream one step ahead (what a
    # DataLoader with pin_memory + non_blocking does), the step waits for it, and the three losses are read back to the
    # host every step (sr.py:88-90 .item()) -- all inside the timed region.
    copy_stream = torch.cuda.Stream(dev)
    staged = [[torch.empty_like(x, device=dev) for x in host] for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]

    def stage(slot):
        with torch.cuda.stream(copy_stream):
            for dst, src in zip(staged[slot], host):
                dst.copy_(src, non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_loop(k):
        stage(0)
        for i in range(k):
            slot = i & 1
            torch.cuda.current_stream().wait_event(ready[slot])
            if i + 1 < k:
                stage(slot ^ 1)                                  # next step's inputs travel while this step computes
            out = gstep(*staged[slot]) if use_graph else step(staged[slot])
            losses_host.copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()            # the caller reads the losses

    e2e_loop(2)
    e2e_ms = timed(lambda: e2e_loop(args.steps), 1) / args.steps
    e2e = {"value": Bg / e2e_ms * 1e3, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes * world,
           "d2h_bytes_per_step": 12 * world, "ms_per_step": e2e_ms}

    cb = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline()
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "ggnn_stage_fwd_bwd (BASELINE.json configs[2]; sharded = configs[3])",
                           "global_batch": Bg, "per_gpu_batch": Bl, "D": D, "verbs": 504, "roles": 190, "labels": 2001,
                           "max_roles": 6, "T": 4, "parallelism": "dp%d" % world,
                           "step": "zero_grad+fwd(verb,pred-noun,gt-noun)+3 losses+bwd+allreduce+clip+adamax",
                           "launch": "cuda_graph_replay" if use_graph else "eager",
                           "collectives": ("reduce_scatter(grads)+allreduce(norm)+all_gather(params), sharded clip+adamax"
                                           if sharded else ("allreduce(grads)" if world > 1 else "none")),
                           "preheat_s": round(preheat_s, 2), "preheat_steps": n_heat,
                           "timed_region_s": round(total_ms / 1e3, 3),
                           "l2": "working set per step (GBs of activations) >> 126 MB L2; no explicit flush",
                           "weights": "random-init (reference default init)", "dropout": "train mode, p=0.5"},
                # host time per step spent queueing the launches: when it approaches ms_per_step the GPU waits for Python
                "host_issue_ms_per_step": host_issue_ms,
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches / args.steps) if args.steps else 0,
                "roofline": roofline}
        if cb is not None:
            line["cpu_baseline"] = cb
        os.write(result_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        # leave without running NCCL / CUDA-graph destructors: a captured or in-flight communicator has been seen to
        # block interpreter shutdown after the result line was already printed
        barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=6144, help="global batch (BASELINE.json: 6144)")
    ap.add_argument("--cta-group", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-compact-rows", action="store_true", help="A/B: R rows per image instead of the compact layout")
    ap.add_argument("--preheat", type=float, default=3.0, help="seconds of untimed back-to-back steps before timing")
    ap.add_argument("--replicated-optimizer", action="store_true",
                    help="N > 1: all-reduce the gradient and run clip + Adamax on every rank (round-1 scheme)")
    ap.add_argument("--graph", action="store_true", help="replay the whole training step from one CUDA graph")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the losses, weights and gradients of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
