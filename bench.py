#!/usr/bin/env python
"""bench.py -- tokens/sec of one Llama-3-8B training step under a Galvatron per-layer hybrid strategy on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]  (N > 1: launched under torchrun)
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]     (CPU restatement of the reference path)

One "step" = forward_backward over the global batch (chunks microbatches) + optimizer step, through the public API
(``llama_model_hp`` -> ``GalvatronModel.forward_backward``), on synthetic tokens of the reference's generator
(``DataLoaderForLlama``) and random-init weights.  Workload at every N: the strategy JSON ``configs/galvatron_config_
llama3-8b_<N>gpus.json`` (per-GPU batch fixed => weak scaling).  Prints ONE JSON line on rank 0.

  value      tokens/s with the step's tokens already resident in HBM (CUDA-event timed, max over ranks)
  e2e        the same loop with the tokens/labels copied from pinned host memory every step and the loss read back
  roofline   the dominant kernel (the tcgen05 GEMM): algorithmic FLOPs / CUDA-event launch time vs the measured cuBLAS peak
  cpu_baseline  the oracle CPU restatement (oracle/gloo_backend.py) on a bounded sample, rank 0 at N=1 only
  probe      two steps on a FIXED batch that is the same on every rank and at every N (loss at init, loss after one update:
             both are N-invariant, so a broken forward or update shows when the driver's N = 1/2/4/8 lines are compared) and,
             at N >= 2, a checksum-of-checksums of the gradient reduction at full size (sum of the reduced shards == sum of the
             unsharded gradients / d, per layer)
  path_legs  (N >= 2) the collectives north_star names, each as a short fixed-strategy run of the SAME model in a child process
             per rank (a failing leg cannot take the headline down): TP=N Megatron-SP (fused all-gather+GEMM / GEMM+reduce-
             scatter), TP=N (fused GEMM+all-reduce, NVLS), Ulysses SP=N (all-to-all), PP=2 x TP=N/2 1F1B (peer-copy p2p),
             ZeRO-3 + checkpointing (and Llama-3-70B ZeRO-3 at N=8, BASELINE config 5): tokens/s, per-collective achieved bus
             GB/s against 900 nominal / 770 measured, and a parity check of the same strategy on the tiny model against the
             oracle (tests/_host_worker.py: loss 5e-3, per-parameter gradients 3e-2 rel-L2).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tokens/sec Llama-3-8B auto-searched hybrid strategy at 1/2/4/8 B200 vs ref CPU"
MODEL = "llama3-8b"
SEQ = 8192
PER_GPU_BATCH = 8


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=4)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--model", default=MODEL)
    p.add_argument("--seq", type=int, default=SEQ)
    p.add_argument("--layers", type=int, default=0, help="debug only: truncate the model (the result is then marked invalid)")
    p.add_argument("--strategy", default=None, help="strategy JSON path (default: configs/ for this N)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                   help="fused: AdamW inside the gradient reduce-scatter kernel; torch: torch.optim.AdamW(fused=True) on fp32 grads")
    p.add_argument("--checkpoint-layers", type=int, default=-1, help="override: checkpoint the first k layers")
    p.add_argument("--legs", default="auto", help="auto (all path legs at N >= 2), none, or a comma-separated list of leg names")
    p.add_argument("--leg", default=None, help="internal: run ONE path leg in this process (spawned per rank by the headline run)")
    p.add_argument("--leg-port", type=int, default=0, help="internal: rendezvous port of the leg")
    p.add_argument("--kernel-breakdown", default="", help="write a per-kernel time table (torch.profiler/CUPTI, ONE extra untimed step "
                   "after the measurements; shares only, never a bench value) to this JSON file")
    p.add_argument("--ncu-step", action="store_true", help="profiling only: after the warm-up run ONE step between cudaProfilerStart/Stop "
                   "(ncu --profile-from-start off captures exactly that step) and exit without a bench line")
    p.add_argument("--total-budget-s", type=float, default=760.0, help="wall-clock budget of the whole bench.py run (legs are skipped beyond it)")
    p.add_argument("--no-probe", action="store_true")
    p.add_argument("--legs-only", action="store_true", help="debug: skip the headline run, run the path legs only (prints {\"path_legs\": ...})")
    p.add_argument("--dump-outputs", default=None, metavar="DIR",
                   help="after the timed steps, write what the last timed step returned (its loss, a fixed seeded sample of the fp32 "
                        "master weights its optimizer update wrote) as DIR/<name>.npy, to compare two builds output for output")
    opts = p.parse_args()
    if opts.steps < 1:
        p.error("--steps must be at least 1")
    return opts


def strategy_for(n_gpus, path=None):
    path = path or os.path.join(ROOT, "configs", "galvatron_config_llama3-8b_%dgpus.json" % n_gpus)
    with open(path) as f:
        return path, json.load(f)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "MEASURED_PEAKS.json bf16_tflops_sustained (measured)"
    return 1400.0, "B200_PROFILING.md fallback (sustained ~1.4 PFLOP/s)"


def ncu_gemm_traffic(flops_per_launch_avg):
    """DRAM bytes per (average) GEMM launch from the committed `ncu --set full` capture: the capture holds three launches of
    known shape; their bytes-per-FLOP ratio is applied to the average launch of the timed region."""
    path = os.path.join(ROOT, "profiles", "r01_ncu_gemm_full_summary.json")
    try:
        with open(path) as f:
            launches = json.load(f)["launches"]
        to_bytes = lambda s: float(s.split()[0]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[s.split()[1]]  # noqa: E731
        total = sum(to_bytes(l["dram__bytes_read.sum"]) + to_bytes(l["dram__bytes_write.sum"]) for l in launches)
        # the three captured launches: gate/up dgrad [8192x28672]x[28672x4096], o-proj wgrad and dgrad [8192|4096 x 4096 x 4096|8192]
        flops = 2.0 * 8192 * 4096 * (28672 + 4096 + 4096)
        return round(total / flops * flops_per_launch_avg), ("dram__bytes_read+write of 3 captured launches (profiles/r01_ncu_gemm_full_summary.json) "
                                                            "scaled by FLOPs to the average launch of this run")
    except Exception:  # noqa: BLE001
        return None, "no ncu capture found"


# ---------------------------------------------------------------------------------------------------------------------
def family_of(model):
    return "gpt" if model.startswith("gpt") else "bert" if model.startswith("bert") else "llama"


def build_model(opts, strategy, backend=None):
    import torch
    from hetu_galvatron_b200.core.runtime.arguments import initialize_galvatron
    family = family_of(opts.model)
    if family == "llama":
        from hetu_galvatron_b200.llama_hf import config_from_meta, llama_model_hp as model_hp, set_model_config
        from hetu_galvatron_b200.llama_hf.meta_configs import _SPECS
        seq_key, layers_key = "n_positions", "n_layers"
    elif family == "gpt":      # galvatron/models/gpt_hf (BASELINE.json configs 1 and 3)
        from hetu_galvatron_b200.gpt_hf import config_from_meta, gpt_model_hp as model_hp, set_model_config
        from hetu_galvatron_b200.gpt_hf.meta_configs import _SPECS
        seq_key, layers_key = "n_positions", "n_layer"
    else:                      # galvatron/models/bert_hf (BASELINE.json config 4: the sequence length is forced, set_seqlen_manually)
        from hetu_galvatron_b200.bert_hf import bert_model_hp as model_hp, config_from_meta, set_model_config
        from hetu_galvatron_b200.bert_hf.meta_configs import _SPECS
        seq_key, layers_key = "max_position_embeddings", "num_hidden_layers"
    spec = dict(_SPECS[opts.model], **{seq_key: opts.seq})
    if opts.layers:
        spec[layers_key] = opts.layers
        n = opts.layers
        for key in ("tp_sizes_enc", "tp_consecutive_flags", "dp_types_enc", "use_sp", "checkpoint", "cp_sizes_enc"):
            if key in strategy:
                strategy[key] = ",".join(strategy[key].split(",")[:n])
        if "pp_division" in strategy:
            pp = strategy["pp_deg"]
            strategy["pp_division"] = ",".join([str(n // pp)] * (pp - 1) + [str(n - n // pp * (pp - 1))])
    if getattr(opts, "checkpoint_layers", -1) >= 0:
        n_l = len(strategy["tp_sizes_enc"].split(","))
        strategy["checkpoint"] = ",".join(["1"] * min(opts.checkpoint_layers, n_l) + ["0"] * max(0, n_l - opts.checkpoint_layers))
    args = initialize_galvatron(galvatron_config_path=strategy, mixed_precision="bf16", fused_optimizer=getattr(opts, "optimizer", "torch") == "fused", sequence_parallel=bool(strategy.get("sequence_parallel", 0)),
                                use_ulysses=False, init_method_std=0.02, seed=1234, local_rank=1, lr=1e-4, adam_weight_decay=0.01,
                                make_vocab_size_divisible_by=128, vocab_tp=strategy.get("vtp", 1), model_size=opts.model,
                                default_dp_type=strategy.get("default_dp_type", "zero2"), chunks=strategy["chunks"],
                                global_train_batch_size=strategy["global_bsz"], pp_deg=strategy["pp_deg"],
                                # (this runtime's key, next to the Search Engine's: the memory profile the strategy was searched with
                                # assumed the SwiGLU / RMSNorm outputs are recomputed in backward instead of saved)
                                recompute_activations=bool(strategy.get("recompute_activations", 0)))
    args.vocab_size = spec["vocab_size"]
    config = set_model_config(config_from_meta(spec), args)
    model = model_hp(config, args)
    return args, config, model


def synthetic_batches(args, config, n_steps, dp_idx, dp_size, pin):
    """DataLoaderForLlama semantics (models/llama_hf/dataloader.py:52-80), seed 1234, this rank's data-parallel slice."""
    import numpy as np
    import torch
    rng = np.random.RandomState(1234)
    gbs, seq = args.global_train_batch_size, config.max_position_embeddings
    out = []
    for _ in range(n_steps):
        lengths = rng.randint(1, seq + 1, (gbs,))
        ids = rng.randint(0, config.vocab_size, (gbs, seq + 1))
        ids[np.arange(seq + 1)[None, :] >= lengths[:, None]] = 0
        lo, hi = dp_idx * gbs // dp_size, (dp_idx + 1) * gbs // dp_size
        x = torch.from_numpy(ids[lo:hi]).long()
        tokens, labels = x[:, :-1].contiguous(), x[:, 1:].contiguous()
        if pin:
            tokens, labels = tokens.pin_memory(), labels.pin_memory()
        out.append((tokens, labels))
    return out


def bert_batch(tokens, labels, vocab_size):
    """DataLoaderForBert semantics (models/bert_hf/dataloader.py:24-120) on top of the seeded token stream: the zero tail of every
    sample is padding (attention mask 0), the second half of the visible part is segment B, 15 % of the visible tokens carry an
    MLM label (-100 elsewhere)."""
    import torch
    g = torch.Generator().manual_seed(int(tokens[0, :8].sum()) + 7)
    seq = tokens.shape[1]
    lengths = (tokens != 0).long().cumsum(1).argmax(1) + 1          # last non-zero position + 1 (padding is the zero tail)
    lengths = lengths.clamp(min=8)
    pos = torch.arange(seq)[None, :]
    mask = pos < lengths[:, None]
    token_type = ((pos >= (lengths[:, None] // 2)) & mask).long()
    mlm = torch.where((torch.rand(tokens.shape, generator=g) < 0.15) & mask, tokens, torch.full_like(tokens, -100))
    return tokens, mlm, mask, token_type


NVLINK_NOMINAL_GBS, NVLINK_MEASURED_GBS = 900.0, 770.0    # per direction per GPU; measured = peer copy (B200_PROFILING.md)
T_START = time.time()


def fixed_probe_batch(config, per_rank):
    """The probe's batch: ``per_rank`` sequences, the same on every rank and at every N (generator seed 4321)."""
    import numpy as np
    import torch
    rng = np.random.RandomState(4321)
    seq = config.max_position_embeddings
    lengths = rng.randint(seq // 2, seq + 1, (per_rank,))
    ids = rng.randint(0, config.vocab_size, (per_rank, seq + 1))
    ids[np.arange(seq + 1)[None, :] >= lengths[:, None]] = 0
    x = torch.from_numpy(ids).long()
    return x[:, :-1].contiguous(), x[:, 1:].contiguous()


def reduction_checksum(model, step_fn, world):
    """Checksum of checksums of the gradient reduction at FULL size (N >= 2): one extra step with the optimizer epilogue
    switched off, so that every unit's reduce-scatter / all-reduce leaves its fp32 result; then, per unit and summed over the
    job,  sum(reduced shards) must equal sum(unsharded bf16 gradients) * prescale * postscale (= / d).  Linear in the data,
    independent of the size, exact up to fp32 rounding of the sums."""
    import torch
    import torch.distributed as dist
    units = list(model.model.units)
    saved = [(u, u.fused_opt) for u in units]
    for u in units:
        u.fused_opt = None
    try:
        step_fn()
        torch.cuda.synchronize()
        rows = []
        for u in units:
            d = u.group.size
            g_in = u.g_flat.double()
            s_in, a_in = g_in.sum() / d, g_in.abs().sum() / d
            red = u.master_grad.double()
            s_out = red.sum() / (d if u.dp_type == "ddp" else 1)
            rows.append(torch.stack([s_in, s_out, a_in]))
        t = torch.stack(rows)
        dist.all_reduce(t)
        rel = ((t[:, 0] - t[:, 1]).abs() / t[:, 2].clamp_min(1e-30))
        worst = int(rel.argmax())
        return {"units": len(units), "max_rel_discrepancy": float(rel.max()), "worst_unit": units[worst].name,
                "ok": bool(rel.max() < 2e-4), "what": "sum_ranks(sum(reduced fp32 shard)) vs sum_ranks(sum(bf16 unsharded grads))/d, relative to sum|g|/d"}
    finally:
        for u, f in saved:
            u.fused_opt = f
            u._master_grad = None
            u.flat_param.grad = None
        torch.cuda.empty_cache()


def summarize_comm(prof, steps):
    """{kind: calls/step, ms/step, achieved bus GB/s (nccl-tests convention), fraction of 900 nominal / 770 measured}.  Times are
    CUDA-event spans of each call ON ITS STREAM, launch to completion: they include waiting for the slowest peer to arrive and the
    SM sharing with whatever compute runs beside the collective (side-stream collectives are hidden behind the GEMMs on purpose), so
    these are in-step figures, below the stand-alone rates of profiles/r02_collectives_*gpu.jsonl.  A fused GEMM + collective is
    judged against its own roofline: the slower of FLOPs / measured GEMM peak and NVLink bytes / 770 GB/s."""
    peak, _ = measured_peaks()
    out = {}
    for kind, recs in sorted(prof.items()):
        ms = sum(r[0].elapsed_time(r[1]) for r in recs)
        nbytes = sum(r[2] for r in recs)
        flops = sum(r[3] for r in recs) if len(recs[0]) > 3 else 0.0
        gbs = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        out[kind] = {"calls_per_step": round(len(recs) / steps, 1), "ms_per_step": round(ms / steps, 3), "bus_bytes_per_step": int(nbytes / steps),
                     "bus_GBps": round(gbs, 1), "frac_of_900_nominal": round(gbs / NVLINK_NOMINAL_GBS, 3),
                     "frac_of_770_measured": round(gbs / NVLINK_MEASURED_GBS, 3)}
        if flops > 0 and ms > 0:
            bound_ms = sum(max(r[3] / (peak * 1e12), r[2] / (NVLINK_MEASURED_GBS * 1e9)) for r in recs) * 1e3
            out[kind].update({"tflops": round(flops / (ms * 1e-3) / 1e12, 1), "roofline_ms_per_step": round(bound_ms / steps, 3),
                              "frac_of_fused_roofline": round(bound_ms / ms, 3)})
    return out


def kernel_breakdown(step_fn, path, ms_per_step):
    """Where one step goes, kernel by kernel: a CUPTI trace of ONE extra step (after all timed regions).  Taken under a profiler, so
    only the shares are meaningful; the step time they are compared with is the CUDA-event one."""
    import collections
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step_fn()
        torch.cuda.synchronize()
    agg = collections.defaultdict(lambda: [0, 0.0])
    for ka in prof.key_averages():
        us = getattr(ka, "self_device_time_total", None)
        if us is None:
            us = getattr(ka, "self_cuda_time_total", 0.0)
        if us > 0:
            a = agg[ka.key[:110]]
            a[0] += ka.count
            a[1] += us
    rows = sorted(([n, c, round(us / 1e3, 3)] for n, (c, us) in agg.items()), key=lambda r: -r[2])
    total = sum(r[2] for r in rows)
    with open(path, "w") as f:
        json.dump({"what": "torch.profiler (CUPTI) kernel times of one training step; kernels on side streams overlap, so the sum may "
                           "exceed the step", "event_timed_ms_per_step": round(ms_per_step, 3), "sum_kernel_ms": round(total, 3),
                   "kernels": [{"name": n, "launches": c, "ms": ms, "share_of_sum": round(ms / total, 4)} for n, c, ms in rows[:60]]}, f, indent=1)


DUMP_WEIGHT_BYTES = 48 << 20     # fp32 weight samples of --dump-outputs, all units together (the files stay under 64 MB)


def dump_outputs(path, model, loss):
    """--dump-outputs: what the last timed step handed back to its caller on this rank -- ``loss.npy`` (float64; absent on a
    pipeline stage without the loss) and, per optimizer-facing parameter (the fp32 flat master of one unit, this rank's shard),
    ``<name>.npy``: its values at a fixed sample of positions (seed 0, sorted, the whole tensor when it is small enough).
    The inputs are the same on every run, but the step is not bit-reproducible (the order of some fp32 accumulations varies), so
    compare with a tolerance: two runs of one build (B200, 1000 W power limit, --steps 2 --warmup 1) gave losses 4e-5 apart (relative)."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    if loss is not None:
        np.save(os.path.join(path, "loss.npy"), np.array([loss], dtype=np.float64))
    params = list(model.named_parameters())
    per_param = DUMP_WEIGHT_BYTES // 4 // max(1, len(params))
    gen = torch.Generator().manual_seed(0)
    for name, p in params:
        flat = p.detach().reshape(-1)
        if flat.numel() > per_param:
            idx = torch.randint(flat.numel(), (per_param,), generator=gen).sort().values
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(path, name + ".npy"), flat.float().cpu().numpy())


def run_ours(opts):
    os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")   # 150+ GiB of long-lived state: avoid fragmentation
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    assert world == opts.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (opts.gpus, world)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)   # bootstrap only (handles, barriers)
    from hetu_galvatron_b200.core.runtime.backend import get_backend, reset_backend
    from hetu_galvatron_b200.core.runtime.utils import get_optimizer_and_param_scheduler
    if opts.legs_only:
        legs = run_path_legs(opts, rank, world, local) if world > 1 else []
        if rank == 0:
            print(json.dumps({"invalid": "--legs-only: no headline measurement", "n_gpus": world, "path_legs": legs}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    spath, strategy = strategy_for(world, opts.strategy)
    args, config, model = build_model(opts, strategy)
    be = get_backend()
    opt, _ = get_optimizer_and_param_scheduler(model, args)
    dp_group = model.vtp_data_group
    dp_idx, dp_size = dp_group.rank_in_group(rank), dp_group.size
    K, W = opts.steps, opts.warmup
    host = synthetic_batches(args, config, 2 * K + W + 1, dp_idx, dp_size, pin=True)
    tokens_per_step = args.global_train_batch_size * config.max_position_embeddings

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step(tokens, labels, it):
        loss = model.forward_backward([tokens], it, None, loss_func=None, attention_mask=None, labels=labels)
        opt.step()
        opt.zero_grad()
        return loss

    it = 0
    # ---- probe: N-invariant losses on a fixed batch, then (N >= 2) the full-size checksum of the gradient reduction -------
    probe = None
    if not opts.no_probe:
        pt, pl = fixed_probe_batch(config, args.global_train_batch_size // dp_size)
        pt, pl = pt.to(dev), pl.to(dev)
        l0 = step(pt, pl, it); it += 1
        l1 = step(pt, pl, it); it += 1
        probe = {"fixed_batch": "%d sequences, seed 4321, identical on every rank and at every N" % pt.shape[0],
                 "loss_at_init": l0, "loss_after_one_update": l1, "finite": bool(l0 == l0 and l1 == l1)}
        if world > 1:
            both = torch.tensor([l0 if l0 is not None else 0.0, l1 if l1 is not None else 0.0], dtype=torch.float64, device=dev)
            lo, hi = both.clone(), both.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            probe["max_spread_over_ranks"] = float((hi - lo).abs().max())
            t, l = host[-1]
            probe["reduction_checksum"] = reduction_checksum(
                model, lambda: model.forward_backward([t.to(dev)], it, None, loss_func=None, attention_mask=None, labels=l.to(dev)), world)
    for i in range(W):                                         # warm-up (untimed)
        t, l = host[i]
        step(t.to(dev, non_blocking=True), l.to(dev, non_blocking=True), it); it += 1

    if opts.ncu_step:
        t, l = host[W]
        t, l = t.to(dev), l.to(dev)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step(t, l, it)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        if rank == 0:
            print(json.dumps({"ncu_step": True, "model": opts.model, "layers": config.num_hidden_layers, "note": "not a bench line"}))
        return

    def timed(resident):
        nonlocal it
        batches = host[W:W + K] if resident else host[W + K:W + 2 * K]
        if resident:
            batches = [(t.to(dev), l.to(dev)) for t, l in batches]
        sync_all()
        launches0 = be.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for t, l in batches:
            if not resident:
                t, l = t.to(dev, non_blocking=True), l.to(dev, non_blocking=True)
            last = step(t, l, it); it += 1                      # forward_backward returns the loss as a python float (D2H read)
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms[0])
        return ms, be.launch_count() - launches0, last

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    be.gemm_profile = []
    ms_res, launches, loss_res = timed(resident=True)
    prof, be.gemm_profile = be.gemm_profile, None
    ms_e2e, _, loss_e2e = timed(resident=False)
    clocks = sampler.stop() if rank == 0 else None
    if opts.dump_outputs and rank == 0:
        dump_outputs(opts.dump_outputs, model, loss_e2e)
    # one more step with every collective bracketed by CUDA events on its own stream: the in-step NVLink roofline
    be.comm_profile = {}
    t, l = host[W]
    step(t.to(dev), l.to(dev), it); it += 1
    torch.cuda.synchronize()
    comm, be.comm_profile = summarize_comm(be.comm_profile, 1), None
    if opts.kernel_breakdown and rank == 0:
        kernel_breakdown(lambda: step(t.to(dev), l.to(dev), it), opts.kernel_breakdown, ms_res / K)
    gemm_ms = sum(rec[0].elapsed_time(rec[1]) for rec in prof)
    gemm_flops = sum(rec[2] for rec in prof)
    gemm_bytes = sum(rec[3] for rec in prof)
    traffic, traffic_note = ncu_gemm_traffic(gemm_flops / max(1, len(prof)))
    peak, peak_src = measured_peaks()
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    h2d = 2 * (args.global_train_batch_size // dp_size) * config.max_position_embeddings * 8
    value = tokens_per_step * K / (ms_res * 1e-3)
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(ms_res / K, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic tokens (DataLoaderForLlama generator, seed 1234), random-init weights",
        "config": {"workload": "%s seq %d, global_bsz %d, strategy %s" % (opts.model, config.max_position_embeddings,
                                                                       args.global_train_batch_size, os.path.basename(spath)),
                   "strategy": {k: strategy[k] for k in ("pp_deg", "chunks", "default_dp_type", "global_bsz") if k in strategy},
                   "tp": sorted(set(strategy["tp_sizes_enc"].split(","))), "checkpointed_layers": strategy.get("checkpoint", "").count("1"),
                   "layers": config.num_hidden_layers, "l2": "inputs (16 GB of bf16 weights + activations per step) far exceed the 126 MB L2",
                   "optimizer": ("AdamW fused into the gradient reduce-scatter kernel (fp32 shards)" if opts.optimizer == "fused"
                                 else "torch.optim.AdamW(fused=True) on fp32 flat shards"),
                   "collectives": "slim peer-memory kernels (128 thr x <=64 regs, one CTA per SM)%s; no NCCL on the path"
                                  % (", NVLS multicast for buffers in a bound arena range" if getattr(be, "nvls", False) else "")},
        "e2e": {"value": round(tokens_per_step * K / (ms_e2e * 1e-3), 1), "unit": "tokens/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4 * max(1, strategy["chunks"]), "ms_per_step": round(ms_e2e / K, 3)},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "achieved": round(achieved, 1), "peak": peak, "unit": "TFLOP/s",
                     "frac": round(achieved / peak, 4) if peak else None, "traffic": traffic, "traffic_note": traffic_note,
                     "algorithmic_bytes_per_launch_avg": gemm_bytes / max(1, len(prof)), "kernel": "gemm_bf16_kernel (tcgen05/TMEM/TMA)",
                     "launches": len(prof), "kernel_ms_per_step": round(gemm_ms / K, 3), "share_of_step": round(gemm_ms / ms_res, 4),
                     "flops_per_launch_avg": gemm_flops / max(1, len(prof)), "peak_source": peak_src},
        "collectives_in_step": comm,
        "clocks": clocks, "loss": {"resident": loss_res, "e2e": loss_e2e}, "probe": probe,
        "memory_gib": {"torch_peak_allocated": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2),
                       "torch_peak_reserved": round(torch.cuda.max_memory_reserved() / 2 ** 30, 2),
                       "arena": round(be.comm.arena_bytes / 2 ** 30, 2)},
    }
    if opts.layers:
        line["invalid"] = "debug run with --layers %d: not the BASELINE workload" % opts.layers
    # ---- release the GPU, then the path legs (N >= 2) or the CPU baseline (N = 1) ------------------------------------------
    del model, opt, host, prof
    reset_backend()
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    if world > 1 and opts.legs != "none":
        try:
            line["path_legs"] = run_path_legs(opts, rank, world, local)
        except Exception as exc:  # noqa: BLE001 -- the headline line must be printed whatever happens to a leg
            line["path_legs"] = [{"error": "%s: %s" % (type(exc).__name__, exc)}]
    if rank == 0 and world == 1 and not opts.no_cpu_baseline:
        line["cpu_baseline"] = cpu_reference_sample(opts)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# path legs: fixed-strategy runs of the collectives north_star names, one child process per rank and leg
# ---------------------------------------------------------------------------------------------------------------------
def leg_catalog(n):
    """name -> {model, strategy (Galvatron JSON, as the Search Engine would write it), tiny (the same strategy for the tiny model of
    tests/_host_worker.py), expect (fused-kernel counters that must be > 0)}"""
    def enc(v, layers=32):
        return ",".join([str(v)] * layers)

    def strat(layers=32, **kw):
        d = {"pp_deg": 1, "tp_sizes_enc": enc(1, layers), "tp_consecutive_flags": enc(1, layers), "dp_types_enc": enc(0, layers),
             "use_sp": enc(0, layers), "checkpoint": enc(0, layers), "cp_sizes_enc": enc(1, layers), "global_bsz": 8, "chunks": 2,
             "pp_division": str(layers), "pipeline_type": "pipedream_flush", "default_dp_type": "zero2", "vtp": 1, "vsp": 0, "embed_sdp": 0}
        d.update(kw)
        return d
    # tiny model whose GEMMs meet the fused kernels' shape rule (M = seq x microbatch a multiple of p x 128) at this p
    heads = max(4, n)
    spec = {"n_positions": 128 * n, "n_heads": heads, "n_kv_heads": max(2, n), "ffn_dim": 384, "dim": 128 if n < 8 else 256}
    legs = {}
    legs["tp%d_megatron_sp" % n] = dict(
        model="llama3-8b", strategy=strat(tp_sizes_enc=enc(n), vtp=n, sequence_parallel=1),
        tiny=dict(global_tp_deg=n, vocab_tp=n, sequence_parallel=True, chunks=2, _spec=spec,
                  _env={"HGB_FUSE_GEMM_RS": "force", "HGB_FUSE_GEMM_AR": "force"}),
        expect=["ag_gemm", "gemm_rs"], what="C7/C8/C9: all-gather+GEMM and GEMM+reduce-scatter fused (layers.py:399-417,1061-1109,449-494)")
    legs["tp%d" % n] = dict(
        model="llama3-8b", strategy=strat(tp_sizes_enc=enc(n), vtp=n, sequence_parallel=0),
        tiny=dict(global_tp_deg=n, vocab_tp=n, chunks=2, _spec=spec, _env={"HGB_FUSE_GEMM_AR": "force"}),
        expect=["gemm_ar"], what="C5/C6: GEMM+all-reduce fused, NVLS broadcast (layers.py:1110-1114, mappings_group.py:139)")
    legs["ulysses%d" % n] = dict(
        model="llama3-8b", strategy=strat(tp_sizes_enc=enc(n), use_sp=enc(1), vtp=n, vsp=1, sequence_parallel=1),
        tiny=dict(global_tp_deg=n, vocab_tp=n, use_ulysses=True, sequence_parallel=True, chunks=2, _spec=spec),
        expect=[], what="C10: Ulysses all-to-all, q/k/v in one launch (transformer.py:1928-2062)")
    t2 = max(1, n // 2)
    legs["pp2_tp%d_1f1b" % t2] = dict(
        model="llama3-8b", strategy=strat(pp_deg=2, tp_sizes_enc=enc(t2), vtp=t2, sequence_parallel=1 if t2 > 1 else 0, chunks=4,
                                          pp_division="16,16"),
        tiny=dict(pp_deg=2, global_tp_deg=t2, vocab_tp=t2, sequence_parallel=t2 > 1, chunks=4, pipeline_type="pipedream_flush",
                  global_train_batch_size=8, _spec=dict(spec, n_positions=128 * t2)),
        expect=[], what="C11: 1F1B-flush schedule, stage boundary = peer copy on a side stream + device flags (pipeline.py:375-701,1080-1257)")
    legs["zero3_ckpt_dp%d" % n] = dict(
        model="llama3-8b", strategy=strat(dp_types_enc=enc(1), checkpoint=enc(1), global_bsz=2 * n, chunks=1, default_dp_type="zero3", embed_sdp=1),
        tiny=dict(sdp=1, global_checkpoint=1, embed_sdp=1, chunks=1, global_train_batch_size=2 * n, zero3_pool_slots=2),
        expect=[], what="C1/C2: ZeRO-3 all-gather (fwd + bwd re-gather) and reduce-scatter+AdamW per layer, pooled buffers, prefetch")
    # BASELINE.json config 3: GPT-3 6.7B, fixed strategy PP=2 x TP=2 x ZeRO-2 data parallel 2, 1F1B-flush (N = 8; PP2 x TP(N/2) below)
    d3 = 2 if n == 8 else 1
    t3 = max(1, n // (2 * d3))
    legs["gpt-6.7b_pp2_tp%d_zero2dp%d_1f1b" % (t3, d3)] = dict(
        model="gpt-6.7b", seq=2048,
        strategy=strat(pp_deg=2, tp_sizes_enc=enc(t3), vtp=t3, global_bsz=8 * d3, chunks=4, pp_division="16,16", default_dp_type="zero2"),
        tiny=dict(_family="gpt", pp_deg=2, global_tp_deg=t3, vocab_tp=t3, default_dp_type="zero2", chunks=4, pipeline_type="pipedream_flush",
                  global_train_batch_size=8, _spec=dict(n_positions=128 * t3, n_head=max(4, t3))),
        expect=[], what="BASELINE config 3: GPT-3 6.7B (gpt_hf family: LayerNorm, bias, GeLU, learned positions), PP2 x TP x ZeRO-2, 1F1B-flush")
    # BASELINE.json config 4: BERT-large, Ulysses-SP 4 x DP 2, sequence length forced to 8192 (N = 8; Ulysses-SP N below)
    s4 = 4 if n == 8 else n
    d4 = n // s4
    legs["bert-large_ulysses%d_dp%d_seq8192" % (s4, d4)] = dict(
        model="bert-large", seq=8192,
        strategy=strat(layers=24, tp_sizes_enc=enc(s4, 24), use_sp=enc(1, 24), vtp=s4, vsp=1, sequence_parallel=1, global_bsz=4 * d4, chunks=2),
        tiny=dict(_family="bert", global_tp_deg=s4, use_ulysses=True, sequence_parallel=True, vocab_tp=s4, default_dp_type="zero2", chunks=2,
                  global_train_batch_size=4 * d4, _spec=dict(max_position_embeddings=64 * s4, num_attention_heads=max(4, s4))),
        expect=[], what="BASELINE config 4: BERT-large (bert_hf family: post-LN, non-causal attention with a padding mask, MLM head), "
                        "Ulysses all-to-all x data parallel, seq 8192")
    if n == 8:
        legs["llama3-70b_zero3_ckpt_dp8"] = dict(
            model="llama3-70b", strategy=strat(layers=80, dp_types_enc=enc(1, 80), checkpoint=enc(1, 80), global_bsz=8, chunks=1,
                                               default_dp_type="zero3", embed_sdp=1),
            tiny=None, expect=[], what="BASELINE config 5: Llama-3-70B SDP=8 ZeRO-3 + activation checkpointing (>= 0.40 s/step of NVLink time)")
    if n == 8:      # config 5 before configs 3 and 4: if the wall-clock budget runs out, the later legs are the ones skipped
        order = [k for k in legs if not k.startswith(("gpt-", "bert-"))] + [k for k in legs if k.startswith(("gpt-", "bert-"))]
        legs = {k: legs[k] for k in order}
    return legs


def _child_env(rank, world, local, port):
    env = {k: v for k, v in os.environ.items() if not k.startswith("TORCHELASTIC") and k not in ("GROUP_RANK", "ROLE_RANK", "ROLE_NAME",
                                                                                                  "GROUP_WORLD_SIZE", "ROLE_WORLD_SIZE")}
    env.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(local), LOCAL_WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
               MASTER_PORT=str(port))
    return env


def run_path_legs(opts, rank, world, local):
    """Every rank spawns ITS process of each leg (the leg's ranks rendezvous on their own port); rank 0 keeps the leg's JSON line.
    The parent ranks stay in step through the bootstrap group; a leg that fails, hangs past its limit or would overrun the
    wall-clock budget is recorded and skipped -- by the same decision on every rank."""
    import torch
    import torch.distributed as dist
    catalog = leg_catalog(world)
    names = list(catalog) if opts.legs == "auto" else [n for n in opts.legs.split(",") if n in catalog]
    base_port = int(os.environ.get("MASTER_PORT", "29500")) + 11
    results = []
    for i, name in enumerate(names):
        limit = 300.0 if "70b" in name else 170.0
        decision = [None]
        if rank == 0:
            left = opts.total_budget_s - (time.time() - T_START)
            decision[0] = "run" if left > limit * 0.6 + 20 else "skipped: %.0f s of the %.0f s budget left" % (left, opts.total_budget_s)
        dist.broadcast_object_list(decision, src=0)
        if decision[0] != "run":
            results.append({"leg": name, "status": decision[0]})
            continue
        cmd = [sys.executable, os.path.abspath(__file__), "--leg", name, "--gpus", str(world), "--steps", "3", "--warmup", "2",
               "--leg-port", str(base_port + 3 * i)]
        t0 = time.time()
        proc = subprocess.Popen(cmd, env=_child_env(rank, world, local, base_port + 3 * i), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        try:
            out, err = proc.communicate(timeout=limit)
            status = "ok" if proc.returncode == 0 else "failed rc=%d" % proc.returncode
        except subprocess.TimeoutExpired:
            proc.kill()                      # exactly the child this rank started
            out, err = proc.communicate()
            status = "killed after %.0f s" % limit
        rec = {"leg": name, "status": status, "what": catalog[name]["what"], "wall_s": round(time.time() - t0, 1)}
        if rank == 0:
            for ln in out.splitlines():
                if ln.startswith("LEG_JSON "):
                    try:
                        rec.update(json.loads(ln[len("LEG_JSON "):]))     # the last complete line wins (perf first, then + parity)
                    except ValueError:
                        pass
            if status != "ok":
                rec["stderr_tail"] = err[-600:]
        # every rank's verdict: a leg counts as ok only if all its ranks exited cleanly
        flag = torch.tensor([1 if status == "ok" else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag[0]) == 0 and status == "ok":
            rec["status"] = "failed on another rank"
        results.append(rec)
    return results


def run_leg(opts):
    """One path leg, one process per GPU (spawned by ``run_path_legs``).  Prints ``LEG_JSON {...}`` on rank 0: first the
    performance part, then again with the tiny-model parity verdict added."""
    os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    leg = leg_catalog(world)[opts.leg]
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from hetu_galvatron_b200.core.runtime.backend import get_backend, reset_backend
    from hetu_galvatron_b200.core.runtime.utils import get_optimizer_and_param_scheduler
    strategy = dict(leg["strategy"])
    lopts = argparse.Namespace(**vars(opts))
    lopts.model, lopts.layers, lopts.checkpoint_layers, lopts.optimizer = leg["model"], 0, -1, "fused"
    lopts.seq = leg.get("seq", opts.seq)
    family = family_of(leg["model"])
    # a leg exists to put its kernels under the driver's eyes: the fused GEMM + collective kernels are forced on for the legs that name
    # them, also at the shapes where the runtime's measured rule (backend.FUSE_MIN_K / FUSE_AR_MIN_K) would pick the unfused pair
    for k, v in ((leg.get("tiny") or {}).get("_env") or {}).items():
        os.environ[k] = v
    t_build = time.time()
    args, config, model = build_model(lopts, strategy)
    be = get_backend()
    be.bg.set_tunable("timeout_ms", 45000)
    opt, _ = get_optimizer_and_param_scheduler(model, args)
    torch.cuda.synchronize()
    build_s = time.time() - t_build
    dp_group = model.vtp_data_group
    dp_idx, dp_size = dp_group.rank_in_group(rank), dp_group.size
    K, W = opts.steps, opts.warmup
    host = synthetic_batches(args, config, K + W + 1, dp_idx, dp_size, pin=False)
    if family == "bert":
        host = [bert_batch(t, l, config.vocab_size) for t, l in host]
    tokens_per_step = args.global_train_batch_size * config.max_position_embeddings
    it, losses = 0, []

    def step(i):
        nonlocal it
        t, l = host[i][:2]
        extra = dict(attention_mask=None) if family != "bert" else dict(attention_mask=host[i][2].to(dev), token_type_ids=host[i][3].to(dev))
        loss = model.forward_backward([t.to(dev)], it, None, loss_func=None, labels=l.to(dev), **extra)
        opt.step(); opt.zero_grad()
        it += 1
        return loss

    for i in range(W):
        losses.append(step(i))
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    launches0 = be.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(W, W + K):
        losses.append(step(i))
    e1.record()
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    tms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms[0])
    launches = be.launch_count() - launches0
    be.comm_profile = {}
    step(W + K)
    torch.cuda.synchronize()
    comm, be.comm_profile = summarize_comm(be.comm_profile, 1), None
    lt = torch.tensor([[x if x is not None else 0.0, 1.0 if x is not None else 0.0] for x in losses], dtype=torch.float64, device=dev)
    dist.all_reduce(lt)                     # the last pipeline stage holds the loss; average the data-parallel replicas
    mean_losses = [round(float(a / max(b, 1.0)), 5) for a, b in lt.tolist()]
    rec = {"model": leg["model"], "seq": config.max_position_embeddings, "global_bsz": args.global_train_batch_size,
           "strategy": {k: (strategy[k] if not isinstance(strategy[k], str) or len(strategy[k]) < 12 else strategy[k].split(",")[0] + " x%d" % len(strategy[k].split(",")))
                        for k in ("pp_deg", "tp_sizes_enc", "use_sp", "dp_types_enc", "checkpoint", "chunks", "default_dp_type", "vtp", "vsp", "sequence_parallel") if k in strategy},
           "tokens_per_s": round(tokens_per_step * K / (ms * 1e-3), 1), "ms_per_step": round(ms / K, 3), "steps": K, "warmup": W,
           "gpu_launches": int(launches), "fused_calls": dict(getattr(be, "n_fused", {})), "nvls_groups": len(getattr(be, "nvls_regions", {}) or {}),
           "collectives": comm, "losses": mean_losses, "build_s": round(build_s, 1),
           "memory_gib": {"torch_peak_allocated": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2), "arena": round(be.comm.arena_bytes / 2 ** 30, 2)},
           "expect_ok": all(getattr(be, "n_fused", {}).get(k, 0) > 0 for k in leg["expect"]), "device_error_flag": be.comm.error_flag()}
    if rank == 0:
        print("LEG_JSON " + json.dumps(rec), flush=True)
    del model, opt, host
    reset_backend()
    dist.barrier()
    dist.destroy_process_group()
    import gc
    gc.collect(); torch.cuda.empty_cache()
    # ---- the same strategy on the tiny model against the oracle (checker: tests/_host_worker.py) -----------------------------
    if leg["tiny"] is not None:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        tiny = dict(leg["tiny"])
        for k, v in tiny.pop("_env", {}).items():
            os.environ[k] = v
        os.environ.update(HOST_TEST_CONFIG=json.dumps(tiny), HOST_TEST_BACKEND="cuda", MASTER_PORT=str(opts.leg_port + 1))
        if family == "llama":
            import _host_worker as worker
        else:                       # checker of the GPT / BERT families: oracle/gpt_bert_ref.py (pinned to HF GPT-2 / BERT)
            import _family_worker as worker
        try:
            rep = worker.main()
            rec["parity"] = {"ok": True, "loss": rep.get("loss"), "oracle_loss": rep.get("ref_loss"), "max_grad_rel_l2": rep.get("max_grad_err"),
                             "worst": rep.get("worst"), "fused_calls": rep.get("fused_calls"), "nvls_groups": rep.get("nvls_groups"),
                             "criterion": "loss 5e-3 rel, every parameter's gradient 3e-2 rel-L2 vs oracle/%s (bf16)"
                                          % ("llama_ref.py" if family == "llama" else "gpt_bert_ref.py")}
        except BaseException as exc:  # noqa: BLE001
            import traceback
            rec["parity"] = {"ok": False, "error": ("%s: %s" % (type(exc).__name__, exc))[:400], "traceback_tail": traceback.format_exc()[-900:]}
        if rank == 0:
            print("LEG_JSON " + json.dumps(rec), flush=True)
        if not rec["parity"]["ok"]:
            sys.exit(3)


# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(opts, budget_s=25.0):
    """The CPU restatement of the reference path (oracle backend, all host threads) on a bounded sample of the workload:
    Llama-3-8B shapes, embedding + lm_head + ONE and then TWO transformer layers, seq 1024, batch 1.  The two samples separate
    the per-layer cost from the embedding/head cost; ``value`` is the full-depth (32-layer) tokens/s they imply -- an
    extrapolation that favours the CPU (seq 1024 instead of 8192: 8x less attention work per token), labelled as such, never a
    like-for-like 8B measurement (SURVEY 8d, BASELINE.md sec. 3)."""
    import torch
    from oracle.gloo_backend import OracleBackend
    from hetu_galvatron_b200.core.runtime.backend import reset_backend, set_backend
    from hetu_galvatron_b200.core.runtime.utils import get_optimizer_and_param_scheduler
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)

    def best_step(n_layers, budget):
        set_backend(OracleBackend())
        sample = argparse.Namespace(**vars(opts))
        sample.layers, sample.seq, sample.optimizer, sample.checkpoint_layers = n_layers, 1024, "torch", -1
        one = ",".join(["1"] * n_layers)
        zero = ",".join(["0"] * n_layers)
        strategy = {"pp_deg": 1, "tp_sizes_enc": one, "tp_consecutive_flags": one, "dp_types_enc": zero, "use_sp": zero,
                    "checkpoint": zero, "global_bsz": 1, "chunks": 1, "default_dp_type": "zero2", "vtp": 1}
        args, config, model = build_model(sample, strategy)
        opt, _ = get_optimizer_and_param_scheduler(model, args)
        batches = synthetic_batches(args, config, 4, 0, 1, pin=False)
        times, t_start = [], time.perf_counter()
        for i, (t, l) in enumerate(batches):
            t0 = time.perf_counter()
            model.forward_backward([t], i, None, loss_func=None, attention_mask=None, labels=l)
            opt.step(); opt.zero_grad()
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_start > budget and i >= 1:
                break
        reset_backend()
        timed_steps = sorted(times[1:]) if len(times) > 1 else times        # the first step pays for allocator / thread-pool warm-up
        return timed_steps[len(timed_steps) // 2], len(times), config.max_position_embeddings

    t1, n1, tok = best_step(1, budget_s * 0.4)
    t2, n2, _ = best_step(2, budget_s * 0.6)
    layer_s = max(t2 - t1, 0.05 * t1)
    other_s = max(t1 - layer_s, 0.0)
    full_layers = 32
    full_s = other_s + full_layers * layer_s
    return {"value": round(tok / full_s, 3), "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": "oracle CPU restatement (fp32 compute, bf16 storage), Llama-3-8B shapes, seq 1024, batch 1: embedding + lm_head + "
                      "1 layer (%d steps, median of the steps after the first %.2f s) and + 2 layers (%d steps, median %.2f s), intra-op threads "
                      "pinned to the host's cores -> %.2f s per layer, %.2f s for the rest; "
                      "value = 1024 tokens / (rest + 32 layers) = extrapolated full-depth rate, NOT a like-for-like seq-8192 run"
                      % (n1, t1, n2, t2, layer_s, other_s),
            "sample_tokens_per_s_1layer": round(tok / t1, 2)}


def run_reference(opts):
    """--impl reference: the reference's path as restated on CPU (the reference has no CPU runtime: SURVEY 8c / BASELINE.md 3),
    all host threads, rank 0 only."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    K = max(1, opts.steps)
    from hetu_galvatron_b200.core.runtime import world as _world
    with _world.simulated(0, 1):        # under torchrun the env says world N; the CPU sample is a single-process job
        base = cpu_reference_sample(opts, budget_s=20.0 * K)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "tokens/s", "n_gpus": opts.gpus, "steps": opts.steps,
            "warmup": opts.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16 storage / fp32 compute",
            "data": "synthetic tokens (DataLoaderForLlama generator, seed 1234), random-init weights",
            "config": {"workload": "%s seq %d (bounded sample: %s)" % (opts.model, opts.seq, base["sample"])},
            "cpu_baseline": base, "e2e": {"value": base["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "ms_per_step": None}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    o = parse()
    if o.impl == "reference":
        run_reference(o)
    elif o.leg:
        run_leg(o)
    else:
        try:
            run_ours(o)
        except Exception:
            # a device-side barrier timeout traps the kernel; its who/where record survives in mapped host memory
            try:
                from hetu_galvatron_b200.core.runtime.backend import get_backend
                sys.stderr.write("rank %s: device error info %s\n" % (os.environ.get("RANK", "0"), get_backend().comm.error_info()))
            except Exception:
                pass
            raise
