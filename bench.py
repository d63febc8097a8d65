#!/usr/bin/env python
"""bench.py — molecules/s for 1000-step GCDM sampling with the B200-native GCPNet denoiser.

Contract (see DESIGN.md §Measurement):
  python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

One bench "step" = one complete sample of the batch: T reverse-diffusion steps + the final decode
(T+1 denoiser forwards), i.e. BASELINE.json's metric "molecules/sec (1000-step sample)".  Workload at N=1 is
BASELINE config[1]: QM9 unconditional, T=1000, batch 128 (19 atoms per molecule, the README demo size);
for N > 1 every GPU gets its own 128 molecules (weak scaling) and the final coordinates are all-gathered once.
`--config geom_hist` is BASELINE config[3]: GEOM-Drugs, 512 molecules IN TOTAL with sizes drawn from the dataset's
number-of-atoms histogram (seed 123), split over the ranks by bdiff.distributed.sample_sharded (LPT by n^2, strong
scaling, one NCCL gather).  Rank 0 prints ONE JSON line.
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
for p in (os.path.join(ROOT, "bio-diffusion_b200"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "molecules/sec (1000-step sample)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="qm9", choices=["qm9", "qm9_cond", "geom", "geom_hist", "geom_train"],
                    help="sampling workloads, or geom_train = BASELINE config 5 (training step, 64 molecules per GPU)")
    ap.add_argument("--train-tf32", action="store_true", help="geom_train: TF32 tensor-core GEMMs instead of fp32")
    ap.add_argument("--batch", type=int, default=None, help="molecules per GPU (default 128; geom 64; geom_hist: 512 in TOTAL)")
    ap.add_argument("--atoms", type=int, default=None, help="atoms per molecule (default 19 qm9 / 44 geom)")
    ap.add_argument("--timesteps", type=int, default=1000)
    ap.add_argument("--mode", default=os.environ.get("BDIFF_MODE", "tensor"), choices=["parity", "tensor"],
                    help="tensor: tcgen05 GEMMs with split-bf16 (hi+lo, >=16-bit) operands and fp32 accumulation, <=1e-4 "
                         "from the reference per forward (default); parity: all-fp32 FFMA")
    ap.add_argument("--no-parity-leg", action="store_true", help="skip the extra fp32 parity-mode chain (tensor mode)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-forwards", type=int, default=0,
                    help="denoiser forwards per CPU sample (bounded sample of the workload; default 8, geom_hist 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_MAX_BYTES = 64 * 1000 * 1000


def dump_outputs(dirname, arrays):
    """Write each tensor of `arrays` (name -> tensor) as `dirname`/<name>.npy in float32.  Past 64 MB in all, every array
    is flattened and cut to the same fraction of its elements (at least one), taken at seeded (hence fixed) positions, so
    that two builds run with the same arguments can still be compared element for element."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    host = {k: v.detach().to("cpu", torch.float32) for k, v in arrays.items()}
    total = sum(4 * v.numel() for v in host.values())
    budget = DUMP_MAX_BYTES - (128 + 4) * len(host)                  # per file: .npy header, the one element always kept
    for name, v in host.items():
        keep = max(1, v.numel() * budget // max(total, 1))
        if keep < v.numel():
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            v = v.reshape(-1)[idx]
        np.save(os.path.join(dirname, name + ".npy"), v.numpy())


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.th = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 9:
                self.rows.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------- workloads
def model_config(args):
    return "geom" if args.config in ("geom_hist", "geom_train") else args.config


def workload_sizes(args, world):
    """Molecule sizes of the whole job (all ranks) and a description.  qm9 / qm9_cond / geom: fixed-size molecules, `batch`
    per GPU (weak scaling).  geom_hist: `batch` (512) molecules in total, sizes ~ GEOM number-of-atoms histogram."""
    if args.config == "geom_hist":
        from bdiff.datasets import GEOM_N_NODES, sample_num_nodes
        total = args.batch or 512
        sizes = sample_num_nodes(GEOM_N_NODES, total, seed=123)
        return sizes, f"GEOM-Drugs unconditional sampling, T={args.timesteps}, batch {total} in total, sizes ~ dataset histogram (seed 123)"
    batch = args.batch or (64 if args.config == "geom" else 128)
    atoms = args.atoms or (44 if args.config == "geom" else 19)
    kind = "property-conditional" if args.config == "qm9_cond" else "unconditional"
    return (torch.full((batch * world,), atoms, dtype=torch.long),
            f"{args.config} {kind} sampling, T={args.timesteps}, batch {batch} x {atoms} atoms per GPU")


def cpu_reference_forwards(config, sizes, forwards, seed=123):
    """`forwards` denoiser forwards (= forwards-1 reverse steps + the decode) of the reference's CPU path (oracle port of
    the PyG/torch_scatter code) on the SAME batch the GPU arm samples.  Returns seconds.  The per-forward cost does not
    depend on the step index (the loop is strictly sequential, SURVEY.md §6), so a bounded number of steps of the T-step
    chain is a fair sample of it."""
    import gcpnet_oracle as O
    ocfg = O.config_named(config)
    sd = O.random_state_dict(ocfg, seed=7)
    ctx = torch.randn((len(sizes), ocfg.num_context), generator=torch.Generator().manual_seed(seed)) if ocfg.num_context else None
    noise = O.SeededNoise(seed)
    t0 = time.perf_counter()
    with torch.no_grad():
        O.sample_chain(sd, ocfg, sizes, noise, num_timesteps=max(1, forwards - 1), context=ctx)
    return time.perf_counter() - t0


def cpu_arm(args, reps):
    """Reference CPU path on this host: the SAME workload as the GPU arm at N=1 (same molecules), `--cpu-forwards` of its
    T+1 denoiser forwards per sample, all host threads (torch intra-op = os.cpu_count()).  value = molecules/s for the
    full T-step sample, scaled from the measured seconds per forward."""
    sizes, desc = workload_sizes(args, 1)
    cfgname = model_config(args)
    fw = max(2, args.cpu_forwards if args.cpu_forwards else (2 if args.config == "geom_hist" else 8))
    cpu_reference_forwards(cfgname, sizes[:2], 2)             # import / allocator warm-up
    # all the host threads the CPU path can USE: over-threading slows the small ops down, so one forward pair is tried
    # at a few intra-op thread counts and the fastest is kept (reported as `cores`; the same procedure in both CPU legs)
    ncpu = os.cpu_count() or 1
    best, best_t = 1, None
    for c in sorted({min(ncpu, x) for x in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(c)
        t = cpu_reference_forwards(cfgname, sizes, 2)
        if best_t is None or t < best_t:
            best, best_t = c, t
    cores = best
    torch.set_num_threads(cores)
    times = [cpu_reference_forwards(cfgname, sizes, fw) for _ in range(max(1, reps))]
    secs = sum(times) / len(times)
    per_fwd = secs / fw
    value = len(sizes) / (per_fwd * (args.timesteps + 1))
    block = {"value": value, "unit": "molecules/s", "cores": cores, "kind": "port", "same_config": True,
             "sample": f"oracle port of the reference PyG path on {cores} host threads: {desc.replace(' per GPU', '')}; "
                       f"{fw} of the {args.timesteps + 1} denoiser forwards per sample ({secs:.1f} s, {1000 * per_fwd:.0f} ms/forward), "
                       f"scaled to the full chain (per-forward cost is step-independent)",
             "seconds_per_sample": secs, "ms_per_forward": 1000 * per_fwd}
    return block, secs, desc


def run_reference(args):
    """--impl reference: the reference's CPU implementation (oracle port; /root/reference does not travel to the
    GPU box and needs PyG/torch_scatter which are not installable offline) on all host cores, same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    block, secs, desc = cpu_arm(args, reps=args.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": block["value"], "unit": "molecules/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * secs, "higher_is_better": True,
        "scaling": "strong" if args.config == "geom_hist" else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": desc, "sample": block["sample"]},
        "cpu_baseline": block,
        "e2e": {"value": block["value"], "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch.distributed as dist
    import bdiff
    from bdiff.distributed import sample_sharded, lpt_shards, shard_imbalance
    import gcpnet_oracle as O   # only for seeded synthetic weights (shapes/magnitudes), not on the timed path

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    T = args.timesteps
    cfgname = model_config(args)
    strong = args.config == "geom_hist"
    dcfg = bdiff.DenoiserConfig.named(cfgname)
    ocfg = O.config_named(cfgname)
    sd = O.random_state_dict(ocfg, seed=7)       # synthetic random-init weights of the named architecture
    net = bdiff.GCPNetDynamicsB200(config=dcfg, mode=args.mode)
    net.load_state_dict(sd, strict=True)
    net.to(dev)
    sampler = bdiff.GCDMSampler(net, use_cuda_graph=True)
    torch.manual_seed(123 + rank)

    sizes_all, desc = workload_sizes(args, world)            # the whole job's molecules (identical on every rank)
    total_mols = int(sizes_all.shape[0])
    if strong:
        shards = lpt_shards(sizes_all.tolist(), world)
        mine = shards[rank]
    else:
        per = total_mols // world
        mine = list(range(rank * per, (rank + 1) * per))
    sizes_mine = sizes_all[torch.tensor(mine, dtype=torch.long)] if mine else sizes_all[:0]
    num_nodes_host = sizes_all.clone().pin_memory() if strong else sizes_mine.clone().pin_memory()
    ctx_host = None
    if dcfg.num_context:
        ctx_host = torch.randn((len(mine), dcfg.num_context), generator=torch.Generator().manual_seed(5 + rank)).pin_memory()
    n_nodes = int(sizes_mine.sum())
    E = int((sizes_mine.long() ** 2).sum())
    width = 3 + dcfg.num_atom_types + int(dcfg.include_charges)
    out_host = torch.empty((int(sizes_all.sum()) if strong else n_nodes, width), pin_memory=True)
    flush_buf = torch.empty(256 * 1024 * 1024 // 4, device=dev)      # > 126 MB L2
    finite_flag = torch.ones((), dtype=torch.bool, device=dev)
    last = []                                                        # the job's samples from the latest chain

    def one_chain(nodes, ctx):
        """The product's public call for this workload; returns the step's result on the device."""
        nonlocal finite_flag
        if strong:
            out, _ = sample_sharded(sampler, nodes, ctx, T)          # LPT shards, chain, ONE NCCL all_gather
            last[:] = [out]
        else:
            out, _, _ = sampler.sample(nodes, ctx, T)
            last[:] = [out]
            if world > 1:
                bufs = [torch.empty_like(out) for _ in range(world)]
                dist.all_gather(bufs, out)                           # single NCCL gather of final coordinates
                last[:] = bufs
        finite_flag = finite_flag & torch.isfinite(out).all()
        return out

    nodes_dev = num_nodes_host.to(dev)
    ctx_dev = ctx_host.to(dev) if ctx_host is not None else None

    def chain_resident():
        one_chain(nodes_dev if not strong else num_nodes_host, ctx_dev)

    def chain_e2e():
        nn = num_nodes_host.to(dev, non_blocking=True)               # H2D of this step's inputs (pinned)
        cdev = ctx_host.to(dev, non_blocking=True) if ctx_host is not None else None
        out = one_chain(nn if not strong else num_nodes_host, cdev)
        out_host.copy_(out, non_blocking=True)                       # D2H of the step's result
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total = 0.0
        barrier()
        for _ in range(k):
            flush_buf.fill_(1.0)                                      # L2 flush between timed iterations (untimed)
            barrier()
            ev0.record()
            fn()
            ev1.record()
            torch.cuda.synchronize()
            total += ev0.elapsed_time(ev1)
        barrier()
        t = torch.tensor([total], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                  # max over ranks
        return t.item() / 1000.0

    def log(msg):
        if rank == 0:
            print(f"[bench +{time.perf_counter() - t_start:7.1f}s] {msg}", file=sys.stderr, flush=True)

    t_start = time.perf_counter()
    for i in range(args.warmup):
        chain_resident()
        torch.cuda.synchronize()
        log(f"warm-up chain {i + 1}/{args.warmup} done")
    sampler.nan_guard_count(reset=True)
    clocks = ClockSampler(local)
    launches0 = sampler_launches(sampler, net)
    if rank == 0:
        clocks.start()
    secs = timed(chain_resident, args.steps)
    final = list(last)                                               # outputs of the last timed chain
    clk = clocks.stop() if rank == 0 else None
    launches = sampler_launches(sampler, net) - launches0
    log(f"timed resident chains done: {secs:.2f} s for {args.steps}")
    secs_e2e = timed(chain_e2e, args.steps)
    log(f"timed e2e chains done: {secs_e2e:.2f} s")
    # correctness guards of the timed chains: finite outputs, and how often the reference's NaN guard (gcpnet.py:1214-1216)
    # zeroed a velocity field (0 expected)
    nan_hits = torch.tensor([sampler.nan_guard_count()], device=dev)
    fin = finite_flag.to(torch.int32).reshape(1)
    if world > 1:
        dist.all_reduce(nan_hits, op=dist.ReduceOp.SUM)
        dist.all_reduce(fin, op=dist.ReduceOp.MIN)
    if not bool(fin.item()):
        raise SystemExit("bench.py: a timed chain produced non-finite outputs")

    mols_total = total_mols * args.steps
    value = mols_total / secs
    e2e_value = mols_total / secs_e2e

    # ---- roofline of the dominant kernel (fused message + scatter), timed live with CUDA events in the library
    bi = torch.repeat_interleave(torch.arange(len(mine), device=dev), sizes_mine.to(dev))
    mask = torch.ones(n_nodes, dtype=torch.bool, device=dev)
    g = torch.Generator().manual_seed(3)
    xh = torch.randn((n_nodes, 3 + dcfg.num_h), generator=g).to(dev)
    tt = torch.full((n_nodes, 1), 0.5, device=dev)
    cnode = ctx_dev[bi] if ctx_dev is not None else None
    prof = None
    for i in range(6):
        flush_buf.fill_(0.0) if i else None
        pr, _ = net.profile_forward(bi, mask, xh, tt, cnode, len(mine))
        if i:   # first call is warm-up
            prof = pr if prof is None else {k: prof[k] + pr[k] for k in pr}
    prof = {k: v / 5 for k, v in prof.items()}
    L = dcfg.num_layers
    ed, xd = dcfg.e_hidden, dcfg.xi_hidden
    hid0 = (64 + xd) // 4
    w_msg = (256 * (512 + ed + hid0 + 9) + 256 + hid0 * (64 + xd) + 3 * (64 + xd) + 32 * hid0 + 32 * 256 + 32
             + 3 * (256 * 273 + 256 + 8 * 32 + 3 * 32 + 32 * 8 + 32 * 256 + 32) + 257)
    bytes_alg = E * (4 * (ed + 3 * xd) + 36) + n_nodes * (2 * 4 * 352) + 4 * w_msg     # SURVEY.md §8(d)
    flops_edge = 821176 if cfgname != "geom" else 793224                                  # per edge per layer
    fused = "layers_fused" in prof        # tensor mode: one persistent kernel runs all L edge + node passes
    flops_node = 575324                                                                   # per node per layer
    if fused:
        t_kernel = prof["layers_fused"] / 1000.0
        launch_flops = L * (E * flops_edge + n_nodes * flops_node)
        bytes_alg = L * bytes_alg
    else:
        t_kernel = prof["edge_message"] / L / 1000.0
        launch_flops = E * flops_edge
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get("tensor_fused" if fused else args.mode)
    except Exception:
        pass
    achieved_gbs = bytes_alg / t_kernel / 1e9
    achieved_tf = launch_flops / t_kernel / 1e12
    tensor_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))     # the kernel is timed inside a long step
    kname = ("k_layers_tc (persistent tcgen05 kernel: the fused per-edge message MLP + segmented scatter-sum and the node "
             "update of all %d layers, tiles scheduled by dependency flags; split-bf16 operands: 3 MMAs per algorithmic "
             "product)" % L if fused
             else "k_edge_message (fp32 fused per-edge GCP message MLP + segmented scatter-sum)")
    common = {
        "kernel": kname, "traffic": traffic, "algorithmic_bytes_per_launch": bytes_alg,
        "algorithmic_flops_per_launch": launch_flops, "kernel_ms": t_kernel * 1000,
        "hbm_achieved_gbs": achieved_gbs, "hbm_peak_gbs": hbm_peak, "hbm_frac": achieved_gbs / hbm_peak,
        "algorithmic_tflops": achieved_tf,
        "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)",
        "note": "the fused pass is compute-bound by construction (~1.3 kFLOP/B, SURVEY.md fact 3); the HBM figure "
                "(BASELINE.json's metric) is carried as hbm_* next to the binding roof.  `achieved` counts ALGORITHMIC "
                "FLOPs of the reference's un-factored fp32 math; the tensor pipe executes 3 bf16 MMAs per product to reach "
                "fp32-class accuracy, so 1/3 of the bf16 peak is the ceiling of this figure",
        "forward_ms_by_kernel": prof,
    }
    if args.mode == "tensor":
        roofline = dict(bound="tensor", achieved=achieved_tf, peak=tensor_peak, unit="TFLOP/s",
                        frac=achieved_tf / tensor_peak, **common)
    else:
        roofline = dict(bound="hbm", achieved=achieved_gbs, peak=hbm_peak, unit="GB/s", frac=achieved_gbs / hbm_peak,
                        **common)

    # ---- tensor mode: one extra chain in all-fp32 parity mode, reported next to the headline
    parity_leg = None
    if args.mode == "tensor" and not args.no_parity_leg and world == 1 and not strong:
        pnet = bdiff.GCPNetDynamicsB200(config=dcfg, mode="parity")
        pnet.load_state_dict(sd, strict=True)
        pnet.to(dev)
        psampler = bdiff.GCDMSampler(pnet, use_cuda_graph=True)
        psampler.sample(nodes_dev, ctx_dev, min(T, 50))               # warm-up / graph capture
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        psampler.sample(nodes_dev, ctx_dev, T)
        ev1.record()
        torch.cuda.synchronize()
        psecs = ev0.elapsed_time(ev1) / 1000.0
        parity_leg = {"value": total_mols / psecs, "unit": "molecules/s", "ms_per_step": 1000 * psecs, "dtype": "f32",
                      "note": "same workload with BDIFF_MODE_PARITY_FP32 (every MAC an fp32 FFMA; 1e-6 from the reference)"}
        log(f"parity-mode chain done: {psecs:.2f} s")

    # ---- "un-fused GPU" denominator (BASELINE.md §3.3): the reference's algorithm as un-fused PyTorch ops (the oracle port;
    #      the reference modules themselves need PyG/torch_scatter and do not travel to this box) on THIS GPU, same batch
    gpu_unfused = None
    if world == 1 and not strong and not args.no_cpu_baseline:
        try:
            sd_dev = {k: v.to(dev) for k, v in sd.items()}
            ei_dev = O.fully_connected_edge_index(bi.cpu(), mask.cpu()).to(dev)     # built once: generous to the baseline
            orig_ei = O.fully_connected_edge_index
            O.fully_connected_edge_index = lambda *_a, **_k: ei_dev
            try:
                with torch.device(dev), torch.no_grad():
                    ref_out = O.denoiser_forward(sd_dev, ocfg, bi, mask, xh, tt, cnode)       # warm-up (+ agreement check)
                    torch.cuda.synchronize()
                    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    nf = 5
                    ev0.record()
                    for _ in range(nf):
                        O.denoiser_forward(sd_dev, ocfg, bi, mask, xh, tt, cnode)
                    ev1.record()
                    torch.cuda.synchronize()
            finally:
                O.fully_connected_edge_index = orig_ei
            ms_fwd = ev0.elapsed_time(ev1) / nf
            ours = net.denoise(bi, mask, xh, tt, cnode, len(mine))
            gpu_unfused = {"value": total_mols / (ms_fwd / 1000.0 * (T + 1)), "unit": "molecules/s", "ms_per_forward": ms_fwd,
                           "kind": "port", "forwards_sampled": nf,
                           "max_abs_diff_vs_ours": float((ours - ref_out).abs().max().item()),
                           "note": "oracle port of the reference's PyG/torch_scatter algorithm run as un-fused PyTorch CUDA ops "
                                   "on the same B200 and batch (edge index precomputed); denoiser forwards only, scaled to "
                                   "the T+1 forwards of a sample"}
            log(f"un-fused GPU port: {ms_fwd:.1f} ms/forward")
        except Exception as ex:      # a baseline leg must never take the measurement down
            gpu_unfused = {"unavailable": f"{type(ex).__name__}: {ex}"}

    imb = shard_imbalance(sizes_all.tolist(), world) if strong else 1.0
    line = {
        "metric": METRIC, "value": value, "unit": "molecules/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000 * secs / args.steps, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32" if args.mode == "parity" else "bf16x2 (split hi+lo operands, f32 accumulate; <=1e-4 of the fp32 reference)",
        "data": "synthetic",
        "config": {"workload": desc,
                   "config_name": args.config, "molecules_total": total_mols, "molecules_this_rank": len(mine),
                   "timesteps": T, "denoiser_forwards_per_step": T + 1, "nodes_rank0": n_nodes, "edges_rank0": E,
                   "mode": args.mode,
                   "precision": ("tensor mode: every GEMM on tcgen05 tensor cores with split-bf16 operands (activations and "
                                 "weights each hi+lo, >=16 significant bits; A_hi.W_hi + A_lo.W_hi + A_hi.W_lo), fp32 "
                                 "accumulation in TMEM, fp32 state, ex2/rcp activations; per-forward error vs the "
                                 "reference's fp32 path <= 1e-4*max(1,|out|) (measured 4e-6..3.5e-5 relative on the six "
                                 "reference fixtures, tests/test_gpu_tc.py), bit-identical reruns")
                                if args.mode == "tensor" else "parity mode: all fp32 FFMA, 1e-6 from the reference",
                   "weights": "random init of the named architecture (seed 7)",
                   "l2": "flushed between timed chains (256 MiB write); inside a chain the working set is "
                         "L2-resident by design",
                   "parallelism": (f"dp{world}: 512 molecules split by LPT on n^2 (max/mean shard cost {imb:.3f}), no collective "
                                   f"in the chain, one final all_gather" if strong else
                                   f"dp{world}: molecule shards, no collective in the chain, one final all_gather")},
        "e2e": {"value": e2e_value, "unit": "molecules/s", "h2d_bytes_per_step": int(num_nodes_host.numel() * 8 +
                (ctx_host.numel() * 4 if ctx_host is not None else 0)),
                "d2h_bytes_per_step": int(out_host.numel() * 4), "ms_per_step": 1000 * secs_e2e / args.steps},
        "gpu_launches": int(launches) * world,
        "chains_finite": True, "nan_guard_hits": int(nan_hits.item()),
        "clocks": clk,
        "roofline": roofline,
    }
    if strong:
        line["shard_cost_imbalance"] = imb
    if parity_leg is not None:
        line["parity_fp32"] = parity_leg
    if gpu_unfused is not None:
        line["gpu_unfused_baseline"] = gpu_unfused
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_arm(args, reps=1)[0]
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"samples": torch.cat(final)})     # [molecules x atoms, 3 + atom types (+1)]
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_train(args):
    """BASELINE config 5: GEOM-Drugs denoiser training step — GCDMTrainLoss (training pass of the library: forward with tape),
    loss.backward() (bdiff_train_backward), DDP-style gradient mean over the ranks (one NCCL all-reduce), adaptive clip +
    AdamW(amsgrad) + EMA kernels.  `batch` (64) molecules per GPU with sizes from the GEOM histogram; a step takes a NEW batch
    (new topology plan), like a data loader would deliver it."""
    import torch.distributed as dist
    import bdiff
    from bdiff.datasets import GEOM_N_NODES, sample_num_nodes
    from bdiff.optim import GCDMTrainTail
    import gcpnet_oracle as O   # seeded synthetic weights + the CPU baseline leg only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dcfg = bdiff.DenoiserConfig.named("geom")
    ocfg = O.config_named("geom")
    sd = O.random_state_dict(ocfg, seed=7)
    net = bdiff.GCPNetDynamicsB200(config=dcfg, mode="parity")
    net.load_state_dict(sd, strict=True)
    net.to(dev)
    net.flatten_parameters()
    net.set_train_precision(args.train_tf32)
    opt = GCDMTrainTail(net.parameters())
    tl = bdiff.GCDMTrainLoss(net, GEOM_N_NODES)
    torch.manual_seed(123 + rank)                                # t and the noise of every step: same in every run
    B = args.batch or 64
    nb = 4                                                       # distinct host batches, cycled
    A = dcfg.num_atom_types
    batches, edges = [], []
    for b in range(nb):
        sizes = sample_num_nodes(GEOM_N_NODES, B, seed=1000 * (rank + 1) + b)
        g = torch.Generator().manual_seed(17 * (rank + 1) + b)
        bi = torch.repeat_interleave(torch.arange(B), sizes)
        n = int(bi.shape[0])
        x = torch.randn((n, 3), generator=g) * 2.0
        x = x - (torch.zeros((B, 3)).index_add_(0, bi, x) / sizes[:, None].float())[bi]
        one_hot = torch.nn.functional.one_hot(torch.randint(0, A, (n,), generator=g), A).float()
        batches.append(tuple(v.pin_memory() for v in (bi, torch.ones(n, dtype=torch.bool), x, one_hot, torch.zeros((n, 0)))))
        edges.append(int((sizes.long() ** 2).sum()))
    dev_batches = [tuple(v.to(dev) for v in hb) for hb in batches]
    loss_host = torch.zeros((), pin_memory=True)
    flush_buf = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    counter = [0]
    finite = [True]
    last = [None]                                                # loss of the latest resident step

    def train_step(batch):
        opt.zero_grad()
        loss = tl(*batch, None)[0].mean()
        loss.backward()
        opt.allreduce_grads()                                    # DDP: mean of the gradients, ONE all-reduce of the flat buffer
        opt.step()
        return loss.detach()

    def step_resident():
        loss = train_step(dev_batches[counter[0] % nb])
        counter[0] += 1
        last[0] = loss
        return loss

    def step_e2e():
        hb = batches[counter[0] % nb]
        counter[0] += 1
        loss = train_step(tuple(v.to(dev, non_blocking=True) for v in hb))      # H2D of this step's batch (pinned)
        loss_host.copy_(loss, non_blocking=True)                                # D2H of the step's result
        torch.cuda.current_stream().synchronize()
        finite[0] = finite[0] and bool(torch.isfinite(loss_host))
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total = 0.0
        barrier()
        for _ in range(k):
            flush_buf.fill_(1.0)
            barrier()
            ev0.record()
            fn()
            ev1.record()
            torch.cuda.synchronize()
            total += ev0.elapsed_time(ev1)
        barrier()
        t = torch.tensor([total], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / 1000.0

    for _ in range(max(args.warmup, 3)):
        step_resident()
    torch.cuda.synchronize()
    clocks = ClockSampler(local)
    l0, k0 = net.launch_count(), opt.kernel_launches
    if rank == 0:
        clocks.start()
    counter[0] = 0
    secs = timed(step_resident, args.steps)
    clk = clocks.stop() if rank == 0 else None
    launches = (net.launch_count() - l0) + (opt.kernel_launches - k0)
    final = None
    if args.dump_outputs:                                        # the last timed step's loss and the weights it left
        final = {"loss": last[0], "parameters": torch.cat([p.detach().reshape(-1) for p in net.parameters()])}
    counter[0] = 0
    secs_e2e = timed(step_e2e, args.steps)
    fin = torch.tensor([int(finite[0])], device=dev)
    if world > 1:
        dist.all_reduce(fin, op=dist.ReduceOp.MIN)
    if not bool(fin.item()):
        raise SystemExit("bench.py: a timed training step produced a non-finite loss")

    # phases of one step (events on the launch stream, batch 0, after the timed region)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    batch = dev_batches[0]
    opt.zero_grad()
    torch.cuda.synchronize()
    ev[0].record()
    loss = tl(*batch, None)[0].mean()
    ev[1].record()
    loss.backward()
    ev[2].record()
    opt.allreduce_grads()
    ev[3].record()
    opt.step()
    ev[4].record()
    torch.cuda.synchronize()
    phases = {k: ev[i].elapsed_time(ev[i + 1]) for i, k in enumerate(("loss_forward", "backward", "allreduce", "optimizer"))}
    # roofline: the step is GEMM-bound; algorithmic FLOPs = forward (793 kFLOP per edge and layer + 575 kFLOP per node and
    # layer, SURVEY.md §8d) x 3 (forward, input gradients, weight gradients)
    E0, n0 = edges[0], int(batch[0].shape[0])
    flops = 3.0 * dcfg.num_layers * (E0 * 793224 + n0 * 575324)
    t_fb = (phases["loss_forward"] + phases["backward"]) / 1000.0
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tensor_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    mols = B * world * args.steps
    line = {
        "metric": "molecules/sec (GEOM-Drugs training step: forward + backward + gradient all-reduce + optimizer)",
        "value": mols / secs, "unit": "molecules/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": 1000 * secs / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32 GEMMs, f32 elsewhere" if args.train_tf32 else "f32",
        "data": "synthetic",
        "config": {"workload": f"GEOM-Drugs denoiser training step, {B} molecules per GPU, sizes ~ dataset histogram, a new batch "
                               f"(new topology plan) every step",
                   "config_name": "geom_train", "edges_per_batch_rank0": edges, "weights": "random init (seed 7)",
                   "objective": "GCDMTrainLoss = reference training-mode L2 objective (t ~ U{0..T}, one denoiser call)",
                   "optimizer": "adaptive gradient-norm clip + AdamW(amsgrad) + EMA 0.9999 (bdiff_optimizer_step)",
                   "l2": "flushed between timed steps (256 MiB write)",
                   "parallelism": f"dp{world}: one batch per rank, gradients averaged with one NCCL all-reduce of the flat gradient buffer per step"},
        "e2e": {"value": mols / secs_e2e, "unit": "molecules/s", "ms_per_step": 1000 * secs_e2e / args.steps,
                "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in batches[0])), "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches) * world,
        "library_calls": "GEMMs of the training pass are cuBLAS SGEMM calls (not counted in gpu_launches)",
        "losses_finite": True, "clocks": clk, "phase_ms_batch0": phases,
        "roofline": {"bound": "tensor", "achieved": flops / t_fb / 1e12, "peak": tensor_peak, "unit": "TFLOP/s",
                     "frac": flops / t_fb / 1e12 / tensor_peak, "traffic": None,
                     "kernel": "forward + backward of the training pass (cuBLAS SGEMMs + element kernels), batch 0",
                     "algorithmic_flops": flops, "ms": 1000 * t_fb,
                     "note": "fp32 SGEMM does not run on the tensor pipe: against the bf16 tensor peak this fraction is small "
                             "by construction; it is reported so that the gap to a tcgen05 training pass is visible"},
    }
    if world == 1 and not args.no_cpu_baseline:
        # the same objective on the host: autograd through the oracle port, first `cpu_mols` molecules of batch 0
        cpu_mols = 32
        bi, mask, x, one_hot, charges = batches[0]
        nn0 = int((bi < cpu_mols).sum())
        sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        torch.manual_seed(1)
        t0 = time.perf_counter()
        lc, _ = O.eval_nll(sdg, ocfg, bi[:nn0], mask[:nn0], x[:nn0], one_hot[:nn0], charges[:nn0], None, GEOM_N_NODES,
                           lambda s_: torch.randn(s_), training=True)
        lc.mean().backward()
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": cpu_mols / dt, "unit": "molecules/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"one forward+backward (torch autograd through the oracle port) of the first {cpu_mols} "
                                          f"molecules of batch 0 ({nn0} atoms), {dt:.1f} s"}
    if rank == 0 and final is not None:
        dump_outputs(args.dump_outputs, final)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def sampler_launches(sampler, net):
    return getattr(sampler, "kernel_launches", 0)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "geom_train":
        run_train(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
