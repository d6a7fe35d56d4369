#!/usr/bin/env python
"""Benchmark of the hot path: designs/sec, forward + backward, on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W                 # this repository (CUDA path)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W    # N ranks, weak scaling
    python bench.py --impl reference ...                          # the reference's CPU path

One "step" = one design step of BASELINE.json config 2 (synthetic 100k-cell netlist, 331 819 pins,
101 levels, 256x256x3 layout image, 1 350 endpoints, fp32): U-Net forward, level-wise propagation
over every level, mask fusion + head, MSE, backward to every parameter gradient (optimizer step
excluded, SURVEY.md 8d).  Prints ONE JSON line on rank 0.

* value  : designs/s with the batch resident in HBM (CUDA events, max over ranks);
* e2e    : the same through the public API from pinned HOST buffers.  The design's STRUCTURE (netlist edges,
           level schedule, the endpoint batch and its path masks) is resident, like the reference's prebuilt DGL
           graph and mask tensor; per step the H2D copy of that step's VALUES -- cell / net features, image,
           labels (51.2 MB) -- and a D2H read of the loss are inside the timed region;
* roofline: the level-wise propagation forward (the HBM-bound kernel family), algorithmic bytes of
           SURVEY.md 8d / its CUDA-event time, against MEASURED_PEAKS.json;
* cpu_baseline: the oracle (a port of the reference arithmetic) on the host cores.
Under torchrun the two bucketed NCCL gradient all-reduces (head + fusion early; GNN + U-Net after the last kernel) are captured inside each rank's CUDA graph and
overlap the backward; `allreduce` reports their stand-alone time, the exposed part and the overlap fraction,
`config5` the 64-design run of SURVEY.md 8d (seeds 0..63 sharded round-robin over the ranks).
"""
import argparse
import importlib
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

# NCCL's own log lines ("NCCL version ...") must not land on stdout next to the ONE JSON line: route them to stderr
# (read when NCCL first initialises its logging, so it is set before torch is imported)
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":      # the one level NCCL_DEBUG_FILE does not apply to
    os.environ["NCCL_DEBUG"] = "WARN"
sys.dont_write_bytecode = True     # the benchmark writes nothing into the (possibly read-only) tree, no __pycache__ either

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG_NAME = "multimodal-fusion-based-pre-routing-timing-prediction-_b200"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, PKG_NAME))

METRIC = "designs/sec fwd+bwd (synthetic 100k-cell netlist+256x256 maps)"
WORKLOAD = "config2: 100k-cell netlist (331819 pins, 101 levels) + 3x256x256 image + 1350 endpoints, fp32"
CPU_SAMPLE_SCALE = 1           # the CPU arm runs the full config-2 design (about 4 s per step on 16 cores)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference's PyTorch path) on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_step(scale, seed=0, threads=None):
    """One bounded CPU sample of config 2 -> estimated seconds per full design.

    The reference's cost is ~linear in pins for the GNN part and fixed for the image / fusion /
    head part, so the sample runs the FULL-size image, masks and 1 350 endpoints but a netlist with
    1/scale of the cells (same 50 cell-levels): t_design = scale * t_gnn + (t_total - t_gnn)."""
    import tm_synth
    from oracle import levelize, restate
    if threads:
        torch.set_num_threads(threads)
    cfg = dict(tm_synth.CONFIGS["c2"])
    cfg["n_cells"] //= scale
    d = tm_synth.make_design(seed=seed, **cfg)
    import tm_engine
    model, cnn = tm_engine.build_models(d.map_size, seed=seed, device="cpu")
    sd_m = {k: v.detach() for k, v in model.state_dict().items()}
    sd_c = {k: v.detach() for k, v in cnn.state_dict().items()}
    t = torch.from_numpy
    ni, ns = levelize.in_csr(d.n, d.net_src, d.net_dst)
    ci, cs = levelize.in_csr(d.n, d.cell_src, d.cell_dst)
    od = dict(n=d.n, levels=[t(x.astype(np.int64)) for x in d.level_lists()],
              net_csr=(t(ni).long(), t(ns).long()), cell_csr=(t(ci).long(), t(cs).long()),
              cell_feat=t(d.cell_feat), net_feat=t(d.net_feat), image=t(d.image), endpoints=t(d.endpoints),
              endpoint_level=t(d.level[d.endpoints].astype(np.int64)), mask_indptr=t(d.mask_indptr).long(),
              mask_cols=t(d.mask_cols).long(), arrival_time=t(d.arrival_time))

    def total():
        t0 = time.perf_counter()
        restate.design_step(sd_m, sd_c, od)
        return time.perf_counter() - t0

    def gnn_only():
        P = {k: v.clone().requires_grad_(True) for k, v in sd_m.items() if k.startswith("gnn.fc_") and "drive" not in k and "attn" not in k}
        t0 = time.perf_counter()
        H = restate.gnn_propagate(P, "gnn", od["n"], od["levels"], od["net_csr"], od["cell_csr"], od["cell_feat"], od["net_feat"])
        H[od["endpoints"]].square().sum().backward()
        return time.perf_counter() - t0

    return total, gnn_only, d.n


def reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port -- the
    reference itself needs DGL, which is not installable here) on all host threads."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    total, gnn_only, n_sample = cpu_step(CPU_SAMPLE_SCALE, threads=threads)
    for _ in range(args.warmup):
        total()
    est = [total() for _ in range(args.steps)]
    sec = float(np.mean(est))
    sample = (f"every step is the full config-2 design ({n_sample} pins, 101 levels, 3x256x256 image, 1350 "
              f"endpoints), forward+backward, oracle port of the reference on {threads} host threads")
    line = {"impl": "reference", "metric": METRIC, "value": 1.0 / sec, "unit": "designs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": sample},
            "cpu_baseline": {"value": 1.0 / sec, "unit": "designs/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": 1.0 / sec, "unit": "designs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "kind 'port': the unmodified reference needs DGL (absent, not installable offline) and cannot travel to "
                    "the GPU box; the port is the same arithmetic without DGL's per-level scheduling and the reference's "
                    "per-level full-column index_copy, and is ~8x FASTER than the reference measured through a fake-DGL "
                    "graph during the survey (35 s/design on 8 cores, SURVEY.md section 6): ratios against this arm are "
                    "conservative"}
    print(json.dumps(line), flush=True)


def _make_c2(seed):
    import tm_synth
    return tm_synth.make_design(seed=seed, **tm_synth.CONFIGS["c2"])


def dump_outputs(out_dir, loss, pred, model, cnn):
    """--dump-outputs: what one timed step hands its caller -- the loss, the predictions and every parameter gradient
    -- as ``<out_dir>/<name>.npy`` in float32 (``grad.model.<param>``, ``grad.cnn.<param>``; 12 MB for config 2).
    The design and the initial weights are seeded, so two builds given the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss, "pred": pred}
    for prefix, mod in (("model", model), ("cnn", cnn)):
        for k, p in mod.named_parameters():
            if p.grad is not None:
                arrays[f"grad.{prefix}.{k}"] = p.grad
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", help="tm_synth.CONFIGS key (c2 = the headline workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the config-3 / config-4 device timings")
    ap.add_argument("--no-graph", action="store_true", help="time the resident loop eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 3 s sustained repeat of the resident loop")
    ap.add_argument("--no-shuffled", action="store_true", help="skip the fresh-endpoint-batch-every-step end-to-end loop")
    ap.add_argument("--config5", type=int, default=64, help="designs of the config-5 run (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the last one's loss, predictions and parameter gradients to DIR/<name>.npy")
    ap.add_argument("--profile-step", action="store_true",
                    help="after the warm-up run ONE step between cudaProfilerStart/Stop and exit "
                         "(for `ncu --profile-from-start off`); prints no bench line")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return reference_arm(args, rank, world)

    # config 5's designs are generated first, by forked workers, while this process has no CUDA context / NCCL threads
    c5_seeds, c5_designs = None, None
    if args.config5 > 0 and args.config == "c2" and not args.no_graph and not args.profile_step:
        import multiprocessing as mp
        import tm_dp
        c5_seeds = tm_dp.shard_designs(list(range(args.config5)), rank, world)
        with mp.get_context("fork").Pool(min(len(c5_seeds), max(1, (os.cpu_count() or 8) // max(world, 1)))) as pool:
            c5_designs = pool.map(_make_c2, c5_seeds)

    import torch.distributed as dist
    importlib.import_module(PKG_NAME)
    import tm_engine
    import tm_lib
    import tm_ops
    import tm_synth
    import tm_unet

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        pg = dist.group.WORLD

    d = tm_synth.make_design(seed=rank, **tm_synth.CONFIGS[args.config])    # one design per rank: weak scaling
    model, cnn = tm_engine.build_models(d.map_size, seed=0, device=dev)      # replicas start identical
    host = tm_engine.HostDesign(d, pin=True)
    batch = tm_engine.DesignBatch.from_host(host, dev)
    step = tm_engine.DesignStep(model, cnn, process_group=pg, world_size=world)
    sched = batch.graph.schedule()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    W = max(args.warmup, 3)
    for _ in range(W):
        step.run(batch)
    sync_all()

    if args.profile_step:
        torch.cuda.profiler.start()
        step.run(batch)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return

    # one step's kernel launches (counted eagerly; a graph replays exactly these)
    launches0 = tm_lib.launch_count()
    step.run(batch)
    sync_all()
    launches_per_step = tm_lib.launch_count() - launches0
    use_graph = not args.no_graph
    run_step = step.capture(batch) if use_graph else (lambda: step.run(batch))
    for _ in range(2):
        run_step()
    sync_all()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # ---- resident-input throughput
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        loss, pred = run_step()
    e1.record()
    sync_all()
    launches = launches_per_step * args.steps
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    if args.dump_outputs and rank == 0:          # now: the loops below replay other graphs that rewrite param.grad
        dump_outputs(args.dump_outputs, loss, pred, model, cnn)

    # ---- end to end from pinned host memory through the public API: every step copies its inputs
    # host -> device and reads its loss back.  The upload of step i+1 is issued on a copy stream before
    # step i computes (a data loader's prefetch), all inside the timed region.
    graph = batch.graph
    copy_stream = torch.cuda.Stream()
    if use_graph:
        # DesignStep.prepare(): structure resident + captured step; per-step VALUES (features, image,
        # labels) are re-uploaded into the graph's static inputs.  Two prepared copies alternate so that
        # the upload of the next step overlaps the replay of the current one.
        preps = [step.prepare(host, dev, graph=graph) for _ in range(2)]
        e2e_h2d = preps[0].nbytes()
        e2e_note = ("DesignStep.prepare(): netlist / endpoint / mask structure resident, step replayed as a CUDA graph; "
                    "per step: features + image + labels uploaded (prefetched on a copy stream), loss copied to pinned memory and "
                    "read by the host one step later")

        loss_host = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]

        def e2e_loop(n):
            # software pipeline of a training loop: while step i computes, step i+1's inputs are uploaded on the copy
            # stream and step i-1's loss (copied to pinned memory right behind its step) is read on the host
            ev = [torch.cuda.Event(), torch.cuda.Event()]
            done = [torch.cuda.Event(), torch.cuda.Event()]
            preps[0].upload(host, copy_stream); ev[0].record(copy_stream)
            out = 0.0
            for i in range(n):
                if i + 1 < n:
                    # (the copy stream must not overwrite the inputs of the prepared copy still in flight two steps back)
                    if i >= 1:
                        copy_stream.wait_event(done[(i + 1) & 1])
                    preps[(i + 1) & 1].upload(host, copy_stream); ev[(i + 1) & 1].record(copy_stream)
                torch.cuda.current_stream().wait_event(ev[i & 1])
                loss_d = preps[i & 1].step()[0]
                loss_host[i & 1].copy_(loss_d, non_blocking=True)     # D2H of this step's loss
                done[i & 1].record()
                if i >= 1:
                    done[(i - 1) & 1].synchronize()
                    out = float(loss_host[(i - 1) & 1])               # host reads the previous step's loss
            done[(n - 1) & 1].synchronize()
            out = float(loss_host[(n - 1) & 1])
            return out
    else:
        e2e_h2d = host.nbytes(per_step_only=True)
        e2e_note = "graph structure + level schedule cached per design; the next step's upload is prefetched on a copy stream"

        def upload():
            with torch.cuda.stream(copy_stream):
                b = tm_engine.DesignBatch.from_host(host, dev, graph=graph)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return b, ev

        def e2e_loop(n):
            nxt = upload()
            out = 0.0
            for i in range(n):
                b2, ev = nxt
                if i + 1 < n:
                    nxt = upload()
                torch.cuda.current_stream().wait_event(ev)
                out = float(step.run(b2)[0].item())          # D2H read of the step's loss
            return out

    e2e_loop(2)
    sync_all()
    t0 = time.perf_counter()
    lv = e2e_loop(args.steps)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())

    # ---- end to end with a FRESH shuffled endpoint batch every step (the reference's DataLoader, train.py:468-486):
    # a design with 3 x 1350 timing paths in the reference's tuple format, read by tm_loader, ONE CUDA-graph capture;
    # per step the host draws the next 1350 path ids, uploads them + the step's values (features, image), the graph
    # re-selects the mask rows on the device (tm_mask_select) and the loss is read back -- all inside the timed region
    e2e_shuffled = None
    if not args.no_shuffled and use_graph and args.config == "c2":
        import tm_loader
        d3 = tm_synth.make_design(seed=1000 + rank, n_endpoints=3 * 1350, **tm_synth.CONFIGS["c2"])
        ld = tm_loader.load_design(tm_loader.design_tuple_from_synth(d3), dev)
        hb = {"cell_feat": torch.from_numpy(d3.cell_feat).pin_memory(), "net_feat": torch.from_numpy(d3.net_feat).pin_memory(),
              "image": torch.from_numpy(d3.image).pin_memory()}
        all_paths = torch.as_tensor(ld.paths, dtype=torch.int64)
        gen = torch.Generator().manual_seed(rank)
        # two captures of the design alternate (upload i+1 while i computes); the TimingGraph's feature tensors are
        # shared, so each capture gets its own static value tensors
        preps_sh = []
        for k in range(2):
            b = ld.batch([ld.paths[i % len(ld.paths)] for i in range(1350)], dynamic=True)
            b.cell_feat, b.net_feat, b.image = b.cell_feat.clone(), b.net_feat.clone(), b.image.clone()
            preps_sh.append((b, step.capture(b)))

        def stage(k, ids):                                         # on the copy stream: ids -> endpoint batch, values
            b = preps_sh[k][0]
            with torch.cuda.stream(copy_stream):
                b.set_endpoints(*ld.batch_tensors(ids))
                b.cell_feat.copy_(hb["cell_feat"], non_blocking=True)
                b.net_feat.copy_(hb["net_feat"], non_blocking=True)
                b.image.copy_(hb["image"], non_blocking=True)

        def shuffled_loop(n):
            state = {"perm": torch.randperm(all_paths.numel(), generator=gen), "k": 0}

            def next_ids():
                if state["k"] + 1350 > state["perm"].numel():
                    state["perm"], state["k"] = torch.randperm(all_paths.numel(), generator=gen), 0
                ids = all_paths[state["perm"][state["k"]:state["k"] + 1350]]
                state["k"] += 1350
                return ids
            ev = [torch.cuda.Event(), torch.cuda.Event()]
            done = [torch.cuda.Event(), torch.cuda.Event()]
            lh = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]
            stage(0, next_ids()); ev[0].record(copy_stream)
            out = 0.0
            for i in range(n):
                if i + 1 < n:
                    if i >= 1:
                        copy_stream.wait_event(done[(i + 1) & 1])          # that capture's previous step has finished
                    stage((i + 1) & 1, next_ids()); ev[(i + 1) & 1].record(copy_stream)
                torch.cuda.current_stream().wait_event(ev[i & 1])
                loss_d = preps_sh[i & 1][1]()[0]
                lh[i & 1].copy_(loss_d, non_blocking=True)
                done[i & 1].record()
                if i >= 1:
                    done[(i - 1) & 1].synchronize()
                    out = float(lh[(i - 1) & 1])
            done[(n - 1) & 1].synchronize()
            return float(lh[(n - 1) & 1])
        shuffled_loop(2)
        sync_all()
        t0 = time.perf_counter()
        lsh = shuffled_loop(args.steps)
        torch.cuda.synchronize()
        sh_s = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(sh_s, op=dist.ReduceOp.MAX)
        h2d_sh = int(sum(v.numel() * v.element_size() for v in hb.values())) + 1350 * (8 + 4 + 4 + 4 + 4)
        e2e_shuffled = {"value": world * args.steps / float(sh_s.item()), "unit": "designs/s", "h2d_bytes_per_step": h2d_sh,
                        "d2h_bytes_per_step": 4, "paths_per_design": int(all_paths.numel()), "batch": 1350, "loss": lsh,
                        "note": "new shuffled 1350-path batch every step (tm_loader.LoadedDesign): the host draws and orders the ids, "
                                "uploads them + the step's values on a copy stream while the previous step computes (two captures of the "
                                "design alternate), the graph re-selects the mask rows on the device, the loss is read one step late"}
        del preps_sh, ld, d3
        torch.cuda.empty_cache()

    # ---- the same resident loop for >= 3 s: does the number survive sustained clocks?
    sustained = None
    if not args.no_sustained:
        n_sus = max(args.steps, int(3.2e3 / (ms_total / args.steps)))
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        s0.record()
        for _ in range(n_sus):
            run_step()
        s1.record()
        sync_all()
        ms_sus = torch.tensor([s0.elapsed_time(s1)], device=dev)
        if world > 1:
            dist.all_reduce(ms_sus, op=dist.ReduceOp.MAX)
        sustained = {"steps": n_sus, "seconds": float(ms_sus.item()) * 1e-3, "ms_per_step": float(ms_sus.item()) / n_sus,
                     "value": world * n_sus / (float(ms_sus.item()) * 1e-3), "unit": "designs/s"}
    clocks = sampler.finish() if rank == 0 else None

    # ---- data parallel: what the gradient exchange costs and how much of it the backward hides
    allreduce = None
    if world > 1 and use_graph:
        bks = list(step._buckets.values())
        cs = step.comm_stream

        def ar_only():
            for b in bks:
                with torch.cuda.stream(cs):
                    dist.all_reduce(b.flat, op=dist.ReduceOp.SUM)
                    b.flat.mul_(1.0 / world)
            torch.cuda.current_stream().wait_stream(cs)
        for _ in range(3):
            ar_only()
        sync_all()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(args.steps):
            ar_only()
        a1.record()
        sync_all()
        # the rank's compute alone: the same step captured without the collectives
        w_, step.world = step.world, 1
        try:
            local_replay = step._capture_local(batch)
        finally:
            step.world = w_
        for _ in range(2):
            local_replay()
        sync_all()
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record()
        for _ in range(args.steps):
            local_replay()
        l1.record()
        sync_all()
        t3 = torch.tensor([a0.elapsed_time(a1) / args.steps, l0.elapsed_time(l1) / args.steps], device=dev)
        dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        ar_ms, local_ms = float(t3[0]), float(t3[1])
        exposed = max(ms_total / args.steps - local_ms, 0.0)
        allreduce = {"buckets": {k: int(b.flat.numel()) * 4 for k, b in step._buckets.items()},
                     "ms_standalone": ar_ms, "step_ms_without_exchange": local_ms, "exposed_ms": exposed,
                     "overlap_frac": max(0.0, min(1.0, 1.0 - exposed / ar_ms)) if ar_ms > 0 else None,
                     "where": "two bucketed ncclAllReduce (head + fusion as soon as they exist; GNN + U-Net as one exchange after the last kernel) on a side stream INSIDE the captured graph"}

    # ---- BASELINE config 5 (SURVEY.md 8d): 64 designs of config-2 shape, seeds 0..63, round-robin over the ranks
    config5 = None
    if c5_designs is not None and use_graph:
        seeds, ds = c5_seeds, c5_designs
        pool5 = torch.cuda.graph_pool_handle()
        t_prep = time.perf_counter()
        preps5 = [step.prepare(tm_engine.HostDesign(dd, pin=False), dev, pool=pool5) for dd in ds]
        t_prep = time.perf_counter() - t_prep
        for pr in preps5[:2]:
            pr.step()
        sync_all()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for pr in preps5:
            loss5, _ = pr.step()
        c1.record()
        sync_all()
        ms5 = torch.tensor([c0.elapsed_time(c1)], device=dev)
        if world > 1:
            dist.all_reduce(ms5, op=dist.ReduceOp.MAX)
        config5 = {"designs": args.config5, "seeds": f"0..{args.config5 - 1}", "per_rank": len(seeds), "ms_total": float(ms5.item()),
                   "value": args.config5 / (float(ms5.item()) * 1e-3), "unit": "designs/s", "prepare_s_per_rank": t_prep,
                   "note": "distinct designs, sharded round-robin (tm_dp.shard_designs); one DP step = every rank's next design + the "
                           "in-graph gradient all-reduce; strong-scaling efficiency = T1 / (n * Tn) over the ms_total of the N = 1 run"}
        del preps5, ds
        torch.cuda.empty_cache()

    # ---- per-family device times on rank 0 (CUDA events on the launching stream)
    def timed(fn, reps=5):
        fn()
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    extra = {}
    if rank == 0:
        gp = [p.detach() for p in step.gnn_params]
        cf, nf = graph.ndata["cell_feat"], graph.ndata["net_feat"]
        H, saved = tm_ops.gnn_forward(sched, cf, nf, gp, save=True)
        S = torch.empty(sched.n, 128, device=dev)
        w1t, w2t = tm_ops.transpose(gp[8]), tm_ops.transpose(gp[10])
        gnb = tm_lib.ws_bytes("tm_gnn_ws_bytes")
        gws = tm_lib.workspace(gnb, dev)

        def prop_only():
            H.zero_()
            tm_lib.call("tm_gnn_forward", sched.struct, 0, sched.num_levels, H, S, w1t, gp[9], w2t, gp[11],
                        saved["A"], saved["LSE"], saved["HID"], gws, gnb, tm_lib.stream())

        S.copy_(torch.rand_like(S))
        t_zero = timed(lambda: H.zero_())
        # both back ends of the propagation, each timed alone: bit 0 of tm_gnn_set_impl = forward as ONE persistent
        # cluster kernel (the library default), 0 = one launch per level (what DesignStep uses next to the image stream)
        variants = {}
        for nm, impl in (("persistent (1 launch, grid barrier per level)", 1), ("per-level launches (PDL-chained)", 0)):
            old_impl = tm_lib.lib().tm_gnn_set_impl(impl)
            variants[nm] = {"ms": timed(prop_only) - t_zero, "grid_barriers": int(tm_lib.lib().tm_gnn_last_barriers())}
            tm_lib.lib().tm_gnn_set_impl(old_impl)
        best = min(variants, key=lambda k: variants[k]["ms"])
        t_prop = variants[best]["ms"]
        G = torch.zeros(sched.n, 128, device=dev)
        GA = torch.empty_like(saved["A"]); GH = torch.empty_like(saved["HID"]); GZ = torch.empty_like(saved["A"])

        def bwd_only():
            tm_lib.call("tm_gnn_backward", sched.struct, H, G, gp[8], gp[10], saved["A"], saved["LSE"], saved["HID"],
                        GA, GH, GZ, gws, gnb, tm_lib.stream())

        t_bwd = timed(bwd_only)
        t_gnn_f = timed(lambda: tm_ops.gnn_forward(sched, cf, nf, gp, save=True))
        t_gnn_b = timed(lambda: tm_ops.gnn_backward(sched, saved, gp, G))
        ust = {}

        def unet_f():
            ust["o"], ust["s"] = tm_unet.unet_forward(cnn, batch.image, need_bwd=True, update_stats=False)

        t_unet_f = timed(unet_f)
        t_unet_b = timed(lambda: tm_unet.unet_backward(cnn, ust["s"], torch.ones_like(ust["o"])))
        peak, peak_src = peaks()
        bytes_f = sched.algorithmic_bytes_fwd()
        ach = bytes_f / (t_prop * 1e-3) / 1e9
        # DRAM bytes of the same 101 launches from an ncu capture (profiles/<round>_traffic.json), if one was committed
        traffic = None
        tj = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if not os.path.isfile(tj):
            tj = os.path.join(ROOT, "profiles", "r1_traffic.json")
        if os.path.isfile(tj) and args.config == "c2":
            traffic = json.load(open(tj)).get("gnn_propagate_fwd_dram_bytes")
        for v in variants.values():
            v["GBps"] = bytes_f / (v["ms"] * 1e-3) / 1e9
            v["frac"] = v["GBps"] / peak
        extra["roofline"] = {"kernel": "tm_gnn_forward (level-wise propagation over %d levels), %s" % (sched.num_levels, best),
                             "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                             "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes": bytes_f,
                             "ms": t_prop, "variants": variants}
        # tensor-pipe family: the TMA-fed tcgen05 3x3 convolution of the U-Net's bf16 mode on its tensor-bound layer
        # (down3.conv2 of BASELINE config 4: 128 -> 128 channels, batch 32 of 64x64 maps; SURVEY 8a layer table)
        pj = os.path.join(ROOT, "MEASURED_PEAKS.json")
        tpeak = float(json.load(open(pj))["bf16_tflops"]) if os.path.isfile(pj) else 1590.0
        cb, ch, cw, cc = 32, 64, 64, 128
        npx = cb * ch * cw
        xb16 = torch.randn(npx, cc, device=dev).bfloat16()
        w16 = torch.randn(cc, cc, 3, 3, device=dev) * 0.05
        pk = tm_lib.ws_bytes("tm_conv3x3_bf16_pack", cw, cc, cc)
        wq16 = torch.empty(9, pk * cc, pk * cc, dtype=torch.bfloat16, device=dev)
        tm_lib.call("tm_conv3x3_pack_bf16", cc, cc, w16, wq16, pk, cc, 0, tm_lib.stream())
        y16 = torch.empty(npx, cc, device=dev)
        t_conv = timed(lambda: tm_lib.call("tm_conv3x3_bf16", cb, ch, cw, cc, cc, pk, xb16, wq16, None, y16, cc, 0,
                                           None, tm_lib.err_flag(dev), tm_lib.stream()), reps=20)
        cflop = 2.0 * 9 * cc * cc * npx
        extra["roofline_tensor"] = {"kernel": "conv3x3_tma_kernel<64> (bf16 operands by TMA, fp32 accumulate in TMEM; 128->128 channels, "
                                              "32 x 64x64 maps = U-Net down3.conv2 of config 4)",
                                    "bound": "tensor", "achieved": cflop / (t_conv * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                                    "frac": cflop / (t_conv * 1e-3) / 1e12 / tpeak, "ms": t_conv, "algorithmic_flops": cflop,
                                    "hbm_GBps": npx * (2 * cc + 4 * cc) / (t_conv * 1e-3) / 1e9,
                                    "traffic": (json.load(open(tj)).get("conv3x3_tma_128x128_32x64x64_dram_bytes")
                                                if os.path.isfile(tj) else None),
                                    "peak_source": "measured burst (MEASURED_PEAKS.json)" if os.path.isfile(pj) else "fallback"}
        del xb16, w16, wq16, y16
        # the largest dense contraction of the design step itself (second layer of the hoisted net-pin MLP, 3xTF32)
        Mg, Ng, Kg = int(sched.net_class.numel()), 128, 256
        Ag = torch.randn(Mg, Kg, device=dev); Wg = torch.randn(Ng, Kg, device=dev); Cg = torch.empty(Mg, Ng, device=dev)
        t_gemm = timed(lambda: tm_ops.gemm_nn(Mg, Ng, Kg, Ag, Kg, Wg, Kg, Cg, Ng, b_is_nk=True))
        tf = 2.0 * Mg * Ng * Kg / (t_gemm * 1e-3) / 1e12
        extra["hoisted_gemm"] = {"kernel": f"tf_gemm_kernel 3xTF32 (M={Mg}, N={Ng}, K={Kg}; 3 tcgen05 MMAs per product)",
                                 "TFLOPs": tf, "ms": t_gemm, "hbm_GBps": (Mg * Kg + Mg * Ng) * 4 / (t_gemm * 1e-3) / 1e9,
                                 "note": "operands are fp32 in HBM: this GEMM is bounded by HBM (353 MB), not the tensor pipe"}
        del Ag, Wg, Cg
        extra["kernels_ms"] = {"gnn_propagate_fwd": t_prop, "gnn_propagate_bwd": t_bwd,
                               "gnn_fwd_total(with hoisted MLPs)": t_gnn_f, "gnn_bwd_total(with weight grads)": t_gnn_b,
                               "unet_fwd": t_unet_f, "unet_bwd": t_unet_b,
                               "gnn_bwd_GBps": sched.algorithmic_bytes_bwd() / (t_bwd * 1e-3) / 1e9}
        if world == 1 and use_graph:
            # the same step with the image branch in its bf16 mode (TMA-fed tcgen05 convolutions, north_star (b)):
            # reported NEXT to the fp32-class headline, never instead of it (predictions then carry the bf16 bar, rtol 2e-2)
            try:
                cnn.math = "bf16"
                run_mixed = step.capture(batch)
                for _ in range(3):
                    run_mixed()
                torch.cuda.synchronize()
                m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                m0.record()
                for _ in range(args.steps):
                    loss_m, _ = run_mixed()
                m1.record()
                torch.cuda.synchronize()
                ms_m = m0.elapsed_time(m1) / args.steps
                extra["mixed_precision_step"] = {"value": 1e3 / ms_m, "unit": "designs/s", "ms_per_step": ms_m,
                                                 "loss": float(loss_m.item()), "dtype": "f32 (netlist branch, 3xTF32) + bf16 operands / fp32 accumulate (U-Net)",
                                                 "note": "not the headline: same design step with cnn.math = 'bf16'"}
            except Exception as e:                                   # noqa: BLE001
                extra["mixed_precision_step"] = {"error": repr(e)}
            finally:
                cnn.math = None
            # the same fp32-class step with the netlist branch restricted to the sub-netlist that can reach this batch's
            # endpoints (DesignStep(prune=True), tm_graph.ConeGraph): identical loss / predictions / gradients, pins no
            # endpoint depends on are not evaluated.  Reported NEXT to the headline, which evaluates every pin.
            try:
                step_p = tm_engine.DesignStep(model, cnn, prune=True)
                batch_p = tm_engine.DesignBatch.from_host(host, dev, graph=batch.graph)
                run_p = step_p.capture(batch_p)
                for _ in range(3):
                    run_p()
                torch.cuda.synchronize()
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                for _ in range(args.steps):
                    loss_p, _ = run_p()
                p1.record()
                torch.cuda.synchronize()
                ms_p = p0.elapsed_time(p1) / args.steps
                cone = batch_p.cone()
                extra["pruned_step"] = {"value": 1e3 / ms_p, "unit": "designs/s", "ms_per_step": ms_p, "loss": float(loss_p.item()),
                                        "pins_evaluated": cone.n_active, "pins": int(sched.n), "fraction": cone.fraction,
                                        "note": "not the headline: DesignStep(prune=True) evaluates only the pins from which one of "
                                                "the batch's 1 350 endpoints is reachable (same loss, predictions and gradients: "
                                                "tests/test_gpu_parity.py::test_design_step_on_cone_subnetlist)"}
                step_p.close()
            except Exception as e:                                   # noqa: BLE001
                extra["pruned_step"] = {"error": repr(e)}
        if world == 1 and not args.no_configs and args.config == "c2":
            # BASELINE configs 3 (GNN only, ~1M pins) and 4 (U-Net alone, 32 x 512x512, bf16): device timings next to
            # the headline (profiles/bench_configs.py; parity for both lives in tests/test_gpu_configs.py)
            spec = importlib.util.spec_from_file_location("bench_configs", os.path.join(ROOT, "profiles", "bench_configs.py"))
            bc = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(bc)
            del H, saved, S, G, GA, GH, GZ
            torch.cuda.empty_cache()
            try:
                extra["other_configs"] = {"config3": bc.config3(), "config4": bc.config4()[0], "layoutnet": bc.layoutnet()}
            except Exception as e:                                   # noqa: BLE001  (report, do not lose the headline line)
                extra["other_configs"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world == 1:
            threads = os.cpu_count() or 1
            total, gnn_only, n_sample = cpu_step(CPU_SAMPLE_SCALE, threads=threads)
            total()
            secs = [total() for _ in range(3)]
            sec = float(np.mean(secs))
            extra["cpu_baseline"] = {"value": 1.0 / sec, "unit": "designs/s", "cores": threads, "kind": "port",
                                     "sample": f"3 steps (after 1 warm-up) of the full config-2 design ({n_sample} pins), "
                                               f"forward+backward, oracle port of the reference; {sec:.2f} s/step"}
        else:
            extra["cpu_baseline"] = None

    if rank == 0:
        h2d = e2e_h2d
        line = {"metric": METRIC, "value": world * args.steps / (ms_total * 1e-3), "unit": "designs/s",
                "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms_total / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD if args.config == "c2" else args.config, "pins": d.n,
                           "levels": d.num_levels, "endpoints": int(d.endpoints.size),
                           "designs_per_step": world, "parallelism": f"dp{world}",
                           "resident_loop": ("CUDA graph replay of the two-stream step" + (
                               "" if world <= 1 else " with the bucketed NCCL all-reduces captured inside"
                               if os.environ.get("TM_DP_GRAPH", "1") != "0" else " + NCCL gradient all-reduce after each replay (TM_DP_GRAPH=0)"))
                           if use_graph else "eager launches",
                           "l2": "working set per step (~1.5 GB of activations) exceeds the 126 MB L2; no flush needed",
                           "arithmetic": "fp32 storage and accumulation everywhere; tensor-core products at >= 21 significant bits "
                                         "(3xTF32 tcgen05 GEMMs / convolutions; fp16 two-term split with power-of-two scales in "
                                         "the propagation's tile MLP and the fused self-term MLP kernels): rtol 1e-3 against the "
                                         "fp32 oracle on predictions, loss and every gradient"},
                "e2e": {"value": world * args.steps / e2e_s, "unit": "designs/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": 4, "note": e2e_note},
                "gpu_launches": launches, "clocks": clocks, "loss": lv, "sustained": sustained, "allreduce": allreduce,
                "config5": config5, "e2e_shuffled": e2e_shuffled}
        line.update(extra)
        tm_lib.check_err_flags()                 # no tensor-core barrier timed out anywhere in this run
        print(json.dumps(line), flush=True)
    if world > 1:
        # captured graphs hold NCCL kernels of this communicator: release them before tearing it down
        del run_step
        step.close()
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
