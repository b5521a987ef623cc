#!/usr/bin/env python
"""bench.py -- edges/sec of the KGE training hot path (BASELINE.json metric) on N B200s.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one pass of the hot path (gather -> score over 1 positive + chunk-shared negatives ->
logsigmoid/self-adversarial loss gradient -> row-sparse Adagrad) over one batch of B synthetic edges.
Workload (default): BASELINE.json configs[1] -- TransE_l2, FB15k shape (14 951 entities, 1 345 relations),
d=400, neg=200, -adv, gamma 19.9, lr 0.25, rc 1e-9 (examples/fb15k/multi_gpu.sh:84-86).

One JSON line on stdout (rank 0).  Sampling is excluded on both arms (DGL's C++ sampler is not
available offline): batches are pre-generated from seeded numpy draws.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "dgl-ke_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

WORKLOADS = {
    # name: (model, n_ent, n_rel, hidden, gamma, lr, rc, neg, double_ent, default batch, description)
    # default batch 14800 = 74 chunks of 200: the contraction GEMMs then launch 148 / 296 CTAs = whole waves of the 148 SMs
    "fb15k_transe_l2": ("TransE_l2", 14951, 1345, 400, 19.9, 0.25, 1e-9, 200, False, 14800,
                        "TransE_l2 FB15k-shape d=400 neg=200 -adv (BASELINE configs[1])"),
    "wikikg2_rotate": ("RotatE", 2500604, 535, 200, 12.0, 0.01, 1e-9, 256, True, 4096,
                       "RotatE wikikg2-shape d=200 -de neg=256 -adv (BASELINE configs[2])"),
    "freebase_complex": ("ComplEx", 86054151, 14824, 400, 143.0, 0.1, 2e-6, 200, False, 14800,
                         "ComplEx Freebase-shape 86M entities d=400 neg=200 -adv (BASELINE configs[3])"),
    "synth_distmult": ("DistMult", 100000000, 10000, 512, 143.0, 0.08, 2e-6, 1024, False, 4096,
                       "DistMult synthetic 100M entities d=512 neg=1024 -adv (BASELINE configs[4])"),
    "freebase_transe_l2": ("TransE_l2", 86054151, 14824, 400, 19.9, 0.25, 1e-9, 200, False, 14800,
                           "TransE_l2 d=400 neg=200 -adv on the Freebase-shaped table (86 M entities, 137.7 GB; 14 824 relations): "
                           "north_star's multi-GPU scaling shape, HBM-resident"),
    "big_transe_l2": ("TransE_l2", 20000000, 1345, 400, 19.9, 0.25, 1e-9, 200, False, 14800,
                      "TransE_l2 d=400 neg=200 -adv on a 20M-entity (32 GB) table: HBM-resident variant of configs[1]"),
}
METRIC = "edges/sec TransE_l2 d=400 neg=200 at 1/2/4/8 B200 vs ref CPU; HBM GB/s %peak"


def bytes_per_edge(de, dr):
    # SURVEY.md 8(d): read (head, tail, neg, rel rows + 4 state scalars) + write of the same
    return 2 * (4 * (3 * de + dr) + 16)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: fb15k_transe_l2 (BASELINE configs[1]) on one GPU, freebase_transe_l2 (the 86 M-entity "
                         "HBM-resident table north_star's scaling target names) on several; the other one is measured beside it")
    ap.add_argument("--edge-placement", default="head-owner", choices=["head-owner", "random"],
                    help="N>1: which edges a rank trains on -- those whose head row it owns (half of the positive-node rows "
                         "are then local), or any (every row remote with probability (N-1)/N)")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="N>1: do not announce the next batch (no row prefetch by the fused kernels; every step gathers its own rows)")
    ap.add_argument("--no-beside", action="store_true", help="skip the second (beside) workload of a default run")
    ap.add_argument("--batch", type=int, default=0, help="edges per step per GPU (0 = workload default)")
    ap.add_argument("--n-ent", type=int, default=0, help="override the entity count (capacity experiments)")
    ap.add_argument("--engine", type=int, default=-1, help="-1 library default, 0 fp32 tiles, 1 tcgen05")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA graphs (profiling)")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--cpu-procs", type=int, default=16, help="reference arm: Hogwild worker processes (default 16, capped by the host's cores: the fastest count on the 128-vCPU GPU hosts, pinned so that the GPU/CPU ratio does not move with a probe; 0 = probe 8/16/32/64/all and use the fastest)")
    ap.add_argument("--cpu-impl", default="auto", choices=["auto", "reference", "port"], help="reference arm: the unmodified reference installed under oracle/_ref, or the oracle port")
    ap.add_argument("--cpu-batch", type=int, default=1000, help="reference arm: batch per worker (dglke_train's 1000)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU: after the timed steps, write what the last of them computed to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port of its PyTorch
    step, Hogwild num_proc workers) on the host cores.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_bench
    import kge_oracle as ko
    # same default workload as the GPU arm: FB15k shape at N=1, the Freebase-shaped table at N>1
    default_wl = "fb15k_transe_l2" if max(args.gpus, int(os.environ.get("WORLD_SIZE", "1"))) <= 1 else "freebase_transe_l2"
    model, n_ent, n_rel, hidden, gamma, lr, rc, neg, de, _, desc = WORKLOADS[args.workload or default_wl]
    if args.n_ent:
        n_ent = args.n_ent
    # host RAM / set-up time bound for the huge shapes: a stated scaled-down entity count (the CPU step's cost is in the
    # arithmetic of the 200 x 200 score blocks, not in the table size)
    cap = 2_000_000
    scaled = n_ent > cap
    n_ent_cpu = min(n_ent, cap)
    hp = ko.Hyper(model=model, hidden_dim=hidden, gamma=gamma, lr=lr, reg_coef=rc, reg_norm=3, adversarial=True,
                  adv_temperature=1.0, double_ent=de)
    ncpu = os.cpu_count() or 1
    B = args.cpu_batch // neg * neg or neg
    steps, warm = max(1, args.steps), max(1, args.warmup)
    t0 = time.time()
    impl = args.cpu_impl
    if impl == "auto":
        impl = "reference" if cpu_bench.reference_installed() else "port"
    # Hogwild workers contend on the shared tables (FB15k has only 15k entity rows), so more workers is not
    # monotonically faster -- on the 128-vCPU GPU-box hosts 16 workers reach ~3x the throughput of 128.  The count is
    # pinned (--cpu-procs, default 16); --cpu-procs 0 probes a few counts briefly and times the best one.
    cands = [min(args.cpu_procs, ncpu)] if args.cpu_procs else sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu} or {ncpu})
    probe = {}
    if len(cands) > 1:
        for c in cands:
            probe[c] = cpu_bench.hogwild_edges_per_sec(hp, n_ent_cpu, n_rel, B, neg, 3, 1, c, impl=impl)[0]
        nproc = max(probe, key=probe.get)
    else:
        nproc = cands[0]
    eps, wall = cpu_bench.hogwild_edges_per_sec(hp, n_ent_cpu, n_rel, B, neg, steps, warm, nproc, impl=impl)
    line = {
        "impl": "reference", "metric": METRIC, "value": eps, "unit": "edges/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": wall / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "batch_per_worker": B, "workers": nproc,
                   "entities": n_ent_cpu, "entities_scaled_down": scaled,
                   "note": ("the UNMODIFIED reference (oracle/_ref: KEModel.forward -> loss.backward() -> update, dgl stubbed) "
                            if impl == "reference" else "oracle port of the reference's PyTorch step (oracle/kge_oracle.py) ") +
                           "under dglke_train's process model: Hogwild workers on shared-memory tables, 1 thread each; sampling excluded"},
        "cpu_baseline": {"value": eps, "unit": "edges/s", "cores": nproc, "kind": impl,
                         "sample": "%d workers x %d steps x %d edges (%.1f s wall incl. setup and probe); probe edges/s by workers: %s"
                                   % (nproc, steps, B, time.time() - t0, {k: round(v) for k, v in probe.items()})},
        "e2e": {"value": eps, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx = [], set(), None
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def cpu_baseline_subprocess(args):
    """Times the CPU oracle on a bounded sample in a fresh process (before CUDA is initialised here)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload or "fb15k_transe_l2",
           "--steps", "8", "--warmup", "2", "--cpu-procs", str(args.cpu_procs), "--cpu-impl", args.cpu_impl]
    if args.n_ent:
        cmd += ["--n-ent", str(args.n_ent)]
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        for l in reversed(out.stdout.strip().splitlines()):
            if l.startswith("{"):
                return json.loads(l)["cpu_baseline"]
        return {"value": None, "unit": "edges/s", "cores": 0, "kind": "port", "sample": "failed: " + out.stderr[-200:]}
    except Exception as e:  # noqa
        return {"value": None, "unit": "edges/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of a one-GPU run")
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline_subprocess(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from dglke_b200.engine import StepEngine, DeviceTable, Hyper
    from dglke_b200.graph import SyntheticSampler

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (libkge_b200 has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # (the relation all-reduce runs beside the cooperative update kernel, which leaves it 16 SMs; capping NCCL with
        # NCCL_MAX_CTAS=16 was measured SLOWER at 2 GPUs -- the cap is left to the environment)
        dist.init_process_group("nccl", device_id=dev)
    default_run = args.workload is None
    primary = args.workload or ("fb15k_transe_l2" if world == 1 else "freebase_transe_l2")
    beside = None
    if default_run and not args.no_beside and not args.batch and not args.n_ent:
        beside = "freebase_transe_l2" if world == 1 else "fb15k_transe_l2"

    line = measure(args, primary, rank, world, local_rank, dev, cpu_base, max(1, args.steps), True)
    if beside is not None:
        torch.cuda.empty_cache()
        other = measure(args, beside, rank, world, local_rank, dev, None, min(max(1, args.steps), 20), False)
        if rank == 0:
            line["beside"] = {k: other[k] for k in ("value", "unit", "ms_per_step", "config", "e2e", "roofline")}
            line["beside"]["note"] = ("the same step on %s, measured in the same process: value(N) of the Freebase-shaped "
                                      "runs against the Freebase-shaped value at N=1 is the like-for-like scaling ratio"
                                      % WORKLOADS[beside][10])
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    if rank == 0:
        print(json.dumps(line), flush=True)
    sys.stdout.flush()
    if world > 1:
        # leave without tearing down NCCL / captured graphs / IPC mappings: destroying a process group whose
        # collectives live inside CUDA graphs has been seen to hang at exit
        os._exit(0)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, log4, tables):
    """What a caller of the timed step holds after its last call, as out_dir/<name>.npy (float32; row ids float64):

      log                        the step's (pos_loss, neg_loss, loss, regularization)
      <table>_emb, <table>_state the updated embedding table and its Adagrad state, for table in (entity, relation)

    tables: {table: (emb, state, ids the step read)}.  A table larger than its share of DUMP_BYTES is written as a
    seeded sample of the rows that step updated (most rows of a large table are never touched), sorted, with their ids
    in <table>_rows.npy.  The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"log": log4}
    share = (DUMP_BYTES - 4096) // len(tables)
    for name, (emb, state, ids) in tables.items():
        row_bytes = 4 * emb.shape[1] + 4
        if emb.shape[0] * row_bytes <= share:
            arrays[name + "_emb"], arrays[name + "_state"] = emb, state
            continue
        rows = torch.unique(ids).cpu().numpy()
        cap = share // (row_bytes + 8)
        if len(rows) > cap:
            rows = np.sort(np.random.default_rng(0).choice(rows, cap, replace=False))
        idx = torch.from_numpy(rows).to(emb.device)
        arrays[name + "_rows"] = torch.from_numpy(rows.astype(np.float64))
        arrays[name + "_emb"], arrays[name + "_state"] = emb[idx], state[idx]
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


def measure(args, workload, rank, world, local_rank, dev, cpu_base, K_steps, full):
    """One workload: device-resident throughput (CUDA graph per step), end-to-end throughput, per-kernel times."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from dglke_b200.engine import StepEngine, DeviceTable, Hyper
    from dglke_b200.graph import SyntheticSampler

    model, n_ent, n_rel, hidden, gamma, lr, rc, neg, de, bdef, desc = WORKLOADS[workload]
    if args.n_ent:
        n_ent = args.n_ent
    B = (args.batch or bdef) // neg * neg
    hp = Hyper(model=model, hidden_dim=hidden, gamma=gamma, lr=lr, reg_coef=rc, reg_norm=3, adversarial=True,
               adv_temperature=1.0, double_ent=de)
    De, Dr = hp.entity_dim, hp.relation_dim

    # ---- tables (resident in HBM before the clock starts) ------------------------------------
    gen = torch.Generator(device=dev).manual_seed(0)
    if world == 1:
        ent = torch.empty((n_ent, De), dtype=torch.float32, device=dev).uniform_(-hp.emb_init, hp.emb_init, generator=gen)
        ent_state = torch.zeros(n_ent, dtype=torch.float32, device=dev)
        rel = torch.empty((n_rel, Dr), dtype=torch.float32, device=dev).uniform_(-hp.emb_init, hp.emb_init, generator=gen)
        rel_state = torch.zeros(n_rel, dtype=torch.float32, device=dev)
        eng = StepEngine(hp, DeviceTable.from_tensors(ent, ent_state), DeviceTable.from_tensors(rel, rel_state), local_rank)
        parallelism = "1 GPU"
    else:
        from dglke_b200.dist import ShardedTrainer
        eng = ShardedTrainer(hp, n_ent, n_rel, dev, seed=0)
        parallelism = "entity rows sharded over %d GPUs (P2P over NVLink), relations replicated + NCCL all-reduce" % world
    if args.engine >= 0:
        eng.h.set_engine(args.engine)

    # ---- batches: NB distinct pre-sampled batches per rank, device and pinned-host copies --------
    NB = 8
    head_range = None
    if world > 1 and args.edge_placement == "head-owner":
        from dglke_b200.dist import shard_rows
        _, lo, hi = shard_rows(n_ent, world, rank)
        head_range = (lo, hi)
    sampler = SyntheticSampler(n_ent, n_rel, B, neg, seed=0, rank=rank, head_range=head_range)
    host, devb = [], []
    for k in range(NB):
        pg, ng = sampler.batch(k)
        hb = [pg.ndata["id"], pg.all_edges()[0], pg.all_edges()[1], pg.edata["id"], ng.ndata["id"]]
        hb = [t.pin_memory() for t in hb]
        host.append((hb, ng.neg_head))
        db = [t.to(dev) for t in hb]
        db += [db[0][db[1]].contiguous(), db[0][db[2]].contiguous()]      # the edges' global endpoint ids (a sampler has them)
        devb.append((db, ng.neg_head))
    Cs = sampler.chunk_size
    h2d = sum(t.numel() * 8 for t in host[0][0])

    pipelined = world > 1 and not args.no_pipeline

    def step_dev(k):
        b, nh = devb[k % NB]
        if world == 1:
            return eng.step(b[0], b[1], b[2], b[3], b[4], Cs, neg, nh, head_ids=b[5], tail_ids=b[6])
        nxt = devb[(k + 1) % NB][0]
        return eng.step(b[0], b[1], b[2], b[3], b[4], Cs, neg, nh, next_batch=(nxt[0], nxt[4]) if pipelined else None)

    def step_host(k):
        b, nh = host[k % NB]
        if world == 1:
            return eng.step_host(b[0], b[1], b[2], b[3], b[4], Cs, neg, nh)
        return eng.step_host(b[0], b[1], b[2], b[3], b[4], Cs, neg, nh, next_host=host[(k + 1) % NB][0] if pipelined else None)

    def prime():
        """(pipelined) every measured sequence starts at batch 0: forget whatever an earlier sequence staged and run
        the step before it, whose fused kernels fetch batch 0's rows"""
        if pipelined:
            eng.eng.announce_next(None)
            step_dev(NB - 1)
            torch.cuda.synchronize()

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def flush():
        if not args.no_flush:
            flush_buf.fill_(1)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W, K = max(3, args.warmup), K_steps
    for k in range(W):
        step_dev(k)
    torch.cuda.synchronize()
    prime()

    # ---- CUDA graphs of the device-resident step (one per batch): no launch gaps inside a step ----
    graphs = None
    if not args.no_graph:
        try:
            graphs = []
            for k in range(NB):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    step_dev(k)
                graphs.append(g)
        except Exception as e:  # noqa
            sys.stderr.write("graph capture failed (%r); timing eager launches\n" % (e,))
            graphs = None
            torch.cuda.synchronize()
    if world > 1:   # every rank must take the same path (a captured NCCL collective needs all ranks)
        ok = torch.tensor([1 if graphs is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            graphs = None

    def timed(run_step, after=None):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        prime()
        barrier()
        for k in range(K):
            flush()
            ev[k][0].record()
            run_step(k)
            if after:
                after()
            ev[k][1].record()
        barrier()
        t = sum(a.elapsed_time(b) for a, b in ev)   # ms of device time inside the K steps
        tt = torch.tensor([t], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    clk = ClockSampler(local_rank) if rank == 0 else None
    if graphs is not None:
        ms_dev = timed(lambda k: graphs[k % NB].replay())
    else:
        ms_dev = timed(step_dev)
    clocks = clk.stop() if clk else None
    if full and args.dump_outputs:
        last = devb[(K - 1) % NB][0]
        dump_outputs(args.dump_outputs, eng.log4, {"entity": (ent, ent_state, torch.cat([last[0], last[4]])),
                                                   "relation": (rel, rel_state, last[3])})

    # launches per step, counted from one eager step
    prime()
    c0 = eng.h.launch_count()
    step_dev(0)
    torch.cuda.synchronize()
    per_step_launches = eng.h.launch_count() - c0
    gpu_launches = per_step_launches * K

    # ---- end to end: host index buffers -> pinned staging -> H2D -> step -> D2H log ---------------
    ms_e2e = timed(step_host, after=eng.sync)

    # ---- per-kernel device time of one step (CUDA events around every launch, L2 flushed) --------
    prime()
    eng.h.profile_enable(True)
    prof = {}
    nprof = 5
    for k in range(nprof):
        flush()
        # keep the GPU busy (~1 ms spin) while the host enqueues the step, so that the event pairs measure
        # back-to-back kernel durations and not the host's launch latency
        torch.cuda._sleep(2_000_000)
        step_dev(k)
        for name, ms in eng.h.profile_read():
            prof[name] = prof.get(name, 0.0) + ms / nprof
    eng.h.profile_enable(False)
    kern_ms = sum(prof.values())
    dominant = max(prof.items(), key=lambda kv: kv[1]) if prof else ("", 0.0)

    used_graph = graphs is not None
    graphs = None
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        eng.close()                     # every rank unmaps the shards: the next workload of this process allocates its own
    if rank != 0:
        return None

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    bpe = bytes_per_edge(De, Dr)
    edges = world * K * B
    value = edges / (ms_dev * 1e-3)
    e2e = edges / (ms_e2e * 1e-3)
    # roofline of the step's kernels: algorithmic bytes of one launch set (= one step) / summed kernel time
    achieved = B * bpe / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else 0.0
    # DRAM traffic of one step from the committed ncu --set full capture -- only when that capture was taken on exactly
    # this workload / batch / schedule on one GPU (profiles/summarize.py writes the key); null otherwise
    traffic, traffic_key = None, "%s|B=%d|launches=%d" % (workload, B, per_step_launches)
    if world == 1:
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))).get(traffic_key)
        except Exception:
            pass
    line = {
        "metric": METRIC, "value": value, "unit": "edges/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "batch_per_gpu": B, "global_batch": B * world, "chunk_size": Cs,
                   "neg_sample_size": neg, "entities": n_ent, "relations": n_rel, "parallelism": parallelism,
                   "l2": "cold: 256 MiB written between timed steps" if not args.no_flush else "warm (no flush)",
                   "launch": "one CUDA graph per step" if used_graph else "eager launches",
                   "sampling": "excluded (pre-generated seeded batches), as on the reference arm",
                   "edge_placement": ("each rank trains on the edges whose head row it owns (tails and negatives anywhere)"
                                      if head_range else "random" if world > 1 else "n/a"),
                   "pipeline": ("next batch announced: its rows are fetched over NVLink by this step's fused kernels (entity reads "
                                "lag the updates by one step, as under the reference's --async_update)") if pipelined else "none",
                   "arithmetic": "fp32 rows; contractions on tcgen05 as 3xTF32 (hi/lo split) with fp32 accumulation" if model in ("TransE_l2", "DistMult", "ComplEx", "RESCAL") else "fp32 CUDA-core tiles",
                   "bytes_per_edge": bpe},
        "e2e": {"value": e2e, "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16,
                "ms_per_step": ms_e2e / K},
        "gpu_launches": gpu_launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": traffic, "traffic_key": traffic_key, "peak_source": peak_src,
                     "kernel": "all %d kernels of one step (CUDA events around each launch, L2 flushed)" % per_step_launches,
                     "algorithmic_bytes_per_launch_set": B * bpe,
                     "kernel_ms": {k: round(v, 5) for k, v in sorted(prof.items(), key=lambda kv: -kv[1])},
                     "dominant_kernel": {"name": dominant[0], "share": dominant[1] / kern_ms if kern_ms else 0.0}},
        "cpu_baseline": cpu_base,
        "clocks": clocks,
    }
    if world > 1:
        # NVLink traffic of one step of one GPU, counted from the batch (not measured by a counter): rows whose owner is a
        # peer.  Reads = the prefetch of the next batch's tail and negative rows by the fused kernels (or the gather when
        # not pipelined); writes = the bulk reductions of the update kernel into those same rows.
        try:
            f = (world - 1) / world
            n_nodes_remote = (B if head_range else 2 * B) * f        # heads are local under head-owner placement
            remote_rows = n_nodes_remote + (B // Cs) * neg * f
            byts = remote_rows * De * 4
            t_fused = sum(v for k, v in prof.items() if "k_fused" in k) * 1e-3
            t_upd = sum(v for k, v in prof.items() if "k_update" in k) * 1e-3
            line["nvlink"] = {"remote_rows_per_step": int(remote_rows), "read_bytes_per_step": int(byts),
                              "write_bytes_per_step": int(byts),
                              "read_GBs_over_the_fused_kernels": (byts / t_fused / 1e9) if (pipelined and t_fused > 0) else None,
                              "write_GBs_over_k_update": (byts / t_upd / 1e9) if t_upd > 0 else None,
                              "note": "analytic: (N-1)/N of the tail and negative rows (+ the heads under random placement) x row bytes"}
        except Exception as e:  # noqa
            line["nvlink"] = {"error": repr(e)}
    return line


if __name__ == "__main__":
    # stdout carries exactly ONE line, the JSON: native libraries that print there (NCCL's version banner ...) are sent
    # to stderr for the duration of the run
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_real_stdout, "w", buffering=1)
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
