"""TEST INFRASTRUCTURE ONLY -- times the reference's CPU implementation of the step on the host cores: the UNMODIFIED
reference's `KEModel.forward -> loss.backward() -> KEModel.update` when its package is installed under oracle/_ref
(impl="reference"; `__graft_entry__.build()` installs it there with oracle/ref_install.py), else the CPU oracle
(oracle/kge_oracle.py, a port of the same PyTorch step; impl="port").  Both run under the reference's own process model:
`num_proc` forked Hogwild workers sharing the tables through shared memory, one intra-op thread
each, a barrier before and after (train.py:290-317, train_pytorch.py:255-259).  Sampling is
excluded (DGL's C++ sampler is not available offline): every worker consumes its own seeded
synthetic index stream, generated before the clock starts.

Used only by bench.py (`cpu_baseline` leg and `--impl reference`)."""
import os
import sys
import time

import numpy as np
import torch as th
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import kge_oracle as ko  # noqa: E402
from ref_install import REF_DIR, installed as reference_installed  # noqa: E402,F401


def make_batches(n_ent, n_rel, B, Ns, n_batches, seed):
    """Seeded synthetic batches: uniform head/tail/neg entity ids and relation ids; tail corruption
    on even steps, head on odd (sampler.py:853-859).  Returns CPU int64 tensors."""
    out = []
    C = B // Ns
    for k in range(n_batches):
        rng = np.random.default_rng(seed + k)
        h, t = rng.integers(0, n_ent, B), rng.integers(0, n_ent, B)
        r, ng = rng.integers(0, n_rel, B), rng.integers(0, n_ent, C * Ns)
        nodes, inv = np.unique(np.concatenate([h, t]), return_inverse=True)
        T = lambda a: th.from_numpy(np.ascontiguousarray(a.astype(np.int64)))
        out.append(dict(node_ids=T(nodes), head_local=T(inv[:B]), tail_local=T(inv[B:]), rel_ids=T(r),
                        neg_ids=T(ng), neg_head=bool(k % 2)))
    return out


def build_reference_model(hp, n_ent, n_rel):
    """The unmodified reference KEModel on CPU tensors (dgl replaced by the ~60-line stub of oracle/ref_harness.py)."""
    os.environ["KGE_REFERENCE_PY"] = REF_DIR
    import ref_harness as rh
    rh.REFERENCE_PY = REF_DIR
    args = rh.make_args(lr=hp.lr, regularization_coef=hp.reg_coef, regularization_norm=hp.reg_norm,
                        neg_adversarial_sampling=hp.adversarial, adversarial_temperature=hp.adv_temperature)
    model = rh.build_reference_model(hp.model, n_ent, n_rel, hp.hidden_dim, hp.gamma, args, hp.double_ent, hp.double_rel)
    return rh, model


def _worker(rank, hp, tables, n_ent, n_rel, B, Ns, steps, warmup, seed, barrier, out_q):
    th.set_num_threads(1)
    batches = make_batches(n_ent, n_rel, B, Ns, warmup + steps, seed + 100003 * rank)
    C = B // Ns
    if isinstance(tables, tuple) and tables[0] == "reference":
        rh, model = tables[1], tables[2]

        def run(b):     # train_pytorch.py:141-152
            pos_g = rh.FakePosGraph(b["node_ids"], b["head_local"], b["tail_local"], b["rel_ids"])
            neg_g = rh.FakeNegGraph(b["neg_ids"], C, Ns, Ns, b["neg_head"])
            loss, log = model.forward(pos_g, neg_g, -1)
            loss.backward()
            model.update(-1)
    else:
        ent, es, rel, rs = tables

        def run(b):
            ko.train_step(hp, ent, es, rel, rs, b["node_ids"], b["head_local"], b["tail_local"], b["rel_ids"],
                          b["neg_ids"], C, Ns, Ns, b["neg_head"])
    for b in batches[:warmup]:
        run(b)
    barrier.wait()
    t0 = time.perf_counter()
    for b in batches[warmup:]:
        run(b)
    barrier.wait()
    dt = time.perf_counter() - t0
    out_q.put((rank, dt))


def hogwild_edges_per_sec(hp, n_ent, n_rel, B, Ns, steps, warmup, num_proc, seed=0, impl="port"):
    """edges/s = num_proc * steps * B / wall (max over workers, which the closing barrier equalises)."""
    if impl == "reference":
        rh, model = build_reference_model(hp, n_ent, n_rel)
        model.share_memory()                    # train.py:291: tables in shared memory, Hogwild workers
        tables = ("reference", rh, model)
    else:
        ent, es, rel, rs = ko.init_tables(hp, n_ent, n_rel, seed=0)
        for t in (ent, es, rel, rs):
            t.share_memory_()
        tables = (ent, es, rel, rs)
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(num_proc)
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, hp, tables, n_ent, n_rel, B, Ns, steps, warmup, seed,
                                               barrier, q)) for r in range(num_proc)]
    for p in procs:
        p.start()
    times = [q.get() for _ in procs]
    for p in procs:
        p.join()
    wall = max(t for _, t in times)
    return num_proc * steps * B / wall, wall
