"""CPU tests of the host-side mirror: flag surface vs the reference's own parser, batch/chunk
bookkeeping, graph objects and samplers (no CUDA calls)."""
import json
import os

import numpy as np
import pytest
import torch as th

from dglke_b200 import utils, graph

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host", "reference_flags.json")


def flag_table(p):
    """[option strings, default, type name, nargs, choices, action class] of every option of parser p, JSON-shaped."""
    rows = [[list(a.option_strings), a.default, getattr(a.type, "__name__", None), a.nargs,
             list(a.choices) if a.choices else None, type(a).__name__]
            for a in p._actions if a.option_strings and a.dest != "help"]
    return json.loads(json.dumps(sorted(rows, key=lambda row: row[0])))


def test_flag_surface_matches_reference_parser():
    """Every option string, default and type of dglke_train's parser (utils.py:199-297, train.py:40-60), against the
    reference's own parser as oracle/gen_golden_host.py recorded it."""
    with open(GOLDEN) as f:
        ref = json.load(f)
    assert flag_table(utils.CommonArgParser()) == ref["common"]
    # train-only flags (train.py:44-60): read from the source since importing dglke.train needs more of DGL
    src_flags = ref["train_only"]
    for flag in ("--gpu", "--mix_cpu_gpu", "--valid", "--rel_part", "--async_update", "--has_edge_importance"):
        assert flag in src_flags
    for flag in src_flags:
        assert any(flag in a.option_strings for a in utils.ArgParser()._actions)


def test_defaults_worth_knowing():
    a = utils.ArgParser().parse_args([])
    assert (a.hidden_dim, a.batch_size, a.neg_sample_size, a.lr, a.gamma) == (400, 1024, 256, 0.01, 12.0)
    assert (a.regularization_coef, a.regularization_norm, a.loss_genre, a.gpu) == (2e-6, 3, "Logsigmoid", [-1])


def test_batch_size_rounding():
    assert utils.get_compatible_batch_size(1000, 256) == 1024     # utils.py:27-33
    assert utils.get_compatible_batch_size(1024, 256) == 1024
    assert utils.get_compatible_batch_size(100, 256) == 100       # smaller than neg: untouched


def test_chunk_layout_matches_reference_rules():
    assert graph.chunk_layout(1000, 200) == (5, 200)
    assert graph.chunk_layout(100, 256) == (1, 100)               # sampler.py:497-500
    assert graph.chunk_layout(1001, 200) is None                  # ragged: skipped (sampler.py:503-504)


def test_pos_graph_and_sampler():
    pg = graph.build_pos_graph([5, 3, 5], [0, 1, 0], [3, 9, 9])
    assert pg.ndata["id"].tolist() == [3, 5, 9]
    h, t = pg.all_edges(order="eid")
    assert pg.ndata["id"][h].tolist() == [5, 3, 5] and pg.ndata["id"][t].tolist() == [3, 9, 9]
    assert pg.number_of_edges() == 3
    s = graph.SyntheticSampler(100, 7, 12, 4, seed=1)
    p1, n1 = next(s)
    p2, n2 = next(s)
    assert (n1.neg_head, n2.neg_head) == (False, True)           # tail first, then head (sampler.py:853-859)
    assert (n1.num_chunks, n1.chunk_size, n1.neg_sample_size) == (3, 4, 4)
    assert n1.ndata["id"][n1.tail_nid].shape[0] == 12
    p1b, _ = graph.SyntheticSampler(100, 7, 12, 4, seed=1).batch(0)
    assert th.equal(p1.ndata["id"], p1b.ndata["id"])             # seeded => reproducible


def test_triple_sampler_epochs_and_partition():
    rng = np.random.default_rng(0)
    h, r, t = rng.integers(0, 50, 100), rng.integers(0, 3, 100), rng.integers(0, 50, 100)
    s = graph.TripleSampler(h, r, t, 50, 3, 20, 5, seed=2)
    seen = []
    for k in range(5):                                            # one epoch = 5 batches of 20
        pg, ng = s.batch(k)
        hh, tt = pg.all_edges()
        seen += list(zip(pg.ndata["id"][hh].tolist(), pg.edata["id"].tolist(), pg.ndata["id"][tt].tolist()))
    assert sorted(seen) == sorted(zip(h.tolist(), r.tolist(), t.tolist()))
    parts = [graph.TripleSampler(h, r, t, 50, 3, 10, 5, seed=2, rank=k, world=2).n_edges for k in range(2)]
    assert sum(parts) == 100


def test_eval_batches_one_chunk_all_entities():
    b = list(graph.eval_batches(np.array([1, 2, 3]), np.array([0, 0, 1]), np.array([4, 5, 6]), 10, 2, True))
    assert len(b) == 2
    pg, ng = b[0]
    assert (ng.num_chunks, ng.chunk_size, ng.neg_sample_size, ng.neg_head) == (1, 2, 10, True)


def test_lazy_log_and_fused_loss_read_device_scalars_lazily():
    """log dict semantics of the reference (pos_loss, neg_loss, loss, regularization floats; loss excludes reg,
    general_models.py:569-576) on top of the device log4 buffer."""
    from dglke_b200.loss import LazyLog, FusedLoss
    log4 = th.tensor([0.25, 0.75, 0.5, 0.125])
    log = LazyLog(log4, has_reg=True)
    log4.zero_()                                   # the log owns a snapshot
    assert sorted(log.keys()) == ["loss", "neg_loss", "pos_loss", "regularization"]
    assert log["loss"] == 0.5 and log["regularization"] == 0.125 and "pos_loss" in log
    assert sum(l[k] for l in [log, log] for k in ["loss"]) == 1.0      # train loop's averaging idiom
    assert sorted(k for k in LazyLog(th.zeros(4), has_reg=False)) == ["loss", "neg_loss", "pos_loss"]
    loss = FusedLoss(th.tensor([0.25, 0.75, 0.5, 0.125]), with_reg=True)
    assert loss.backward() is None and abs(float(loss) - 0.625) < 1e-7 and loss.item() == float(loss)


def test_loss_generator_argument_errors_match_the_reference():
    """loss.py:58-62, base_loss.py:83-84: the same ValueErrors for the same argument combinations."""
    from dglke_b200.loss import LossGenerator, LazyLog
    for genre in ("Hinge", "Logistic", "Logsigmoid", "BCE"):
        g = LossGenerator(None, genre)
        assert g.neg_label == (0 if genre == "BCE" else -1) and g.pairwise is False
    assert LossGenerator(None, "Hinge", pairwise=True).pairwise and LossGenerator(None, "Logistic", pairwise=True).pairwise
    with pytest.raises(ValueError):
        LossGenerator(None, "Logsigmoid", pairwise=True)
    with pytest.raises(ValueError):
        LossGenerator(None, "BCE", pairwise=True)
    with pytest.raises(ValueError):
        LossGenerator(None, "Hinge", neg_adversarial_sampling=True, pairwise=True)
    with pytest.raises(ValueError):
        LossGenerator(None, "Huber")
    # the pairwise form logs 'loss' (+ 'regularization') only (loss.py:78-80)
    assert sorted(LazyLog(th.zeros(4), has_reg=True, only_loss=True).keys()) == ["loss", "regularization"]
    assert sorted(LazyLog(th.zeros(4), has_reg=False, only_loss=True).keys()) == ["loss"]


def test_unsupported_options_raise_instead_of_falling_back():
    from dglke_b200 import _lib
    with pytest.raises(_lib.KgeError):
        _lib.make_cfg("TransR", 8, 8, 12.0, 0.1, 0.1, 0.0, 3, False, 1.0, False, 8, 8, 8)
    with pytest.raises(ValueError):
        _lib.make_cfg("DistMult", 8, 8, 12.0, 0.1, 0.1, 0.0, 3, False, 1.0, False, 8, 8, 8, loss_genre="Huber")


def test_triple_filter_marks_exactly_the_true_corruptions():
    """Filtered evaluation (sampler.py:514-597 filter_false_neg -> neg_g.edata['bias'] = -1): brute force."""
    from dglke_b200.graph import TripleFilter, eval_batches
    rng = np.random.default_rng(0)
    n_ent, n_rel, n = 50, 4, 600
    h, r, t = rng.integers(0, n_ent, n), rng.integers(0, n_rel, n), rng.integers(0, n_ent, n)
    f = TripleFilter(h, r, t, n_rel)
    known = set(zip(h.tolist(), r.tolist(), t.tolist()))
    for neg_head in (False, True):
        got = f.bias(h[:40], r[:40], t[:40], n_ent, neg_head)
        want = np.zeros((40, n_ent), np.float32)
        for i in range(40):
            for e in range(n_ent):
                if ((e, r[i], t[i]) if neg_head else (h[i], r[i], e)) in known:
                    want[i, e] = -1
        assert np.array_equal(got, want)
        assert all(got[i, (h if neg_head else t)[i]] == -1 for i in range(40))      # the positive's own copy is filtered
        cand = np.sort(rng.choice(n_ent, 20, replace=False))
        assert np.array_equal(f.bias(h[:40], r[:40], t[:40], 20, neg_head, cand), want[:, cand])
    # a triple nobody has seen filters nothing
    assert f.bias([0], [0], [0], n_ent, False).sum() == -sum(1 for e in range(n_ent) if (0, 0, e) in known)
    for pg, ng in eval_batches(h[:10], r[:10], t[:10], n_ent, 4, True, known=f):
        b = ng.edata["bias"]
        assert tuple(b.shape) == (pg.number_of_edges(), n_ent) and b.dtype == th.float32
        assert ng.num_chunks == 1 and ng.neg_sample_size == n_ent
