"""On-disk dataset readers (SURVEY 8f-3) against the reference's own classes (dataloader/KGDataset.py), CPU only.

Every case writes its files with the write_*_case functions below and reads them with dglke_b200.dataset; the id arrays,
dictionaries, counts and emitted map files must equal what the unmodified reference's reader returned for the same
files (tests/golden/host/reference_datasets.json, recorded by oracle/gen_golden_host.py), and the id arrays must equal
the ones the files were constructed from."""
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "host", "reference_datasets.json")


def reference_result(key):
    with open(GOLDEN) as f:
        return json.load(f)[key]


def summary(ds, path=None):
    """What a caller reads off a dataset object, JSON-shaped; with `path`, also the map files a raw_udd_* reader wrote."""
    ids = lambda m: None if m is None else [[k, int(v)] for k, v in m.items()]
    split = lambda s: None if s is None else [np.asarray(a).tolist() for a in s]
    out = dict(n_entities=int(ds.n_entities), n_relations=int(ds.n_relations), emap_fname=ds.emap_fname,
               rmap_fname=ds.rmap_fname, entity2id=ids(ds.entity2id), relation2id=ids(ds.relation2id),
               **{s: split(getattr(ds, s)) for s in ("train", "valid", "test")})
    if path is not None:
        out["maps"] = [open(os.path.join(path, f)).read() for f in ("entities.tsv", "relations.tsv")]
    return out


def _graph(n_ent=37, n_rel=5, n=120, seed=0):
    rng = np.random.default_rng(seed)
    return rng.integers(0, n_ent, n), rng.integers(0, n_rel, n), rng.integers(0, n_ent, n)


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(np.asarray(x), np.asarray(y))


ORDERS = ["hrt", "htr", "rht", "rth", "thr", "trh"]
DELIMS = ["\t", "|", ","]
RAW_ORDERS = ["hrt", "trh", "rht"]
UDD_FILES = ["ent.map", "rel.map", "tr.txt", "va.txt", "te.txt"]
RAW_FILES = ["tr.tsv", "va.tsv", "te.tsv"]


def _line(order, h, r, t, delim):
    # parse_srd_format gives the COLUMN of head / relation / tail (KGDataset.py:53-65): write the inverse
    from dglke_b200.dataset import parse_srd_format
    cols = [None, None, None]
    ch, cr, ct = parse_srd_format(order)
    cols[ch], cols[cr], cols[ct] = h, r, t
    return delim.join(str(c) for c in cols)


def _ename(i):
    return "/m/entity %d" % i          # names with a space and a slash


def _rname(i):
    return "rel.%d" % i


def write_udd_case(d, order, delim):
    """udd_<order> files (UDD_FILES) with integer ids in directory d; returns the (h, r, t) arrays they hold."""
    h, r, t = _graph()
    open(os.path.join(d, "ent.map"), "w").write("".join("e%d%s%d\n" % (i, delim, i) for i in range(37)))
    open(os.path.join(d, "rel.map"), "w").write("".join("r%d%s%d\n" % (i, delim, i) for i in range(5)))
    for name, sl in (("tr.txt", slice(0, 80)), ("va.txt", slice(80, 100)), ("te.txt", slice(100, 120))):
        open(os.path.join(d, name), "w").write("".join(_line(order, a, b, c, delim) + "\n" for a, b, c in zip(h[sl], r[sl], t[sl])))
    return h, r, t


def write_raw_udd_case(d, order):
    """raw_udd_<order> files (RAW_FILES) with entity and relation names in a new directory d; returns (h, r, t)."""
    h, r, t = _graph(seed=3)
    os.makedirs(d)
    for name, sl in (("tr.tsv", slice(0, 80)), ("va.tsv", slice(80, 100)), ("te.tsv", slice(100, 120))):
        open(os.path.join(d, name), "w").write(
            "".join(_line(order, _ename(a), _rname(b), _ename(c), "\t") + "\n" for a, b, c in zip(h[sl], r[sl], t[sl])))
    return h, r, t


def write_built_in_case(d):
    """FB15k and Freebase layouts under d; returns (h, r, t)."""
    h, r, t = _graph(seed=5)
    # FB15k layout: dictionaries 'id \\t name', triples by name
    fb = os.path.join(d, "FB15k")
    os.makedirs(fb)
    open(os.path.join(fb, "entities.dict"), "w").write("".join("%d\t/m/%03d\n" % (i, i) for i in range(37)))
    open(os.path.join(fb, "relations.dict"), "w").write("".join("%d\t/r/%d\n" % (i, i) for i in range(5)))
    for name, sl in (("train.txt", slice(0, 80)), ("valid.txt", slice(80, 100)), ("test.txt", slice(100, 120))):
        open(os.path.join(fb, name), "w").write("".join("/m/%03d\t/r/%d\t/m/%03d\n" % (a, b, c) for a, b, c in zip(h[sl], r[sl], t[sl])))
    # Freebase layout: the dictionaries start with their COUNT, triples are ids ordered head, tail, relation
    fr = os.path.join(d, "Freebase")
    os.makedirs(fr)
    open(os.path.join(fr, "entity2id.txt"), "w").write("37\n" + "".join("/m/%d\t%d\n" % (i, i) for i in range(37)))
    open(os.path.join(fr, "relation2id.txt"), "w").write("5\n" + "".join("r%d\t%d\n" % (i, i) for i in range(5)))
    for name, sl in (("train.txt", slice(0, 80)), ("valid.txt", slice(80, 100)), ("test.txt", slice(100, 120))):
        open(os.path.join(fr, name), "w").write("".join("%d\t%d\t%d\n" % (a, c, b) for a, b, c in zip(h[sl], r[sl], t[sl])))
    return h, r, t


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("delim", DELIMS)
def test_udd_integer_files(tmp_path, order, delim):
    from dglke_b200.dataset import get_dataset
    d = str(tmp_path)
    h, r, t = write_udd_case(d, order, delim)
    ds = get_dataset(d, "mine", "udd_" + order, delim, UDD_FILES)
    assert (ds.n_entities, ds.n_relations, ds.entity2id, ds.emap_fname, ds.rmap_fname) == (37, 5, None, "ent.map", "rel.map")
    _same(ds.train, (h[:80], r[:80], t[:80]))
    _same(ds.valid, (h[80:100], r[80:100], t[80:100]))
    _same(ds.test, (h[100:], r[100:], t[100:]))
    ds3 = get_dataset(d, "mine", "udd_" + order, delim, UDD_FILES[:3])
    assert ds3.valid is None and ds3.test is None
    assert summary(ds) == reference_result("udd_" + order + delim)
    # id out of range is an error, as in the reference (KGDataset.py:709-719)
    open(os.path.join(d, "bad.txt"), "w").write(_line(order, 37, 0, 0, delim) + "\n")
    with pytest.raises(AssertionError):
        get_dataset(d, "mine", "udd_" + order, delim, ["ent.map", "rel.map", "bad.txt"])
    open(os.path.join(d, "bad2.txt"), "w").write(_line(order, "x", 0, 0, delim) + "\n")
    with pytest.raises(ValueError):
        get_dataset(d, "mine", "udd_" + order, delim, ["ent.map", "rel.map", "bad2.txt"])


@pytest.mark.parametrize("order", RAW_ORDERS)
def test_raw_udd_string_files_build_the_same_dictionaries(tmp_path, order):
    from dglke_b200.dataset import get_dataset
    d = str(tmp_path / "mine")
    h, r, t = write_raw_udd_case(d, order)
    ds = get_dataset(d, "mykg", "raw_udd_" + order, "\t", RAW_FILES)
    # ids are assigned in order of first appearance: source, destination, (relation) line by line
    first = []
    for a, c in zip(h, t):
        for x in (a, c):
            if _ename(x) not in first:
                first.append(_ename(x))
    assert list(ds.entity2id.keys()) == first and list(ds.entity2id.values()) == list(range(len(first)))
    assert ds.n_entities == len(first) and ds.n_relations == len(set(r.tolist()))
    inv = {v: k for k, v in ds.entity2id.items()}
    assert [inv[i] for i in ds.train[0][:5]] == [_ename(x) for x in h[:5]]
    assert (ds.emap_fname, ds.rmap_fname) == ("entities.tsv", "relations.tsv")
    # the reference builds the same dictionaries in the same insertion order (-> the same map files) and the same ids
    assert summary(ds, d) == reference_result("raw_udd_" + order)
    # one file = train only
    d1 = str(tmp_path / "one")
    os.makedirs(d1)
    open(os.path.join(d1, "tr.tsv"), "w").write("".join(_line(order, _ename(a), _rname(b), _ename(c), "\t") + "\n" for a, b, c in zip(h, r, t)))
    one = get_dataset(d1, "mykg", "raw_udd_" + order, "\t", ["tr.tsv"])
    assert one.valid is None and one.test is None and len(one.train[0]) == 120
    with pytest.raises(AssertionError):
        get_dataset(d1, "FB15k", "raw_udd_" + order, "\t", ["tr.tsv"])           # a dataset name is required


def test_edge_importance_column(tmp_path):
    """4th column = importance (> 0).  The reference's reader calls np.float, which numpy >= 1.24 no longer has, so
    there is nothing to diff against; the values are checked against what was written."""
    from dglke_b200.dataset import get_dataset
    h, r, t = _graph(n=30)
    w = np.random.default_rng(1).uniform(0.1, 2.0, 30)
    d = str(tmp_path)
    open(os.path.join(d, "e"), "w").write("x\n" * 37)
    open(os.path.join(d, "r"), "w").write("x\n" * 5)
    open(os.path.join(d, "tr"), "w").write("".join("%d\t%d\t%d\t%r\n" % (a, b, c, float(x)) for a, b, c, x in zip(h, r, t, w)))
    ds = get_dataset(d, "w", "udd_hrt", "\t", ["e", "r", "tr"], has_edge_importance=True)
    assert len(ds.train) == 4
    np.testing.assert_array_equal(ds.train[3], w)
    open(os.path.join(d, "tr0"), "w").write("0\t0\t0\t0.0\n")
    with pytest.raises(AssertionError):
        get_dataset(d, "w", "udd_hrt", "\t", ["e", "r", "tr0"], has_edge_importance=True)


def test_built_in_layouts_without_network(tmp_path):
    from dglke_b200.dataset import get_dataset
    d = str(tmp_path)
    with pytest.raises(FileNotFoundError) as e:
        get_dataset(d, "FB15k", "built_in")
    assert "FB15k" in str(e.value) and "data.dgl.ai" in str(e.value)
    with pytest.raises(NotImplementedError):
        get_dataset(d, "wikikg2", "built_in")
    with pytest.raises(AssertionError):
        get_dataset(d, "nosuch", "built_in")
    h, r, t = write_built_in_case(d)
    ds = get_dataset(d, "FB15k", "built_in")
    assert (ds.n_entities, ds.n_relations, ds.emap_fname, ds.rmap_fname) == (37, 5, "entities.dict", "relations.dict")
    _same(ds.train, (h[:80], r[:80], t[:80]))
    _same(ds.test, (h[100:], r[100:], t[100:]))
    df = get_dataset(d, "Freebase", "built_in")
    assert (df.n_entities, df.n_relations, df.entity2id, df.emap_fname) == (37, 5, None, "entity2id.txt")
    _same(df.train, (h[:80], r[:80], t[:80]))
    for name, mine in (("FB15k", ds), ("Freebase", df)):
        assert summary(mine) == reference_result("built_in_" + name)
