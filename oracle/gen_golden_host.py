"""Generates tests/golden/host/*.json from the UNMODIFIED reference (KGE_REFERENCE_PY = its python/ directory):

    python oracle/gen_golden_host.py

reference_flags.json     dglke_train's option table (CommonArgParser) and the train-only flags its train.py adds
reference_datasets.json  what the reference's dataset readers return for the files tests/test_dataset.py writes

TEST INFRASTRUCTURE ONLY: the tests compare the package against these files and never import the reference.
"""
import importlib
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "dgl-ke_b200"), os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import ref_harness as rh  # noqa: E402
import test_dataset as td  # noqa: E402
from test_host_logic import flag_table  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "host")


def flags():
    rh.import_reference()
    common = flag_table(importlib.import_module("dglke.utils").CommonArgParser())
    # importing dglke.train needs more of DGL than the stand-ins provide: its own add_argument calls are read instead
    src = open(os.path.join(rh.REFERENCE_PY, "dglke", "train.py")).read()
    return dict(common=common, train_only=re.findall(r"add_argument\(\s*['\"](--[A-Za-z0-9_]+)['\"]", src))


def datasets():
    rh.import_reference()
    kg = importlib.import_module("dglke.dataloader.KGDataset")

    def no_download(url, path, filename):
        raise RuntimeError("the reference reader tried to download %s" % url)
    kg._download_and_extract = no_download          # every layout below exists on disk
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for order in td.ORDERS:
            for delim in td.DELIMS:
                d = tempfile.mkdtemp(dir=tmp)
                td.write_udd_case(d, order, delim)
                out["udd_" + order + delim] = td.summary(kg.get_dataset(d, "mine", "udd_" + order, delim, td.UDD_FILES))
        for order in td.RAW_ORDERS:
            d = os.path.join(tmp, "raw_" + order)
            td.write_raw_udd_case(d, order)
            out["raw_udd_" + order] = td.summary(kg.get_dataset(d, "mykg", "raw_udd_" + order, "\t", td.RAW_FILES), d)
        d = tempfile.mkdtemp(dir=tmp)
        td.write_built_in_case(d)
        for name in ("FB15k", "Freebase"):
            out["built_in_" + name] = td.summary(kg.get_dataset(d, name, "built_in"))
    return out


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    for name, fn in (("reference_flags.json", flags), ("reference_datasets.json", datasets)):
        with open(os.path.join(OUT, name), "w") as f:
            json.dump(fn(), f, separators=(",", ":"))
            f.write("\n")
        print("wrote", name, os.path.getsize(os.path.join(OUT, name)), "bytes")
