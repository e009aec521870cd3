"""`python -m tsg.run <reference script>`: every training script of the three reference directories, UNMODIFIED, on a
tiny synthetic TU-format dataset (40 PROTEINS-shape graphs written by tsg.tu.write, read back by the scripts' own loaders).

 * reach: through the real launcher path each script gets past imports, argparse, data loading, preprocessing and model
   construction and into its first forward, where the tsg drop-in refuses the CPU tensor ("no CPU path") -- with the B2
   patches sitting on the script's OWN classes at that moment.
 * e2e: the launcher's compat layer (SURVEY A.3 shims) carries every script to its final print on CPU with the
   reference's own math (sag over the oracle-backed torch_geometric), including the stage-2 code after training that
   crashes as shipped (evaluate() signature, int into os.environ, int default of a str option, np.matrix into sklearn).

The script cases need the original project's source tree (launcher_driver.REF) and skip without it.  One helper
process per mode runs all cases concurrently."""
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

sys.path.insert(0, HERE)
from launcher_driver import REF, cases  # noqa: E402

needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "sag")),
                                     reason="the original project's source tree is not present")

IDS = [f"{d}-{s}" + (f"-{m}" if m else "") for d, s, m, _ in cases()]


def _run(mode, tmp):
    r = subprocess.run([sys.executable, os.path.join(HERE, "launcher_driver.py"), mode, str(tmp)], capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    return {f"{x['dir']}-{x['script']}" + (f"-{x['method']}" if x.get("method") else ""): x for x in res}


@pytest.fixture(scope="module")
def reach(tmp_path_factory):
    return _run("reach", tmp_path_factory.mktemp("reach"))


@pytest.fixture(scope="module")
def e2e(tmp_path_factory):
    return _run("e2e", tmp_path_factory.mktemp("e2e"))


@needs_reference
@pytest.mark.parametrize("case", IDS)
def test_script_reaches_the_tsg_drop_ins(reach, case):
    r = reach[case]
    assert not r["ok"] and "no CPU path" in r["error"], f"{case}: {r['error']}\n{r['tail']}"
    where = r["where"]
    d = case.split("-")[0]
    if d == "sag":
        # train*.py -> tripletnet / network.py (reference) -> tsg.nn.GCNConv.forward
        assert any(w.startswith("sag/network.py") for w in where), where
        assert any(w.startswith("tsg/nn.py:forward") for w in where), where
        assert r["script_classes_patched"] == {"network.GCNConv is tsg.nn.GCNConv": True}
    else:
        assert any(w.endswith("encoders.py:forward") or w.endswith("encoders_GAT.py:forward") for w in where), where
        assert any(w.startswith("tsg/dense_patch.py") for w in where), where
        assert r["script_classes_patched"] and all(r["script_classes_patched"].values()), r["script_classes_patched"]
        if "GAT" in case:
            assert r["script_classes_patched"].get("encoders_GAT.DGATHead.forward") is True
            assert any(w == "tsg/dense_patch.py:dgathead_forward" for w in where), where
        if d == "eigengcn":
            assert r["script_classes_patched"].get("encoders.Pool.forward") is True


@needs_reference
@pytest.mark.parametrize("case", IDS)
def test_compat_layer_carries_the_script_to_its_end(e2e, case):
    r = e2e[case]
    assert r["ok"], f"{case}: {r['error']}\n{r['where']}\n{r['tail']}"
    assert "accuracy" in r["tail"] or "performance" in r["tail"], r["tail"]
    if case == "sag-train_triplet_pre_train":
        assert r["fixes"], "the evaluate() signature fix did not apply"


def test_device_hygiene_shims_unit():
    """The CPU<->CUDA mixing shims are no-ops for matching devices (their CUDA side is tests/test_shim.py's gpu test)."""
    import torch
    import torch.nn.functional as F
    from tsg import run
    run.install()
    m = torch.nn.Sequential(torch.nn.Linear(3, 2))
    x = torch.randn(4, 3)
    assert m(x).shape == (4, 2)
    assert F.cross_entropy(m(x), torch.tensor([0, 1, 0, 1])).ndim == 0
    assert bool(torch.tensor([1, 2]).eq(torch.tensor([1, 3]))[0])
    os.environ["TSG_TEST_INT"] = 3
    assert os.environ.pop("TSG_TEST_INT") == "3"
    import argparse
    p = argparse.ArgumentParser(); p.add_argument("--pool_sizes", type=str, default="10"); p.set_defaults(pool_sizes=10)
    assert p.parse_args([]).pool_sizes == "10"
