"""CPU: the drop-in boundary as the reference's training scripts use it (SURVEY 8b, INTEGRATION.md recipe A).

With ``PYTHONPATH=<repo>:<reference>`` the UNMODIFIED ``train_small_graphs.py``, ``train_pubmed.py`` and
``train_large_graphs.py`` must import (they do ``from utils import *`` and rely on the reference's whole ``utils``
namespace, which the repo's ``utils.py`` re-exports), parse their default arguments, and construct every DGG model
through the string lookup ``models.__dict__[args.model](..., args=args)`` (train_small_graphs.py:387-397) -- against
THIS repo's ``model.py`` / ``dgm.py``.  Runs only where ``DGG_REFERENCE_ROOT`` names a reference checkout;
``torch_geometric`` is not installable here, so the test registers the oracle's stub first (test infrastructure)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("DGG_REFERENCE_ROOT", "")

pytestmark = pytest.mark.skipif(not REF, reason="no reference checkout (set DGG_REFERENCE_ROOT)")

MODELS = ["GCN_DGG", "GCN_DGG_00", "GCN_DGG_Ablations", "GCN_DGG_00_LargeGraphs", "GCNII_DGG", "SAGE_DGG",
          "SAGE_DGG_00", "GAT_DGG_00", "GAT_DGG_Ablations", "GCN", "GCNII", "SAGE", "GAT"]

CHILD = r'''
import os, sys, types
import torch
from oracle import ref_loader
ref_loader.install_pyg_stub()                       # PyG is not installable in this container
import torch_geometric
for sub in ("transforms", "datasets", "loader"):    # the scripts only touch these inside load_data / main
    assert hasattr(torch_geometric, sub)
import utils, model as models, dgm
here = os.environ["DGGB_REPO_ROOT"]
assert os.path.samefile(os.path.dirname(models.__file__), here), models.__file__      # OUR model.py / dgm.py
assert os.path.samefile(os.path.dirname(dgm.__file__), here), dgm.__file__
assert os.path.samefile(os.path.dirname(utils.__file__), here)
assert utils.REFERENCE_UTILS and os.path.samefile(os.path.dirname(utils.REFERENCE_UTILS), os.environ["DGGB_REF_ROOT"])
for name in ("load_citation", "remove_interclass_edges", "calc_learned_edges_stats", "accuracy", "str2bool",
             "add_noisy_edges", "sparse_mx_to_torch_sparse_tensor", "np", "torch", "F"):
    assert hasattr(utils, name), name
assert utils.add_noisy_edges.__module__ == "utils" and "chunk_rows" in utils.add_noisy_edges.__code__.co_varnames
built = []
for script in ("train_small_graphs", "train_pubmed", "train_large_graphs"):
    mod = __import__(script)                         # module level: imports + the argparse definitions only
    args = mod.parser.parse_args([])
    for name in os.environ["DGGB_MODELS"].split(","):
        args.model = name
        net = models.__dict__[args.model](nfeat=33, nlayers=args.layer, nhidden=args.hidden, nclass=5,
                                          dropout=args.dropout, lamda=args.lamda, alpha=args.alpha,
                                          variant=args.variant, args=args)
        n_par = sum(p.numel() for p in net.parameters())
        assert n_par > 0
        if "GCN" in name:
            assert len(net.params1) > 0 and len(net.params2) > 0     # optimiser groups (train_small_graphs.py:399-414)
        built.append((script, name))
print("BUILT", len(built))
'''


def test_unmodified_scripts_import_and_build_every_model(tmp_path):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, REF])
    env["DGGB_REPO_ROOT"], env["DGGB_REF_ROOT"], env["DGGB_MODELS"] = ROOT, REF, ",".join(MODELS)
    # cwd: neither tree (python -c puts the cwd first on sys.path; PYTHONPATH order is what is under test)
    res = subprocess.run([sys.executable, "-W", "ignore", "-c", CHILD], cwd=str(tmp_path), env=env,
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert "BUILT %d" % (3 * len(MODELS)) in res.stdout


def test_launcher_puts_the_repo_before_the_script_directory():
    """``python <reference>/train_x.py`` prepends the SCRIPT's directory to sys.path, which would shadow the drop-in
    ``model.py``; ``run_reference_script.py`` (and ``python -P`` on 3.11+) keeps the repo first."""
    code = ("import sys; sys.argv=['run_reference_script.py', %r, '--help']\n"
            "import runpy\n"
            "try:\n    runpy.run_path(%r, run_name='__main__')\nexcept SystemExit as e:\n    print('EXIT', e.code)\n"
            "import model, os; print('MODEL', os.path.dirname(os.path.abspath(model.__file__)))\n"
            % (os.path.join(REF, "train_small_graphs.py"), os.path.join(ROOT, "run_reference_script.py")))
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    env["DGGB_PYG_STUB"] = "1"
    res = subprocess.run([sys.executable, "-W", "ignore", "-c", code], cwd=REF, env=env, capture_output=True, text=True,
                         timeout=600)
    assert "EXIT 0" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]       # argparse --help exits 0
    assert "MODEL " + ROOT in res.stdout
