"""Import the UNMODIFIED reference modules under the chainer stub from the checkout of the original
chainer-differentiable-mpc that DIFFMPC_REFERENCE names.

Not part of the test suite.  Used by
tests/golden/make_golden.py to produce the committed fixtures and to pin the
numpy oracle (oracle/) against the live reference.

Shims applied (SURVEY.md H1/H8):
  * torch.lu_solve needs a 3-D right-hand side with torch>=1.9 -> unsqueeze/squeeze.
  * `lu_fp32=False` additionally removes the reference's float32 cast inside
    util.xpbatch_lu_solve (util.py:522-526) so the live reference becomes the
    "fp64-clean" oracle the 1e-10 parity target is defined against.
"""
import importlib
import os
import sys

import numpy as np

REF = os.environ.get("DIFFMPC_REFERENCE", "")
HERE = os.path.dirname(os.path.abspath(__file__))
STUB = os.path.join(os.path.dirname(HERE), "_chainer_stub")


def available():
    return bool(REF) and os.path.isdir(os.path.join(REF, "lqr"))


def load(lu_fp32=True):
    """Returns a dict of the reference modules."""
    assert available(), "set DIFFMPC_REFERENCE to a checkout of the original chainer-differentiable-mpc"
    for p in (STUB, REF, os.path.join(REF, "lqr"), os.path.join(REF, "mpc")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    util = importlib.import_module("util")

    def xpbatch_lu_solve(lu_and_piv, b):
        LU, piv = lu_and_piv
        b = np.array(b, copy=True)
        vec = (b.ndim == 2)
        tb = torch.from_numpy(b)
        tLU = torch.from_numpy(np.asarray(LU))
        tpiv = torch.from_numpy(np.asarray(piv))
        if lu_fp32:
            tb = tb.float()
            tLU = tLU.float()
        if vec:
            tb = tb.unsqueeze(-1)
        out = torch.lu_solve(tb, tLU, tpiv)
        if vec:
            out = out.squeeze(-1)
        return out.cpu().numpy()

    util.xpbatch_lu_solve = xpbatch_lu_solve
    mods = {"util": util}
    for name in ("lqr_recursion", "differentiable_lqr", "pnqp", "active_constrained_lqr",
                 "mpc_step", "box_ddp"):
        try:
            m = importlib.import_module(name)
        except Exception as e:  # approximate.py etc. only need chainer symbols
            raise RuntimeError("cannot import reference module %s: %r" % (name, e))
        if hasattr(m, "xpbatch_lu_solve"):
            m.xpbatch_lu_solve = xpbatch_lu_solve
        mods[name] = m
    return mods
