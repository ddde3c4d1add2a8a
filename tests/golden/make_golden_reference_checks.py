"""Golden data for the tests that compare the oracle with the reference package itself
(atong01/conditional-flow-matching @ cacd4dc8, torchcfm 1.0.7), so that they run without a checkout of it:

    python tests/golden/make_golden_reference_checks.py <path of a reference checkout>

writes
  reference_signatures.json  public signatures of the reference classes, parsed from its source
  reference_checks.npz       glue_*: OTPlanSampler.get_map / sample_plan of the unmodified reference on the
                             oracle POT shim;  shim_*: the calls the reference's OWN test suite made into that shim
                             while it passed (134 tests), with their inputs and results

The reference's suite runs in a subprocess with this file loaded as a pytest plugin (-p): the plugin wraps the
shim's public functions and torch.cdist and records each outermost shim call.  To keep the file small:
  * calls that differ only in their random inputs are recorded once;
  * a cost matrix is stored as the two point sets it is the torch.cdist of, with its form (d, d**2 or
    d**2 / max) -- every cost matrix the suite builds is one of these;
  * a result of more than SMALL entries is stored as its row sums, column sums, the column of each row's largest
    entry (the whole assignment of an exact plan) and a seeded sample of entries.
"""
import ast
import json
import os
import pickle
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SHIM_FUNCS = ("unif", "emd", "emd2", "sinkhorn", "sinkhorn2")
SMALL, N_SAMPLE = 1024, 512
SIG_CLASSES = {
    "torchcfm/optimal_transport.py": ["OTPlanSampler"],
    "torchcfm/conditional_flow_matching.py": ["ConditionalFlowMatcher", "ExactOptimalTransportConditionalFlowMatcher",
                                              "TargetConditionalFlowMatcher", "SchrodingerBridgeConditionalFlowMatcher",
                                              "VariancePreservingConditionalFlowMatcher"],
    "torchcfm/models/models.py": ["MLP"],
}


def cost_from_points(x0, x1, form):
    """The cost matrix of `form` between two point sets, computed the way the reference computes it."""
    import torch
    d = torch.cdist(torch.from_numpy(x0), torch.from_numpy(x1))
    if form == "d":
        return d.numpy()
    d2 = d ** 2
    return (d2 / d2.max() if form == "d2n" else d2).numpy()


def sample_index(shape):
    """The entries of a large result that are stored: fixed by the seed, the same in generator and test."""
    return np.random.default_rng(0).choice(int(np.prod(shape)), size=N_SAMPLE, replace=False)


# ---------------------------------------------------------------- pytest plugin side (inside the reference run)
_calls, _depth, _cdist = [], [0], []


def _wrap(mod, name):
    fn = getattr(mod, name)

    def wrapped(*args, **kwargs):
        _depth[0] += 1
        try:
            out = fn(*args, **kwargs)
        finally:
            _depth[0] -= 1
        if _depth[0] == 0:  # sinkhorn2 calls sinkhorn: only the call the reference made is recorded
            _calls.append((name, [np.array(a) if isinstance(a, np.ndarray) else a for a in args], dict(kwargs),
                           np.array(out), _cdist[-1] if _cdist else None))
        return out

    setattr(mod, name, wrapped)


def pytest_configure(config):
    if os.environ.get("CFM_GOLDEN_RECORD"):
        import ot
        import torch
        assert "oracle" in ot.__version__, ot.__file__
        for name in SHIM_FUNCS:
            _wrap(ot, name)
        cdist = torch.cdist

        def cdist_recorded(a, b, *args, **kwargs):
            _cdist[:] = [(a.detach().numpy().copy(), b.detach().numpy().copy())]
            return cdist(a, b, *args, **kwargs)

        torch.cdist = cdist_recorded


def pytest_unconfigure(config):
    path = os.environ.get("CFM_GOLDEN_RECORD")
    if path:
        with open(path, "wb") as f:
            pickle.dump(_calls, f)


# ---------------------------------------------------------------- generator side
def signatures(reference):
    out = {}
    for rel, classes in SIG_CLASSES.items():
        tree = ast.parse(open(os.path.join(reference, rel)).read())
        for node in tree.body:
            if isinstance(node, ast.ClassDef) and node.name in classes:
                for fn in node.body:
                    if isinstance(fn, ast.FunctionDef) and (not fn.name.startswith("_") or fn.name == "__init__"):
                        out[f"{node.name}.{fn.name}"] = [a.arg for a in fn.args.args]
            if isinstance(node, ast.FunctionDef) and not node.name.startswith("_"):
                out[node.name] = [a.arg for a in node.args.args]
    return out


def glue(out):
    import torch
    from torchcfm.optimal_transport import OTPlanSampler
    torch.manual_seed(5)
    x0, x1 = torch.randn(64, 3, 2), torch.randn(64, 3, 2)
    out["glue_x0"], out["glue_x1"] = x0.numpy(), x1.numpy()
    for tag, method, kw in (("exact", "exact", {}), ("sk03", "sinkhorn", dict(reg=0.3)),
                            ("sk005n", "sinkhorn", dict(reg=0.05, normalize_cost=True))):
        ref = OTPlanSampler(method, **kw)
        out[f"glue_{tag}_pi"] = ref.get_map(x0, x1)
        np.random.seed(3)
        a, b = ref.sample_plan(x0, x1)
        out[f"glue_{tag}_a"], out[f"glue_{tag}_b"] = a.numpy(), b.numpy()


def record_reference_suite(reference, out):
    with tempfile.TemporaryDirectory() as tmp:
        rec = os.path.join(tmp, "calls.pkl")
        env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "oracle"), reference, HERE]),
                   CFM_GOLDEN_RECORD=rec)
        r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(reference, "tests"), "-p",
                            "make_golden_reference_checks", "-p", "no:cacheprovider", "-c", os.devnull,
                            f"--rootdir={tmp}", "-q"], cwd=tmp, env=env, capture_output=True, text=True)
        tail = r.stdout.strip().splitlines()[-1]
        assert r.returncode == 0 and "134 passed" in tail, r.stdout[-3000:] + r.stderr[-2000:]
        calls = pickle.load(open(rec, "rb"))
    meta, seen = [], set()
    for name, args, kwargs, res, points in calls:
        key = (name, repr([(a.shape, a.dtype.str) if isinstance(a, np.ndarray) else a for a in args]),
               repr(sorted(kwargs.items())))
        if key in seen:
            continue
        seen.add(key)
        k = len(meta)
        entry = {"fn": name, "args": [], "kwargs": kwargs, "out_shape": list(res.shape), "out_dtype": res.dtype.str}
        for i, a in enumerate(args):
            if not isinstance(a, np.ndarray):
                entry["args"].append(a)
            elif a.ndim == 1 and np.array_equal(a, np.full(a.shape, 1.0 / a.size)):
                entry["args"].append({"unif": a.size})
            else:
                form = next(f for f in ("d", "d2", "d2n") if points is not None
                            and np.array_equal(cost_from_points(*points, f), a))
                out[f"shim_{k}_arg{i}_x0"], out[f"shim_{k}_arg{i}_x1"] = points
                entry["args"].append({"cost": form})
        if res.size <= SMALL:
            out[f"shim_{k}_out"] = res
        else:
            out[f"shim_{k}_out_rows"] = res.sum(1, dtype=np.float64)
            out[f"shim_{k}_out_cols"] = res.sum(0, dtype=np.float64)
            out[f"shim_{k}_out_argmax"] = res.argmax(1)
            out[f"shim_{k}_out_sample"] = res.reshape(-1)[sample_index(res.shape)]
        meta.append(entry)
    out["shim_calls"] = np.array(json.dumps(meta))
    return len(calls), len(meta), tail


def main():
    reference = os.path.abspath(sys.argv[1])
    sys.path[:0] = [os.path.join(ROOT, "oracle"), reference]
    import ot
    assert "oracle" in ot.__version__, ot.__file__
    import torchcfm
    assert torchcfm.__file__.startswith(reference), torchcfm.__file__

    sig_path = os.path.join(HERE, "reference_signatures.json")
    with open(sig_path, "w") as f:
        json.dump(signatures(reference), f, indent=1, sort_keys=True)
        f.write("\n")
    out = {}
    glue(out)
    n_calls, n_kept, tail = record_reference_suite(reference, out)
    path = os.path.join(HERE, "reference_checks.npz")
    np.savez_compressed(path, **out)
    print("wrote", sig_path, path, f"({n_calls} shim calls, {n_kept} kept; reference suite: {tail})")


if __name__ == "__main__":
    main()
