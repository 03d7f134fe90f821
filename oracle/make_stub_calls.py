"""Record the calls the REFERENCE's python makes into its CUDA extension module, as tests/golden/ref_stub_calls.json.

Test infrastructure; needs the reference tree (oracle/ref_shim.REF).  The reference's vptq/ops/quant_gemm.py is
loaded with a recorder standing where its pybind module `vptq.libvptq` would be, and quant_gemm is called on a
seeded layer with 1 token (its quant_gemv branch) and 4 tokens (its dequant branch).  Each call is stored as the
function name and, per positional argument, None, the int, or the tensor's shape and dtype.
tests/test_host_logic.py replays these calls against integration/libvptq.py.

    python oracle/make_stub_calls.py
"""
import importlib.util
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402
import vptq_oracle as vo  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_stub_calls.json")


def describe(a):
    if a is None or isinstance(a, (bool, int)):
        return a
    if isinstance(a, torch.Tensor):
        return {"shape": list(a.shape), "dtype": str(a.dtype).replace("torch.", "")}
    raise TypeError(type(a))


def main():
    calls = []

    class Recorded(Exception):
        pass

    def recorder(name):
        def f(*args, **kwargs):
            assert not kwargs, kwargs
            calls.append({"fn": name, "args": [describe(a) for a in args]})
            raise Recorded
        return f

    rec = types.ModuleType("vptq.libvptq")
    for n in ("quant_gemv", "dequant", "quant_gemv_v2"):
        setattr(rec, n, recorder(n))
    saved = {k: v for k, v in sys.modules.items() if k == "vptq" or k.startswith("vptq.")}
    for k in saved:
        del sys.modules[k]
    for pkg in ("vptq", "vptq.utils", "vptq.ops"):
        sys.modules[pkg] = types.ModuleType(pkg)
        sys.modules[pkg].__path__ = [os.path.join(ref_shim.REF, *pkg.split("."))]
    for name in ("accelerate", "sentence_transformers"):
        sys.modules.setdefault(name, types.ModuleType(name))
    st = types.ModuleType("sentence_transformers.SentenceTransformer")
    st.SentenceTransformer = type("SentenceTransformer", (), {})
    sys.modules.setdefault("sentence_transformers.SentenceTransformer", st)
    sys.modules["vptq.libvptq"] = rec
    sys.modules["vptq"].libvptq = rec

    def load(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m

    load("vptq.utils.pack", os.path.join(ref_shim.REF, "vptq/utils/pack.py"))
    qg = load("vptq.ops.quant_gemm", os.path.join(ref_shim.REF, "vptq/ops/quant_gemm.py"))
    assert qg.__dict__["__cuda_ops_installed"] is True and qg.vptq_ops is rec
    L = vo.make_layer(in_features=256, out_features=64, vector_len=8, num_centroids=256, num_res_centroids=16, seed=3)
    t = lambda a, dt: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).view(dt)
    for tokens in (1, 4):
        x = torch.zeros(tokens, 256, dtype=torch.float16)
        try:
            qg.quant_gemm(x, None, t(L.indices, torch.int32), t(L.centroids, torch.float16).view(1, -1), None, None, None,
                          t(L.res_centroids, torch.float16).view(1, -1), t(L.perm, torch.int16),
                          t(L.weight_scale, torch.float16), t(L.weight_bias, torch.float16), 8, -1, 1, 256, -1, 16, True,
                          256, 0, 256, 64, 0, 0)
        except Recorded:
            pass
    assert [c["fn"] for c in calls] == ["quant_gemv", "dequant"], calls
    with open(OUT, "w") as f:
        json.dump(calls, f, indent=1)
        f.write("\n")
    print(f"wrote {OUT}")


if __name__ == "__main__":
    main()
