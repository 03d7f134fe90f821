"""Record the reference's own CUDA kernels on the inputs of tests/test_gpu_vs_ref_cuda.py.

Test infrastructure; needs a B200 and oracle/_ref/libvptq.so (the unmodified reference extension, built
by oracle/build_ref.sh).  For every case of that test it runs the reference's quant_gemv (1 and 2 tokens)
and dequant on exactly the tensors the test builds, and stores their 16-bit outputs as raw bits:

  gemv/<case>/<tokens>   the whole output [tokens, out_features]
  dequant/<case>         a fixed, seeded sample of the weight matrix (positions in dequant_pos/<case>)
  sha/...                a digest of the inputs, so that a change of the seeded layers is caught

    python oracle/make_ref_cuda_golden.py [OUT_DIR]     # default tests/golden/ref_cuda/
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, os.path.join(ROOT, "tests"), ROOT):
    sys.path.insert(0, p)
import vptq_oracle as vo  # noqa: E402
from _gpu import make_module, x_to_t  # noqa: E402
from test_gpu_vs_ref_cuda import (CASES, DEQUANT_CASES, DEQUANT_SAMPLES, GEMV_TOKENS, bits,  # noqa: E402
                                  input_digest)


def ref_tensors(L, m):
    G, v = L.num_codebooks, L.vector_len
    cent = m.centroids.weight.view(G, L.num_centroids, v)
    rcent = m.res_centroids.weight.view(G, L.num_res_centroids, v) if L.res_bits else None
    ocent = m.outlier_centroids.weight.view(1, L.num_outlier_centroids, L.outlier_vector_len) if L.enable_outlier else None
    return cent, rcent, ocent


def main(out_dir):
    so = os.path.join(HERE, "_ref", "libvptq.so")
    spec = importlib.util.spec_from_file_location("libvptq", so)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    out = {}
    for name in sorted(CASES):
        L = vo.make_layer(seed=2024, **CASES[name])
        m = make_module(L)
        cent, rcent, ocent = ref_tensors(L, m)
        xs = [vo.make_x(t, L.in_features, L.dtype, seed=t) for t in GEMV_TOKENS]
        out[f"sha/gemv/{name}"] = np.array(input_digest(L, xs))
        for tokens, x_np in zip(GEMV_TOKENS, xs):
            y = ref.quant_gemv(x_to_t(x_np, L), m.indices, cent, None, rcent, m.outlier_indices, ocent, m.perm,
                               m.weight_scale, m.weight_bias, m.bias, L.in_features, L.out_features)
            torch.cuda.synchronize()
            out[f"gemv/{name}/{tokens}"] = bits(y)
            print(f"gemv {name} tokens={tokens}: finite={bool(torch.isfinite(y).all())}")
    for name in DEQUANT_CASES:
        L = vo.make_layer(seed=2025, **CASES[name])
        m = make_module(L)
        cent, rcent, ocent = ref_tensors(L, m)
        inv = torch.argsort(m.perm.view(torch.uint16).to(torch.int64)).to(torch.uint16).view(torch.int16)
        W = ref.dequant(m.indices, cent, None, rcent, m.outlier_indices, ocent, inv, m.weight_scale,
                        m.weight_bias, L.vector_len, L.in_features, L.out_features)
        torch.cuda.synchronize()
        assert tuple(W.shape) == (L.out_features, L.in_features)
        pos = np.sort(np.random.default_rng(7).choice(W.numel(), DEQUANT_SAMPLES, replace=False)).astype(np.int32)
        out[f"sha/dequant/{name}"] = np.array(input_digest(L, []))
        out[f"dequant_pos/{name}"] = pos
        out[f"dequant/{name}"] = bits(W).reshape(-1)[pos]
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "outputs.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path} ({os.path.getsize(path)} bytes)")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_cuda"))
