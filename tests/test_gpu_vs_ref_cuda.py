"""GPU-side anchor: our kernels vs the UNMODIFIED reference CUDA kernels on identical tensors.

The reference's outputs are stored under tests/golden/ref_cuda/ (recorded on a B200 by
oracle/make_ref_cuda_golden.py from the reference extension compiled for sm_100a by oracle/build_ref.sh),
so this comparison runs without the reference.  The inputs are the seeded layers below; their digest is
stored with the outputs and checked first.

north_star: "Outputs match the reference kernels on identical (indices, centroids,
residual_centroids, perm, outliers, x) within 1e-3 relative fp16".  The reference GEMV accumulates
four columns per thread in fp16 (csrc/kernels/quant_gemv.cuh:34,140-141), so its own distance to
exact arithmetic is a few 1e-4; both distances are asserted.
"""
import hashlib
import os

import numpy as np
import pytest

import vptq_oracle as vo
from _util import GOLDEN_DIR, parity_error

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(GOLDEN_DIR, "ref_cuda", "outputs.npz")
GEMV_TOKENS = (1, 2)
DEQUANT_CASES = ["llama3_k65536_r256", "outliers", "bf16"]
DEQUANT_SAMPLES = 32768       # stored elements of each reference weight matrix (seeded positions)


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN, allow_pickle=False)


CASES = {
    "llama3_k65536_r256": dict(in_features=4096, out_features=1024, vector_len=8, num_centroids=65536, num_res_centroids=256),
    "k65536_r0": dict(in_features=2048, out_features=1024, vector_len=8, num_centroids=65536),
    "cfg1_k256": dict(in_features=4096, out_features=4096, vector_len=8, num_centroids=256),
    "k4096_r4096_v12": dict(in_features=1536, out_features=768, vector_len=12, num_centroids=4096, num_res_centroids=4096),
    "outliers": dict(in_features=2048 + 128, out_features=1024, vector_len=8, num_centroids=4096, num_res_centroids=256,
                     outlier_size=128, outlier_vector_len=4, num_outlier_centroids=4096, bias=True),
    "bf16": dict(in_features=2048, out_features=1024, vector_len=8, num_centroids=65536, num_res_centroids=256, dtype="bf16"),
}


def input_digest(L, xs):
    """sha256 over every input tensor of the layer and the activations."""
    h = hashlib.sha256()
    for a in (L.indices, L.centroids, L.res_centroids, L.outlier_indices, L.outlier_centroids, L.perm,
              L.weight_scale, L.weight_bias, L.bias, *xs):
        h.update(b"-" if a is None else np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def bits(t):
    """16-bit CUDA tensor -> its raw bits (uint16 numpy)."""
    import torch
    return t.detach().contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


def from_bits(b, dtype):
    return vo.to_f32(b.view(np.float16) if dtype == "fp16" else b, dtype)


@pytest.mark.parametrize("name", sorted(CASES))
def test_gemv_matches_reference_cuda(ref, name):
    import torch
    from _gpu import from_t, make_module, x_to_t
    L = vo.make_layer(seed=2024, **CASES[name])
    xs = [vo.make_x(t, L.in_features, L.dtype, seed=t) for t in GEMV_TOKENS]
    assert str(ref[f"sha/gemv/{name}"]) == input_digest(L, xs), "seeded inputs differ from the recorded ones"
    m = make_module(L)
    tol = 1e-3 if L.dtype == "fp16" else 8e-3
    for tokens, x_np in zip(GEMV_TOKENS, xs):
        y_ours = from_t(m(x_to_t(x_np, L)))
        torch.cuda.synchronize()
        y_ref = from_bits(ref[f"gemv/{name}/{tokens}"], L.dtype)
        assert y_ours.shape == y_ref.shape
        y_star = vo.quant_gemm(x_np, L)
        e_ours = parity_error(y_ours, y_star)
        assert e_ours <= tol
        if not np.isfinite(y_ref).all():
            # seen on B200 for the outlier configuration: the reference kernel returned NaN in one run and
            # finite values in others on the same inputs; nothing to compare with then -- our distance to
            # exact arithmetic is asserted above
            print(f"{name} tokens={tokens}: ours-vs-exact {e_ours:.2e}  reference kernel output is not finite, skipped")
            continue
        e_ref, e_mut = parity_error(y_ref, y_star), parity_error(y_ours, y_ref)
        print(f"{name} tokens={tokens}: ours-vs-exact {e_ours:.2e}  ref-vs-exact {e_ref:.2e}  ours-vs-ref {e_mut:.2e}")
        assert e_mut <= max(tol, 2 * e_ref), (e_mut, e_ref)


@pytest.mark.parametrize("name", DEQUANT_CASES)
def test_dequant_matches_reference_cuda(ref, name):
    import torch
    from _gpu import from_t, make_module
    L = vo.make_layer(seed=2025, **CASES[name])
    assert str(ref[f"sha/dequant/{name}"]) == input_digest(L, []), "seeded inputs differ from the recorded ones"
    m = make_module(L)
    W = from_t(m.dequant())
    torch.cuda.synchronize()
    assert W.shape == (L.out_features, L.in_features)
    pos = ref[f"dequant_pos/{name}"]
    W, W_ref = W.reshape(-1)[pos], from_bits(ref[f"dequant/{name}"], L.dtype)
    # the reference rounds C+R to 16 bit and then fma-rounds again (csrc/kernels/dequant.cuh:87,98);
    # ours evaluates in fp32 and rounds once.  |diff| <= ulp * (|W| + 0.5*|C+R|*|scale|), and
    # |C+R|*|scale| <= |W| + |wbias|.
    ulp = 2.0 ** -10 if L.dtype == "fp16" else 2.0 ** -7
    wb = np.abs(vo.to_f32(L.weight_bias, L.dtype)).max()
    bound = 2 * ulp * (np.abs(W_ref) + wb) + 1e-7
    bad = np.abs(W - W_ref) > bound
    assert not bad.any(), f"{int(bad.sum())} of {bad.size} sampled elements beyond the double-rounding bound"
