"""Option B of INTEGRATION.md as a real file: copy it to `vptq/libvptq.py` of a reference checkout (or put this
directory's parent on sys.path as package `vptq`) and the reference's own python -- `vptq/ops/quant_gemm.py:22-26`
does `import vptq.libvptq as vptq_ops` -- runs on libvptq_b200.so through the C ABI of include/vptq_b200.h.
The three functions below have the signatures of the reference's pybind11 module (csrc/ops.cc:9-38,44-55).
tests/test_host_logic.py::test_reference_python_binds_our_library_through_the_stub replays against this module
the calls the reference's quant_gemm.py makes into it (recorded by oracle/make_stub_calls.py)."""
import ctypes, torch
from vptq_b200 import native          # LinearDesc (= struct vptq_linear_desc), lib(), check(), workspace()

def _desc(q_indice, centroids, residual_centroids, q_indice_outliers, outliers_centroids, perm,
          weight_scale, weight_bias, bias, in_features, out_features):
    G, K, v = centroids.shape                      # [num_codebooks, num_centroids, vector_len]
    S = 0 if q_indice_outliers is None else q_indice_outliers.shape[-1]
    return native.make_desc(
        dtype=centroids.dtype, in_features=in_features, out_features=out_features, vector_len=v,
        num_centroids=K, num_res_centroids=-1 if residual_centroids is None else residual_centroids.shape[1],
        num_codebooks=G, group_size=(in_features - S) // G, outlier_size=S,
        outlier_vector_len=-1 if outliers_centroids is None else outliers_centroids.shape[-1],
        num_outlier_centroids=-1 if outliers_centroids is None else outliers_centroids.shape[1],
        indices=q_indice, centroids=centroids, res_centroids=residual_centroids,
        outlier_indices=q_indice_outliers, outlier_centroids=outliers_centroids, perm=perm,
        weight_scale=weight_scale, weight_bias=weight_bias, bias=bias)

def quant_gemv(input, q_indice, centroids, q_indice_residual, residual_centroids, q_indice_outliers,
               outliers_centroids, perm, weight_scale, weight_bias, bias, in_features, out_features):
    # replaces vptq::wquant_act16_gemv (csrc/quant_gemv.cu:241-294); note the reference passes PERM here
    assert q_indice_residual is None, "packed layers keep the residual index inside q_indice"
    d = _desc(q_indice, centroids, residual_centroids, q_indice_outliers, outliers_centroids, perm,
              weight_scale, weight_bias, bias, in_features, out_features)
    x2 = input.reshape(-1, in_features)
    y = torch.empty(x2.shape[0], out_features, dtype=input.dtype, device=input.device)   # caller allocates
    native.quant_gemv(d, x2, y)                    # -> vptq_b200_quant_gemv(desc, x, ldx, y, ldy, tokens, ws, ws_bytes, flags, stream)
    return y.reshape(*input.shape[:-1], out_features)

def dequant(q_indice, centroids, q_indice_residual, residual_centroids, q_indice_outliers,
            outliers_centroids, invperm, weight_scale, weight_bias, groupsize, in_features, out_features):
    # replaces vptq::dequant (csrc/dequant.cu:227-287).  The reference passes argsort(perm) here
    # (quant_gemm.py:208-211,239); the C ABI wants perm itself and inverts on the device.
    perm = None if invperm is None else torch.argsort(invperm.view(torch.uint16).to(torch.int64)).to(torch.int16)
    d = _desc(q_indice, centroids, residual_centroids, q_indice_outliers, outliers_centroids, perm,
              weight_scale, weight_bias, None, in_features, out_features)
    w = torch.empty(out_features, in_features, dtype=centroids.dtype, device=centroids.device)
    native.dequant(d, w)                           # -> vptq_b200_dequant(desc, w_out, ws, ws_bytes, stream)
    return w

def quant_gemv_v2(act, bias, indices, centroids, residual_indices, residual_centroids, scale_weights,
                  scale_bias, out_features):
    from vptq_b200.ops import quant_gemv_v2 as f   # -> vptq_b200_quant_gemv_v2(...)
    G, K, v = centroids.shape
    Kr = 0 if residual_centroids is None else residual_centroids.shape[1]
    return f(act, bias, indices, centroids, residual_indices, residual_centroids, scale_weights, scale_bias, v, G, K, Kr, out_features)
