"""CPU-side tests: wire format, module surface / state_dict layout, C-ABI symbol table and
argument validation (no GPU compute is attempted here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import vptq_oracle as vo
from _util import golden_names, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------- wire format (vptq_b200.pack)
@pytest.mark.parametrize("name", golden_names())
def test_pack_matches_reference_fixture(name):
    from vptq_b200.pack import pack_index, unpack_index_tensor
    L, x, ref = load_golden(name)
    idx = torch.from_numpy(L.meta["idx"].astype(np.uint16))
    ridx = torch.from_numpy(L.meta["ridx"].astype(np.uint16)) if L.meta["ridx"] is not None else None
    packed = pack_index(idx, L.index_bits, ridx, L.res_bits)
    assert packed.dtype == torch.int32
    assert np.array_equal(packed.numpy(), ref["packed_ref"])
    i2, r2 = unpack_index_tensor(packed, L.index_bits, L.group_size, L.res_bits, L.group_size if L.res_bits else 0)
    assert np.array_equal(i2.numpy().astype(np.uint16), ref["u_idx"])
    if L.res_bits:
        assert np.array_equal(r2.numpy().astype(np.uint16), ref["u_ridx"])
    else:
        assert r2 is None


def test_pack_int16_views_and_all_widths():
    from vptq_b200.pack import pack_index, unpack_index_tensor
    g = torch.Generator().manual_seed(0)
    for ib, rb in ((16, 16), (16, 8), (13, 0), (4, 2), (12, 12), (15, 3), (1, 0)):
        n = 41
        idx = torch.randint(0, 1 << ib, (2, 3, n), generator=g)
        ridx = torch.randint(0, 1 << rb, (2, 3, n), generator=g) if rb else None
        as_i16 = lambda t: t.to(torch.uint16).view(torch.int16)       # checkpoint storage view
        p = pack_index(as_i16(idx), ib, as_i16(ridx) if rb else None, rb)
        assert np.array_equal(p.numpy(), vo.pack_index(idx.numpy(), ib, None if ridx is None else ridx.numpy(), rb))
        i2, r2 = unpack_index_tensor(p, ib, n, rb, n if rb else 0)
        assert torch.equal(i2, idx)
        if rb:
            assert torch.equal(r2, ridx)
    with pytest.raises(ValueError):
        pack_index(torch.zeros(1, 1, 4, dtype=torch.int16), 20, torch.zeros(1, 1, 4, dtype=torch.int16), 16)


# ---------------------------------------------------------------- module surface
HF_KW = dict(vector_lens=[-1, 8], num_centroids=[-1, 65536], num_res_centroids=[-1, 256], group_num=1,
             group_size=4096, outlier_size=0, indices_as_float=False, enable_norm=True, enable_perm=True,
             is_indice_packed=True, enable_proxy_error=False)


def test_vquantlinear_meta_construct_and_state_dict_layout():
    """Names / shapes / dtypes of the Llama-3 v8-k65536-256 checkpoints (vqlinear.py:89-240)."""
    from vptq import VQuantLinear       # the alias HF imports
    with torch.device("meta"):
        m = VQuantLinear(4096, 14336, bias=False, **HF_KW)
    sd = {k: (tuple(v.shape), v.dtype) for k, v in m.state_dict().items()}
    assert sd == {
        "perm": ((4096,), torch.int16),
        "weight_scale": ((4096,), torch.float32),
        "weight_bias": ((4096,), torch.float32),
        "indices": ((1, 1792, 3072), torch.int32),
        "centroids.weight": ((1, 65536 * 8), torch.float32),
        "res_centroids.weight": ((1, 256 * 8), torch.float32),
    }
    assert (m.padding, m.num_indices, m.total_index_bits) == (0, 1792, 24)
    assert not m.enable_outlier and m.enable_residual


def test_vquantlinear_outlier_unpacked_layout():
    from vptq_b200 import VQuantLinear
    m = VQuantLinear(272, 100, vector_lens=[4, 6], num_centroids=[64, 1024], num_res_centroids=[-1, 16],
                     group_num=2, group_size=128, outlier_size=16, indices_as_float=True, enable_norm=False,
                     enable_perm=True, is_indice_packed=False, bias=True, dtype=torch.float16)
    sd = {k: (tuple(v.shape), v.dtype) for k, v in m.state_dict().items()}
    assert sd["indices"] == ((2, 17, 128), torch.int16)
    assert sd["res_indices"] == ((2, 17, 128), torch.float16)
    assert sd["outlier_indices"] == ((1, 25, 16), torch.float16)
    assert sd["outlier_centroids.weight"] == ((1, 256), torch.float16)
    assert sd["perm"] == ((272,), torch.int64)
    assert sd["bias"] == ((100,), torch.float16)
    assert (m.padding, m.outlier_padding) == (2, 0)
    with pytest.raises(RuntimeError):
        VQuantLinear(8, 8, [-1, 8], [-1, 4], [-1, -1], 1, 8, 0, False, vector_quant_dim="in")
    with pytest.raises(ValueError):
        VQuantLinear(8, 8, [-1, 8], [-1, 4], [-1, -1], 1, 8, 0, False, vector_quant_dim="diag")


def test_hf_integration_swaps_in_our_module():
    """transformers.integrations.vptq.replace_with_vptq_linear builds OUR VQuantLinear unchanged."""
    tv = pytest.importorskip("transformers.integrations.vptq")
    import torch.nn as nn
    from types import SimpleNamespace
    import vptq_b200

    class Net(nn.Module):          # flat on purpose: this transformers version indexes model._modules[name]
        def __init__(self):
            super().__init__()
            self.q_proj = nn.Linear(256, 256, bias=False)
            self.o_proj = nn.Linear(256, 128, bias=True)
            self.lm_head = nn.Linear(128, 10)

    layer = dict(vector_lens=[-1, 8], num_centroids=[-1, 256], num_res_centroids=[-1, 16], group_num=1,
                 group_size=256, outlier_size=0, indices_as_float=False, enable_norm=True, enable_perm=True)
    cfg = SimpleNamespace(shared_layer_config={}, config_for_layers={"q_proj": layer, "o_proj": layer})
    net = Net()
    try:
        tv.replace_with_vptq_linear(net, modules_to_not_convert=["lm_head"], quantization_config=cfg)
    except Exception as e:    # transformers internals differ between versions; the import path is what matters
        pytest.skip(f"installed transformers integration not callable standalone: {e!r}")
    assert isinstance(net.q_proj, vptq_b200.VQuantLinear) and isinstance(net.o_proj, vptq_b200.VQuantLinear)
    assert isinstance(net.lm_head, nn.Linear)
    assert net.o_proj.bias is not None and net.q_proj.indices.dtype == torch.int32
    assert net.q_proj.indices.is_meta and not net.q_proj.enable_proxy_error


def test_no_cpu_fallback():
    from vptq_b200 import VQuantLinear
    m = VQuantLinear(64, 16, [-1, 8], [-1, 16], [-1, -1], 1, 64, 0, False, is_indice_packed=True,
                     dtype=torch.float16, enable_proxy_error=False)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 64, dtype=torch.float16))


# ---------------------------------------------------------------- C ABI
def _header_symbols():
    src = open(os.path.join(ROOT, "include", "vptq_b200.h")).read()
    return sorted(set(re.findall(r"VPTQ_B200_API[^;(]*?(vptq_b200_\w+)\s*\(", src)))


def test_c_abi_exports_every_declared_symbol():
    from vptq_b200 import native
    L = native.lib()
    syms = _header_symbols()
    assert len(syms) == 15 and sorted(native.EXPORTS) == syms
    for s in syms:
        assert hasattr(L, s), s
    assert L.vptq_b200_abi_version() == native.ABI_VERSION


def test_c_abi_struct_layout_matches_header():
    from vptq_b200 import native
    # 2 + 10 int32 (48 B), 17 pointer/int64 slots, then lists_tile_cols + one reserved int32
    assert ctypes.sizeof(native.LinearDesc) == 48 + 17 * 8 + 8
    assert native.LinearDesc.indices.offset == 48
    assert native.LinearDesc.lists_tab.offset == 48 + 16 * 8 and native.LinearDesc.lists_tile_cols.offset == 48 + 17 * 8


def _desc(**over):
    from vptq_b200 import native
    d = native.LinearDesc()
    d.struct_size = ctypes.sizeof(native.LinearDesc)
    base = dict(dtype=0, in_features=4096, out_features=4096, vector_len=8, num_centroids=65536,
                num_res_centroids=256, num_codebooks=1, group_size=4096, outlier_size=0, outlier_vector_len=-1,
                num_outlier_centroids=-1, indices=0x10000, index_stride_codebook=512 * 3072, index_stride_row=3072,
                centroids=0x20000, centroid_stride=65536 * 8, res_centroids=0x30000, res_centroid_stride=2048)
    base.update(over)
    for k, v in base.items():
        setattr(d, k, v)
    return d


def test_c_abi_validation_and_workspace_without_gpu():
    from vptq_b200 import native
    L = native.lib()
    ws = L.vptq_b200_workspace_bytes(ctypes.byref(_desc()), 1, native.OP_GEMV)
    # fixed zero-at-rest head (256 KiB of counters + 4 MiB of 64-bit accumulators); this layer reduces its
    # column chunks through a thread-block cluster, so no global partial-sum scratch behind it (B200
    # geometry assumed without a GPU)
    ZERO = 65536 * 4 + 65536 * 64
    assert ws == ZERO
    # with slice x tile lists the combos meet in the 64-bit fixed-point accumulators of that head
    with_lists = _desc(lists_stream=0x40000, lists_tab=0x50000, lists_tile_cols=4096)
    assert L.vptq_b200_workspace_bytes(ctypes.byref(with_lists), 1, native.OP_GEMV) == ZERO
    # 16 codebook groups -> more than 8 chunks -> global-memory split-K scratch behind the counters
    many = _desc(num_codebooks=16, group_size=256, index_stride_row=192, index_stride_codebook=512 * 192)
    assert L.vptq_b200_workspace_bytes(ctypes.byref(many), 1, native.OP_GEMV) == ZERO + 16 * 4096 * 4
    for bad, msg in ((dict(vector_len=7), "vector_len"), (dict(num_centroids=1000), "power of two"),
                     (dict(group_size=4000), "in_features"), (dict(index_stride_row=100), "index_stride_row"),
                     (dict(res_centroids=0), "res_centroids"), (dict(dtype=3), "dtype"),
                     (dict(struct_size=8), "ABI"), (dict(in_features=70000, group_size=70000), "65535")):
        assert L.vptq_b200_workspace_bytes(ctypes.byref(_desc(**bad)), 1, native.OP_GEMV) == 0
        assert msg in native.last_error(), (bad, native.last_error())
    if not torch.cuda.is_available():
        rc = L.vptq_b200_quant_gemv(ctypes.byref(_desc()), 0x1000, 4096, 0x2000, 4096, 1, None, 0, 0, None)
        assert rc < 0 and native.last_error()


# ---------------------------------------------------------------- checkpoint compatibility
def _manifest():
    import json
    return json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_manifest.json")))


@pytest.mark.parametrize("cfg", sorted(_manifest()))
def test_state_dict_matches_reference_module_and_round_trips_through_safetensors(cfg, tmp_path):
    """Key names, shapes and storage dtypes of the REFERENCE module's state_dict (manifest generated from
    /root/reference/vptq/layers/vqlinear.py by oracle/make_state_manifest.py), and a safetensors save / load of ours
    (the format the public checkpoints ship in; uint16 payloads travel behind int16 views)."""
    from safetensors.torch import load_file, save_file
    from vptq_b200 import VQuantLinear
    ent = _manifest()[cfg]
    m = VQuantLinear(**ent["kwargs"], dtype=torch.float16, device="cpu", enable_proxy_error=False)
    ours = {k: [list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()}
    assert ours == ent["state"]
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for p in m.state_dict().values():
            if p.dtype.is_floating_point:
                p.copy_(torch.randn(p.shape, generator=g).to(p.dtype))
            else:
                info = torch.iinfo(p.dtype)
                p.copy_(torch.randint(info.min, info.max, p.shape, generator=g, dtype=torch.int64).to(p.dtype))
    path = str(tmp_path / "layer.safetensors")
    save_file({k: v.contiguous() for k, v in m.state_dict().items()}, path)
    m2 = VQuantLinear(**ent["kwargs"], dtype=torch.float16, device="cpu", enable_proxy_error=False)
    res = m2.load_state_dict(load_file(path), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert a.dtype == b.dtype and torch.equal(a, b), k
    if ent["kwargs"]["enable_perm"] and ent["kwargs"]["is_indice_packed"]:
        assert m2.perm.dtype == torch.int16          # uint16 feature indices behind an int16 view


def test_reference_python_binds_our_library_through_the_stub():
    """INTEGRATION.md option B: with integration/libvptq.py standing where the reference's pybind module
    `vptq.libvptq` would be, the REFERENCE's vptq/ops/quant_gemm.py takes its CUDA branch and reaches libvptq_b200.so.
    The calls it makes there (1 token: quant_gemv, 4 tokens: dequant) are recorded from the reference in
    tests/golden/ref_stub_calls.json (oracle/make_stub_calls.py); replayed against the stub with CPU tensors, each is
    refused by OUR argument check, not silently computed by a torch fallback."""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("_libvptq_stub", os.path.join(ROOT, "integration", "libvptq.py"))
    stub = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(stub)
    calls = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_stub_calls.json")))
    assert [c["fn"] for c in calls] == ["quant_gemv", "dequant"]
    arg = lambda a: torch.zeros(a["shape"], dtype=getattr(torch, a["dtype"])) if isinstance(a, dict) else a
    for c in calls:
        with pytest.raises(RuntimeError, match="CUDA tensor"):
            getattr(stub, c["fn"])(*[arg(a) for a in c["args"]])
