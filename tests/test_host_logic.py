"""CPU tests of the host-side logic above the C ABI: the torch restatement of the loader's unpack code in
rtp_llm_b200/device.py is bit-exact against the golden vectors produced by the reference's own code, and the
strategy / impl classes expose the reference's method surface."""
import inspect
import os

import numpy as np
import pytest
import torch

from rtp_llm_b200 import attention, device, linear


@pytest.mark.parametrize("fmt", ["gptq", "awq"])
def test_unpack_groupwise_torch_matches_reference(golden_dir, fmt):
    g = np.load(os.path.join(golden_dir, f"quant_unpack_{fmt}.npz"))
    impl = device.B200Impl(device="cpu")
    qp, zs, sc = impl.unpack_groupwise(torch.from_numpy(g["qweight"]), torch.from_numpy(g["qzeros"]),
                                       torch.from_numpy(g["scales"]), gptq=fmt == "gptq", awq=fmt == "awq")
    assert np.array_equal(qp.numpy(), g["q_packed"])
    assert np.array_equal(zs.numpy().view(np.uint16), g["zeros_x_scales"].view(np.uint16))
    assert np.array_equal(sc.numpy().view(np.uint16), g["scales_out"].view(np.uint16))


@pytest.mark.parametrize("fmt", ["gptq", "awq"])
def test_unpack_groupwise_8bit_torch_matches_reference(golden_dir, fmt):
    g = np.load(os.path.join(golden_dir, f"quant_unpack8_{fmt}.npz"))
    impl = device.B200Impl(device="cpu")
    q, zs, sc = impl.unpack_groupwise(torch.from_numpy(g["qweight"]), torch.from_numpy(g["qzeros"]),
                                      torch.from_numpy(g["scales"]), gptq=fmt == "gptq", awq=fmt == "awq", weight_bits=8)
    assert q.dtype == torch.int8 and np.array_equal(q.numpy(), g["q"])
    assert np.array_equal(zs.numpy().view(np.uint16), g["zeros_x_scales"].view(np.uint16))
    assert np.array_equal(sc.numpy().view(np.uint16), g["scales_out"].view(np.uint16))


def test_int8_quantiser_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "quant_int8.npz"))
    q, s = device.B200Impl(device="cpu").symmetric_quantize_last_axis_of_batched_matrix(torch.from_numpy(g["weight"]))
    assert np.array_equal(q.numpy(), g["q"])
    assert np.array_equal(s.numpy(), g["scale"])


def test_interfaces_have_the_reference_surface():
    # XQAAttnOp method set (XQAAttnOp.cc:158-176)
    for m in ("support", "prepare", "update", "update_kv_cache_offset", "forward"):
        assert callable(getattr(attention.B200DecodeAttnOp, m))
    # FMHAImplBase strategy (fmha_impl_base.py:99-175)
    sig = inspect.signature(attention.B200DecodeImpl.forward)
    assert list(sig.parameters)[1:] == ["qkv", "kv_cache", "layer_idx"]
    assert callable(attention.B200DecodeImpl.prepare_cuda_graph) and callable(attention.B200DecodeImpl.support)
    assert list(inspect.signature(attention.B200DecodeImpl.__init__).parameters)[1:] == \
        ["attn_configs", "attn_inputs", "parallelism_config"]
    # LinearBase strategy (linear_base.py:25-49)
    assert list(inspect.signature(linear.B200WeightOnlyLinear.can_handle).parameters) == \
        ["quant_config", "weight", "weight_scales", "hw_kernel_config", "weight_scale_2", "input_scale"]
    assert list(inspect.signature(linear.B200WeightOnlyLinear.__init__).parameters)[1:] == \
        ["weight", "weight_scales", "input_scales", "bias", "quant_config", "weight_scale_2"]
    # DeviceBase hooks (device_base.py:56-90)
    for m in ("apply_int8", "preprocess_groupwise_weight_params", "preprocess_weights_for_mixed_gemm"):
        assert callable(getattr(device.B200Impl, m))


def test_strategy_selection_rules():
    class Q:  # stands in for config/quant_config.py objects
        def __init__(self, m):
            self._m = m

        def get_method(self):
            return self._m
    L = linear.B200WeightOnlyLinear
    w8 = torch.zeros(4, 4, dtype=torch.int8)
    assert L.can_handle(Q("awq"), w8, torch.ones(1, 4))
    assert L.can_handle(Q("GPTQ"), w8, torch.ones(1, 4))
    assert L.can_handle(Q("int8"), w8, torch.ones(4))
    assert not L.can_handle(Q("fp8"), torch.zeros(4, 4, dtype=torch.float8_e4m3fn), torch.ones(4))
    assert not L.can_handle(Q("awq"), w8, torch.ones(4), weight_scale_2=torch.ones(1))
    assert L.can_handle(None, torch.zeros(4, 4, dtype=torch.float16), None)


def test_attn_op_support_gate():
    class C:
        head_num, kv_head_num, size_per_head, tokens_per_block, kernel_tokens_per_block = 32, 8, 128, 64, 64
        kv_cache_dtype = "BASE"

    class I:
        is_prefill = True
    assert attention.B200DecodeAttnOp(C()).support(I()) is False          # decode only
    C.size_per_head = 96
    I.is_prefill = False
    assert attention.B200DecodeAttnOp(C()).support(I()) is False          # head_dim 64 / 128 / 256 only
    C.size_per_head = 64
    on_sm100 = torch.cuda.is_available() and torch.cuda.get_device_capability()[0] == 10
    assert attention.B200DecodeAttnOp(C()).support(I()) is on_sm100      # a served shape: supported exactly where the kernels run


def test_bench_reference_arm_runs_on_cpu_and_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times beside ours) needs no GPU and prints one JSON line."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--model", "tiny", "--batch", "2",
                          "--ctx", "64"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "tokens/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_algorithmic_bytes_match_baseline_md():
    """SURVEY 8(d) / BASELINE.md section 3: the bytes the roofline fraction is computed from."""
    import dataclasses
    from rtp_llm_b200.decode_step import LLAMA3_8B, weight_bytes
    cfg = LLAMA3_8B
    H, qkv_n, I = cfg.hidden, (cfg.head_num + 2 * cfg.kv_head_num) * cfg.head_dim, cfg.inter
    per_layer = lambda c: (weight_bytes(c, H, qkv_n) + weight_bytes(c, cfg.head_num * cfg.head_dim, H)
                           + weight_bytes(c, H, 2 * I) + weight_bytes(c, I, H))
    assert H * qkv_n + cfg.head_num * cfg.head_dim * H + H * 2 * I + I * H == 218_103_808          # E per layer
    assert abs(per_layer(dataclasses.replace(cfg, quant="int4")) * cfg.layers - 3.708e9) < 5e6
    assert abs(per_layer(dataclasses.replace(cfg, quant="f16")) * cfg.layers - 13.959e9) < 5e6
    assert abs(per_layer(dataclasses.replace(cfg, quant="int8")) * cfg.layers - 6.982e9) < 5e6
    kv = 2 * 32 * 2048 * cfg.kv_head_num * cfg.head_dim * 2 * cfg.layers
    assert abs(kv - 8.590e9) < 5e6 and abs(2 * H * cfg.vocab - 1.051e9) < 1e6


def test_gate_up_interleave_order():
    """ops.gate_up_order: rows 2i / 2i+1 of every 128-column tile = gate / up column tile*64+i (fused SiLU*mul layout: the
    pair sits in neighbouring lanes of one warp)."""
    from rtp_llm_b200 import ops
    inter = 192
    order = ops.gate_up_order(inter)
    assert sorted(order.tolist()) == list(range(2 * inter))
    for t in range(inter // 64):
        tile = order[t * 128:(t + 1) * 128]
        assert tile[0::2].tolist() == list(range(t * 64, t * 64 + 64))
        assert tile[1::2].tolist() == list(range(inter + t * 64, inter + t * 64 + 64))
    w = torch.arange(2 * inter).repeat(3, 1)
    assert torch.equal(ops.interleave_gate_up(w, inter)[0], order)
    # packed int4 (low nibble = even column): unpack -> reorder -> repack must equal reordering the nibble matrix
    g = torch.Generator().manual_seed(0)
    packed = torch.randint(0, 256, (2, inter), generator=g, dtype=torch.uint8)
    nib = torch.stack([packed & 0xF, packed >> 4], dim=-1).reshape(2, -1)
    got = ops.interleave_gate_up(packed, inter, packed_int4=True)
    got_nib = torch.stack([got & 0xF, got >> 4], dim=-1).reshape(2, -1)
    assert torch.equal(got_nib, nib.index_select(-1, order))


def test_library_staleness_is_judged_by_content(tmp_path, monkeypatch):
    """build.py records a digest of every source the library was built from; _lib.load() compares it (ADVICE r1: an edited
    kernel must never run against an old libb200_decode.so; file times do not survive the copy to the GPU box)."""
    from rtp_llm_b200 import build as b
    d = b.source_digest()
    assert len(d) == 64 and d == b.source_digest()
    stamp = tmp_path / "lib.stamp"
    monkeypatch.setattr(b, "STAMP", str(stamp))
    assert b.stamp_matches()                      # no stamp: a library of unknown origin is used as it is
    stamp.write_text(d)
    assert b.stamp_matches()
    stamp.write_text("0" * 64)
    assert not b.stamp_matches()                  # sources changed since the build -> load() rebuilds (or fails loudly)
