"""Which kernel each layer of the forward runs on, per conv math mode (lib/nets/network.py: tc_format, mask_stage_code,
fp16_twins) -- the routing table of the static stage and the mask stage, pinned without a GPU."""
import pytest

from lib.nets.network import Network, _conv_tc_formats, fp16_twins, mask_stage_code, tc_format

ALL = {"tf32", "tf32x3", "f16x3", "fp16"}  # a 3-D conv with 32 or a multiple of 64 input channels, ks 1 or 3
NO_FP16 = {"tf32", "tf32x3", "f16x3"}      # cin = 96, or a 2x2x2 / stride-2 conv; also the classifier's first FC

# mode -> (conv with every format, conv without fp16 weights, k2s2 writing a fresh dense tensor (requests a twin),
#          k2s2 writing into the 128-wide level-1 slice (no twin), classifier FC, bottleneck fusion)
TABLE = {
    "exact": ("f16x3", "f16x3", "f16x3", "f16x3", "f16x3", "f16x3"),
    "f16x3": ("f16x3", "f16x3", "f16x3", "f16x3", "f16x3", "f16x3"),
    "tf32x3": ("tf32x3", "tf32x3", "tf32x3", "tf32x3", "tf32x3", "tf32x3"),
    "mixed": ("tf32", "tf32", "tf32", "tf32", "tf32", "tf32"),
    "tf32": ("tf32", "tf32", "tf32", "tf32", "tf32", "tf32"),
    "fp16": ("fp16", "tf32", None, "tf32", None, None),
    "fp32": (None, None, None, None, None, None),
}
MASK_CODE = {"exact": 2, "f16x3": 1, "tf32x3": 1, "mixed": 2, "tf32": 1, "fp16": 2, "fp32": 0}


def test_table_covers_every_mode():
    assert set(TABLE) == set(Network.MATH_MODES) == set(MASK_CODE)


@pytest.mark.parametrize("mode", sorted(TABLE))
def test_static_stage_routing(mode):
    math = Network.MATH_MODES[mode][0]
    conv_all, conv_no16, k2s2_dense, k2s2_slice, fc, fused = TABLE[mode]
    twins = fp16_twins(math)
    assert twins == (mode == "fp16")
    assert tc_format(math, ALL, "conv", True) == conv_all
    assert tc_format(math, NO_FP16, "conv", True) == conv_no16
    # k2s2 layers of the colour / geometry stacks ask for a twin; it exists only in fp16 math and for a dense output
    assert tc_format(math, NO_FP16, "conv", True, out32=True, twin=twins) == k2s2_dense
    assert tc_format(math, NO_FP16, "conv", True, out32=True, twin=False) == k2s2_slice
    assert tc_format(math, NO_FP16, "linear") == fc
    assert tc_format(math, ALL, "fused", True) == fused
    assert tc_format(math, NO_FP16, "fused", True) == fused
    for op in ("conv", "fused"):  # geometry, input layout or activation outside the tensor-core kernel; fusion switched off
        assert tc_format(math, ALL, op, False) is None
    assert tc_format(math, set(), "conv", True) is None  # C_out / C_in the tensor-core kernel does not take
    assert tc_format(math, set(), "linear") is None      # an FC with C_in < 1024


@pytest.mark.parametrize("mode", sorted(TABLE))
def test_fp16_conv_without_fp32_output_stays_on_cuda_cores(mode):
    math = Network.MATH_MODES[mode][0]
    want = "fp16" if math == "fp16" else TABLE[mode][1]
    assert tc_format(math, ALL, "conv", True, out32=False, twin=True) == want
    if math == "fp16":  # only fp16 weights run without an fp32 output; the TF32 kernel needs one and no twin
        assert tc_format(math, NO_FP16, "conv", True, out32=False, twin=True) is None
        assert tc_format(math, NO_FP16, "conv", True, out32=True, twin=True) is None


@pytest.mark.parametrize("mode", sorted(MASK_CODE))
def test_mask_stage_code(mode):
    mask_math = Network.MATH_MODES[mode][1]
    assert mask_stage_code(mask_math, ALL) == MASK_CODE[mode]
    assert mask_stage_code(mask_math, {"tf32"}) == min(MASK_CODE[mode], 1)  # no fp16 weights: the TF32 canvas
    assert mask_stage_code(mask_math, set()) == 0


def test_packed_formats():
    assert set(_conv_tc_formats(64, 64, 3)) == ALL
    assert set(_conv_tc_formats(32, 64, 1)) == ALL
    assert set(_conv_tc_formats(256, 32, 1)) == ALL  # merged RPN heads: C_in = RPN_CHANNELS, C_out padded to 32/64/128k
    assert set(_conv_tc_formats(96, 64, 3)) == NO_FP16
    assert set(_conv_tc_formats(64, 64, 2)) == NO_FP16
    assert _conv_tc_formats(2, 64, 3) == ()   # mask_backbone.geometry.0
    assert _conv_tc_formats(64, 18, 1) == ()  # C_out the tensor-core kernel does not take
