"""Precision routing of typed device passes (sdpa_precision_supported_for): a host-side rule, no GPU needed."""
import itertools


def test_bf16_operands_resolve_auto_to_the_bf16_kernel(sdpa):
    """bf16 operands are rounded already, so AUTO takes the bf16 tensor-core kernel (which reads them in place) wherever it
    takes the shape, and the fp32 kernel elsewhere."""
    ps = sdpa.precision_supported_for
    assert ps("bf16", "auto", 128, 128) == (True, "bf16")
    assert ps("bf16", "auto", 64, 256) == (True, "bf16")
    assert ps("bf16", "auto", 256, 256) == (True, "bf16")
    assert ps("bf16", "auto", 100, 36) == (True, "f32")
    assert ps("bf16", "auto", 300, 64) == (False, "f32")
    assert ps(sdpa.DTYPE_BF16, sdpa.PREC_AUTO, 80, 48) == (True, "bf16")


def test_fp32_and_fp64_operands_keep_the_fp64_rule(sdpa):
    shapes = [(128, 128), (64, 64), (80, 48), (64, 256), (128, 256), (200, 64), (100, 100), (100, 36), (1, 1), (300, 64), (8, 8)]
    for (dk, dv), prec in itertools.product(shapes, ("auto", "f32", "bf16", "bf16x3")):
        expect = sdpa.precision_supported(prec, dk, dv)
        assert sdpa.precision_supported_for("f32", prec, dk, dv) == expect, (prec, dk, dv)
        assert sdpa.precision_supported_for("f64", prec, dk, dv) == expect, (prec, dk, dv)


def test_explicit_precisions_do_not_depend_on_the_dtype(sdpa):
    for (dk, dv), prec in itertools.product([(128, 128), (64, 256), (100, 36), (136, 200)], ("f32", "bf16", "bf16x3")):
        assert sdpa.precision_supported_for("bf16", prec, dk, dv) == sdpa.precision_supported(prec, dk, dv)


def test_unknown_dtype_is_unsupported(sdpa):
    assert sdpa.lib().sdpa_precision_supported_for(3, 0, 128, 128, None) == 0
    assert sdpa.lib().sdpa_precision_supported_for(-1, 0, 128, 128, None) == 0
