"""GPU parity of the tcgen05 depthwise kernel on shapes that stress its border-class bias table and its item walk, compared
byte for byte with the C oracle (including the canary bytes between output pixels).

Wide channel counts (14x14x576, 7x7x960, and C = 1040, whose weight blocks exceed what stays resident) are walked by 1 or 3
CTAs, so that one CTA's run of items crosses many channel blocks and spatial tiles; C = 144 / 176 leave the last channel pair
half empty; images of 1 and 2 rows or columns, and paddings of 0 and 2, produce border classes that a 3x3 window with padding
1 on a larger image never does.  Every shape runs with the compact shared-memory table where it fits and with the global
table (QNNP_CUDA_DW_BIAS_GLOBAL=1)."""
import pytest

from tests import cases as CS, util as U

pytestmark = pytest.mark.gpu

DW_EDGE_CASES = [
    (CS.conv_case("dw_c576_14_b3", 3, 14, 14, 576, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("dw_c576_s2_14_b3", 3, 14, 14, 576, 1, 1, stride=(2, 2), **CS.DW_TC), {}),
    (CS.conv_case("dw_c960_7_b4", 4, 7, 7, 960, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("dw_c1040_6_b2_16ch", 2, 6, 6, 1040, 1, 1, **CS.DW_TC), dict(QNNP_CUDA_DW_NO_PAIR="1")),
    (CS.conv_case("dw_c144_20_b2", 2, 20, 20, 144, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("dw_c176_18_b2", 2, 18, 18, 176, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("dw_c176_s2_20_b2", 2, 20, 20, 176, 1, 1, stride=(2, 2), **CS.DW_TC), {}),
    (CS.conv_case("tiny_c64_1x1_b3", 3, 1, 1, 64, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("tiny_c64_2x2_b3", 3, 2, 2, 64, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("tiny_c32_1x9_b2", 2, 1, 9, 32, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("tiny_c32_9x2_b2", 2, 9, 2, 32, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("tiny_c48_s2_2x2_b3", 3, 2, 2, 48, 1, 1, stride=(2, 2), **CS.DW_TC), {}),
    (CS.conv_case("tiny_c576_2x2_b5", 5, 2, 2, 576, 1, 1, **CS.DW_TC), {}),
    (CS.conv_case("dw_c48_11x13_pad2x1_b2", 2, 11, 13, 48, 1, 1, ks=(3, 3), pad=(2, 1, 2, 1)), {}),
    (CS.conv_case("dw_c32_s2_5x6_pad2_b3", 3, 5, 6, 32, 1, 1, ks=(3, 3), stride=(2, 2), pad=(2, 2, 2, 2)), {}),
    (CS.conv_case("dw_c64_9x12_nopad_b2", 2, 9, 12, 64, 1, 1, ks=(3, 3)), {}),
]


@pytest.mark.timeout(120, method="thread")   # a wedged kernel must fail the test, not hang the box
@pytest.mark.parametrize("table", ["smem", "global"])
@pytest.mark.parametrize("ctas", [0, 1, 3])
@pytest.mark.parametrize("case,env", DW_EDGE_CASES, ids=lambda v: v.get("name") or "+".join(v) or "router")
def test_q8dwconv_border_classes(gpu_lib, oracle_c, case, env, ctas, table, monkeypatch):
    monkeypatch.setenv("QNNP_CUDA_DW_UMMA", "1")
    if table == "global":
        monkeypatch.setenv("QNNP_CUDA_DW_BIAS_GLOBAL", "1")
    if ctas:
        monkeypatch.setenv("QNNP_CUDA_MAX_CTAS", str(ctas))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    x, k, b, kw = U.conv_setup(case)
    before = gpu_lib.dw_umma_launch_count()
    got = U.run_conv(gpu_lib, case, x, k, b, kw)
    assert gpu_lib.dw_umma_launch_count() == before + 1, "expected the tcgen05 depthwise kernel"
    U.assert_same_bytes(got, U.run_conv(oracle_c, case, x, k, b, kw), case["name"])
