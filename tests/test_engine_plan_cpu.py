"""CPU: the weight-pack job list of each network (which parameters are packed, in which modes, with which operand dims)
against tests/golden/pack_plans.json.

The golden file was written with:

    import json
    import rbunet

    models = {"RobustUNet(3,1,64)": rbunet.RobustUNet(3, 1, 64), "RobustUNet(4,3,16)": rbunet.RobustUNet(4, 3, 16),
              "UNet(3,2)": rbunet.UNet(3, 2), "UNet(3,5)": rbunet.UNet(3, 5)}
    plans = {}
    for key, m in models.items():
        names = {id(p): n for n, p in m.named_parameters()}
        plans[key] = [[names[id(src)], mode, list(shape), Nn, T, K, cout, src2 is not None]
                      for (_, src, src2, shape, Nn, T, K, mode, cout) in m.engine._pack_plan()]
    with open("tests/golden/pack_plans.json", "w") as f:
        f.write("{\\n" + ",\\n".join(f" {json.dumps(k)}: [\\n" + ",\\n".join(f"  {json.dumps(j)}" for j in v) + "\\n ]"
                                    for k, v in plans.items()) + "\\n}\\n")
"""
import json
import os

import pytest

MODELS = {"RobustUNet(3,1,64)": ("RobustUNet", (3, 1, 64)), "RobustUNet(4,3,16)": ("RobustUNet", (4, 3, 16)),
          "UNet(3,2)": ("UNet", (3, 2)), "UNet(3,5)": ("UNet", (3, 5))}


@pytest.mark.parametrize("key", list(MODELS))
def test_pack_plan_matches_golden(golden_dir, key):
    import rbunet
    with open(os.path.join(golden_dir, "pack_plans.json")) as f:
        want = json.load(f)[key]
    cls, args = MODELS[key]
    m = getattr(rbunet, cls)(*args)
    names = {id(p): n for n, p in m.named_parameters()}
    got = []
    for (pkey, src, src2, shape, Nn, T, K, mode, cout) in m.engine._pack_plan():
        assert pkey == (id(src), mode)
        got.append([names[id(src)], mode, list(shape), Nn, T, K, cout, src2 is not None])
    assert got == want
