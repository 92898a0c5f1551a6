"""Golden vectors from the REFERENCE's own SuperPoint definition.

The reference ships its network as executable Python: the `SuperPointNet` class in swarm_loop/superpoint.ipynb, the very
module its TensorRT engine is exported from (cell "torch.onnx.export(model, ...)").  This script EXECUTES that class where
it lies under /root/reference (nothing is copied into the repository), loads the seeded weights the tests use
(omniswarm_b200.synth.superpoint_weights -- the trained superpoint_v1.pth is not in the tree), runs it on synthetic images
and stores inputs and outputs as tests/golden/ref_superpoint.npz.

    python tests/golden/make_ref_superpoint.py          (needs /root/reference; the committed .npz travels without it)
    python tests/golden/make_ref_superpoint.py --check  compare the committed fixture with the notebook instead of writing it

tests/test_oracle_pins.py::test_network_oracle_matches_the_references_own_module compares oracle/frontend_ref.py with the
fixture.
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from omniswarm_b200 import synth                     # noqa: E402

NOTEBOOK = "/root/reference/swarm_loop/superpoint.ipynb"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_superpoint.npz")
CASES = [(0, 64, 96), (1, 48, 80), (2, 120, 160)]        # (image seed, H, W): H, W multiples of 8 as the engine requires


def reference_module():
    """the class the reference exports to ONNX: the LAST `class SuperPointNet` cell before the torch.onnx.export cell"""
    nb = json.load(open(NOTEBOOK))
    src = None
    for c in nb["cells"]:
        s = "".join(c["source"])
        if "torch.onnx.export" in s:
            break
        if c["cell_type"] == "code" and s.lstrip().startswith("class SuperPointNet"):
            src = s
    assert src is not None, "SuperPointNet not found in the reference notebook"
    ns = {"torch": torch}
    exec(compile(src, NOTEBOOK, "exec"), ns)
    return ns["SuperPointNet"]


def run_reference(img_u8, weights, scale="mul"):
    """scale = "mul": the input convention of the reference's C++ runtime, cv::Mat::convertTo(CV_32F, 1/255.0) = (float)v *
    (float)(1/255.0) (superpoint_tensorrt.cpp:127) -- what the oracle restates;  "div": the notebook's own
    `img.astype(np.float32)/255`, one ulp away on some pixels"""
    net = reference_module()()
    net.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in weights.items()})
    net.eval()
    f = img_u8.astype(np.float32)[None, None]
    x = torch.from_numpy(f * np.float32(1.0 / 255.0) if scale == "mul" else f / 255)
    with torch.no_grad():
        semi, desc = net.forward(x, False)
    return semi[0].numpy().copy(), desc[0].numpy().copy()


def main(check=False):
    torch.set_num_threads(1)
    w = synth.superpoint_weights(0)
    out = {}
    for seed, H, W in CASES:
        img = synth.image(seed, H, W)
        semi, desc = run_reference(img, w, "mul")
        out[f"img_{seed}"] = img
        out[f"semi_{seed}"] = semi
        out[f"desc_{seed}"] = desc
        if seed == 0:                                   # the notebook's own input scaling, for the record
            out["semi_div_0"], out["desc_div_0"] = run_reference(img, w, "div")
    if check:
        z = np.load(OUT)
        assert sorted(z.files) == sorted(out) and all(np.array_equal(z[k], v) for k, v in out.items()), \
            "tests/golden/ref_superpoint.npz differs from the notebook's outputs"
        print("ref_superpoint.npz matches the notebook")
        return
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main(check="--check" in sys.argv[1:])
