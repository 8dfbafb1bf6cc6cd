"""Generates tests/golden/warp_small.npz by running the REFERENCE'S OWN classes -- src/models/ConvNet_TPS.py and
src/models/UNet.py (+ unet_parts.py) of a miccunifi/ladi-vton checkout, imported unmodified -- CPU fp32, with the seeded weights of
ladi_vton_b200.synthetic.warp_state_dict.  The reference forward calls `.cuda()` on a few constants (ConvNet_TPS.py:213-216); so that
the script runs without a GPU, `torch.Tensor.cuda` is patched to a no-op for the duration of the script:

    python tests/golden/make_golden_warp.py <ladi-vton checkout>

tests/test_oracle_pins.py imports this module for build_weights() / build_inputs(); only main() reads the checkout.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)


def build_weights():
    from ladi_vton_b200 import synthetic as S
    from ladi_vton_b200.warp import ConvNet_TPS, UNetVanilla, control_points
    tps_sd = S.warp_state_dict(ConvNet_TPS(256, 192, 21, 3).param_shapes(), 11, ctrl_bias=torch.atanh(control_points()).view(-1))
    unet_sd = S.warp_state_dict(UNetVanilla(24, 3, True).param_shapes(), 12)
    return tps_sd, unet_sd


def build_inputs():
    g = torch.Generator().manual_seed(5)
    return (torch.rand((2, 3, 256, 192), generator=g) * 2 - 1, torch.rand((2, 21, 256, 192), generator=g), torch.rand((1, 24, 32, 48), generator=g))


def main(reference):
    sys.path.insert(0, reference)
    torch.Tensor.cuda = lambda self, *a, **k: self
    from src.models.ConvNet_TPS import ConvNet_TPS as RefTPS  # reference files, unmodified
    from src.models.UNet import UNetVanilla as RefUNet
    tps_sd, unet_sd = build_weights()
    tps = RefTPS(256, 192, 21, 3).eval()
    tps.load_state_dict(tps_sd, strict=False)  # the gridGen buffers are the reference's own
    unet = RefUNet(24, 3, True).eval()
    unet.load_state_dict(unet_sd)
    a, b, x = build_inputs()
    with torch.no_grad():
        grid, pts = tps(a, b)[:2]
        y = unet(x)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "warp_small.npz"), points=pts.numpy(), grid_sub=grid[:, ::8, ::8].contiguous().numpy(),
                        unet_out=y.numpy(), inverse_kernel=tps.gridGen.inverse_kernel.numpy(),
                        repr_sub=tps.gridGen.target_coordinate_repr[::97].contiguous().numpy())
    print("wrote warp_small.npz; control points range", float(pts.abs().max()), "unet out std", float(y.std()))


if __name__ == "__main__":
    main(sys.argv[1])
