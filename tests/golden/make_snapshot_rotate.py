"""Generate tests/golden/snapshot_rotate.npz: a REGRESSION SNAPSHOT of this project's rotate_fc2, rotate_ada_lin and
block_diag (fpqvar_b200.rotation_utils) on a small layer (ffn.fc2 = Linear(64, 16), ada_lin = SiLU + Linear(16, 96)).

    python tests/golden/make_snapshot_rotate.py

The stored values are this project's own output, not the reference's: the reference's rotate_utils/rotation_utils.py
was not available when the snapshot was written, so it pins the current behaviour only.  The fixture holds the layer's
state before and after and the two rotation matrices, so the test needs no random number generator.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


class Layer(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.ffn = torch.nn.Module()
        self.ffn.fc2 = torch.nn.Linear(64, 16)
        self.ada_lin = torch.nn.Sequential(torch.nn.SiLU(), torch.nn.Linear(16, 96))


def main():
    from fpqvar_b200 import rotation_utils as R
    torch.manual_seed(0)
    layer = Layer()
    out = {f"in/{k}": v.numpy().copy() for k, v in layer.state_dict().items()}
    q64, q16 = R.get_orthogonal_matrix(64, "hadamard", "cpu"), R.get_orthogonal_matrix(16, "hadamard", "cpu")
    R.rotate_fc2(layer, q64)
    R.rotate_ada_lin(layer, q16)
    out.update({f"out/{k}": v.numpy() for k, v in layer.state_dict().items()})
    out.update({"Q64": q64.numpy(), "Q16": q16.numpy(), "block_diag": R.block_diag([q16, q16]).numpy()})
    path = os.path.join(HERE, "snapshot_rotate.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
