#!/usr/bin/env python
"""Record one forward of the reference's own network for tests/test_oracle.py::test_oracle_vs_reference_forward.

Imports SIGGRAPHGenerator(dist=True) unmodified from the reference tree (located by oracle/ref_shims.py), loads the
seeded synthetic state_dict of oracle/synth.py and runs `forward(L, ab, mask, 0.5)` on one 64x64 synthetic image.
Stored: the inputs, the regression output in full, the upsampled class distribution at a seeded sample of pixels
(all 529 channels; the full tensor is 8.7 MB) and the state_dict key set.  Needs the reference tree:

    python tests/golden/make_ref_forward_golden.py        -> tests/golden/ref_forward_64.npz
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_shims, synth  # noqa: E402

SEED = 1234
PIXELS = 64


def main():
    torch.set_num_threads(8)
    model = ref_shims.import_reference_model()
    net = model.SIGGRAPHGenerator(dist=True)
    net.load_state_dict(synth.torch_state_dict(SEED))
    net.eval()
    L, ab, m = synth.synthetic_batch(1, 64, seed=7, max_hints=4)
    reg, dist = net.forward(L[0], ab[0], m[0], 0.5)
    yx = np.random.RandomState(0).randint(0, 64, (2, PIXELS))
    out = {"L": L, "ab": ab, "mask": m,
           "reg": reg.detach().numpy().astype(np.float32),
           "dist_yx": yx.astype(np.int32),
           "dist_at_yx": dist.detach().numpy()[0][:, yx[0], yx[1]].astype(np.float32),
           "state_dict_keys": np.array(sorted(net.state_dict().keys()))}
    np.savez_compressed(os.path.join(HERE, "ref_forward_64.npz"), **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
