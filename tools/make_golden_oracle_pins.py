#!/usr/bin/env python
"""Generate tests/golden/oracle_vs_reference.npz: outputs of the REFERENCE modules that tests/test_oracle_vs_reference.py pins
the oracle against.

    python tools/make_golden_oracle_pins.py <reference source directory (the one holding models/ and utils.py)>

The inputs come from ``inputs()`` in the test (numpy's legacy ``RandomState``, whose streams are frozen across numpy versions),
so only the reference's outputs are stored.  The generator runs on the shipped checkpoint, which is tests/golden/weights_g.npz;
the discriminator on tests/golden/weights_d.npz.  Nothing in here is used at test time.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
OUT = os.path.join(GOLDEN, "oracle_vs_reference.npz")


def main(src):
    sys.path[:0] = [src, ROOT, os.path.join(ROOT, "tests")]
    if "pesq" not in sys.modules:                  # discriminator.py imports pesq at module level; the forward never calls it
        stub = types.ModuleType("pesq")
        stub.pesq = lambda *a, **k: 0.0
        sys.modules["pesq"] = stub
    from models.generator import TSCNet
    from models.discriminator import Discriminator
    import utils as ref_utils
    from test_oracle_vs_reference import inputs

    def load(name):
        z = np.load(os.path.join(GOLDEN, name))
        return {k: torch.from_numpy(z[k]) for k in z.files}

    x = inputs()
    g = {}
    m = TSCNet(64, 201)
    m.load_state_dict(load("weights_g.npz"), strict=True)
    m.eval()
    with torch.no_grad():
        g["tscnet_real"], g["tscnet_imag"] = (t.numpy() for t in m(x["tscnet"]))
    c = ref_utils.power_compress(x["compress"])
    g["compress"] = c.numpy()
    g["uncompress"] = ref_utils.power_uncompress(c[:, 0:1], c[:, 1:2]).numpy()
    D = Discriminator(ndf=16)
    D.load_state_dict(load("weights_d.npz"), strict=True)
    D.train()
    D.layers[15].p = 0.0                           # dropout off so that the train-mode output (one power iteration) is deterministic
    with torch.no_grad():
        g["disc_train"] = D(x["disc_x"], x["disc_y"]).numpy()
    np.savez_compressed(OUT, **g)
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
