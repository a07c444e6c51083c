"""tools/tst_probe.py -- one single-layer conv model through the CUDA path against the restatement (debug aid for the conv epilogue).
usage: python tools/tst_probe.py "dict(k=1, s=1, c=32, co=64, h=20, w=20)" """
import sys

import numpy as np

sys.path.insert(0, ".")
from __graft_entry__ import load_package
from oracle import oraclebind as ob

kw = eval(sys.argv[1])
pkg = load_package()
blob = pkg.marsfile.build_single_layer("conv", **kw).to_bytes()
gm = pkg.MarsModel(blob)
om = ob.OracleModel(blob)
rng = np.random.default_rng(2)
W = om.weights_size
fill = rng.integers(0, 256, size=om.arena_bytes - W, dtype=np.uint8)
om.arena()[W:W + fill.size] = fill
gm.mirror()[W:W + fill.size] = fill
gm.arena_upload()
om.run()
for i in range(om.num_layers):
    rc = gm.run_layer(i)
    if rc != 0:
        print("FAIL run_layer", rc, pkg.lib().mars_b200_last_error())
        sys.exit(1)
got = gm.arena_download()
want = om.arena()[: got.size]
d = np.nonzero(got != want)[0]
print(kw, "OK" if d.size == 0 else "DIFF %d bytes, first at %d (W=%d)" % (d.size, d[0], W))
