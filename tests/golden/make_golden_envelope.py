"""Regenerate tests/golden/envelope.npz: the reproducibility envelope of the reference's optimiser on fresh objects.

    python tests/golden/make_golden_envelope.py        # CPU only; writes tests/golden/envelope.npz

The scene is synthetic.make_scene(12, 20, seed=42) with the scale prior, 100 iterations.  Every object runs through
oracle/torch_oracle (the op-for-op port of the reference's optimiser, pinned bit for bit to the reference's recorded
trajectories by tests/test_oracle_golden.py) twice: once as is, and once with every projection matrix moved up by one
fp32 ulp.  The scene's inputs are stored beside the trajectories, so the test that reads them does not depend on how
synthetic.py draws a scene.  One torch thread, as for the other fixtures: torch's reductions may split across
threads, and the port's bits would then depend on the thread count.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)

N_OBJ, V, ITERS, SEED = 12, 20, 100, 42


def main():
    from odam_b200 import api, synthetic
    from oracle import c_oracle, torch_oracle
    c_oracle.build()
    torch.set_num_threads(1)
    scene = synthetic.make_scene(N_OBJ, V, seed=SEED)
    tracks = api.pack_scene(scene)
    prior = api.prior_table()
    out = {k: np.zeros((N_OBJ, ITERS, 9), np.float32) for k in ("ref_params", "ulp_params")}
    out.update({k: np.zeros((N_OBJ, ITERS), np.float32) for k in ("ref_loss", "ulp_loss")})
    for i in range(N_OBJ):
        a, b = tracks.view_off[i], tracks.view_off[i + 1]
        P32 = scene.P_cws[i].astype(np.float32)
        args = (scene.translate[i], scene.angle[i], scene.dims[i])
        kw = dict(prior33=prior[tracks.cls[i]].reshape(3, 3), n_iters=ITERS, anomaly=False)
        for tag, P in (("ref", P32), ("ulp", np.nextafter(P32, np.float32(np.inf)))):
            r = torch_oracle.run(*args, P, tracks.box[a:b], tracks.mask[a:b], **kw)
            out[f"{tag}_params"][i], out[f"{tag}_loss"][i] = r["params"], r["loss"]
        print(f"object {i}: final loss {out['ref_loss'][i, -1]:.4f} (+1 ulp: {out['ulp_loss'][i, -1]:.4f})")
    path = os.path.join(HERE, "envelope.npz")
    np.savez_compressed(path, translate=scene.translate, angle=scene.angle, dims=scene.dims, cls=scene.cls,
                        P_cws=scene.P_cws, box=scene.box, mask=scene.mask, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
