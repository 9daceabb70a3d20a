#!/usr/bin/env python
"""Write the stored records of the full-size parity cases, tests/golden/records/<config>.npz, on a GPU:

    python tests/make_records.py [OUT_DIR] [CONFIG ...]        (defaults: tests/golden/records, c2 c3 c4 c5)

Config 2 to 5 are too large for full golden vectors, so tests/test_gpu_parity.py checks them against these records
(parity.make_record / parity.check_record).  A record holds two things:
  * digests of the arrays that must be bit-identical to the reference build (indices, colour, depth, final_T), taken
    from this project's CUDA path, whose last GPU test run before the records were added (profiles/r02_pytest_gpu.txt:
    all 69 GPU tests passed, none skipped, so with reference builds present) asserted exactly these arrays
    bit-identical to the unmodified reference build (oracle/_ref) at each of these configs;
  * the bars for every float array (feature map, gradients, images): block and channel sums of the CPU oracle's result,
    i.e. of the reference algorithm restated in oracle/f3dgs_oracle.c and pinned against reference-built golden vectors
    (tests/test_oracle_golden.py), independent of the code under test.
Before writing, the script requires the two sources to agree: the oracle's radii, point_list, ranges and num_rendered
bit for bit, its n_contrib up to compare()'s threshold ties, and the CUDA result within the record's bars.
Inputs are not stored: scenegen regenerates them bit-identically from (config, views=1) and the fixed upstream
gradients of scenegen.upstream_grads().  TEST INFRASTRUCTURE ONLY.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, os.path.join(ROOT, "feature-3dgs_b200"), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import parity  # noqa: E402
import scenegen  # noqa: E402

CASES = {"c2": True, "c3": True, "c4": True, "c5": False}  # config -> with gradients (config 5 is forward-only)


def main(out_dir, names):
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name in names:
        sc = scenegen.make_config(name, views=1)
        cam = sc.cameras[0]
        grads = scenegen.upstream_grads(cam.image_height, cam.image_width, sc.C) if CASES[name] else None
        ours = parity.run_ours(sc, cam, grads=grads)
        orc = parity.run_oracle(sc, cam, grads=grads, threads=os.cpu_count())
        for k in ("radii", "point_list", "ranges", "num_rendered"):
            assert np.array_equal(np.asarray(ours[k]), np.asarray(orc[k])), (name, k)
        ties = int(np.sum(ours["n_contrib"] != orc["n_contrib"]))
        assert ties <= max(2, int(1e-4 * ours["n_contrib"].size)), (name, "n_contrib", ties)
        rec = parity.make_record(ours, orc)
        rec.update(config=np.asarray(name), gpu=np.asarray(torch.cuda.get_device_name(0)),
                   torch=np.asarray(torch.__version__), n_contrib_ties=np.int64(ties))
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **rec)
        bad = parity.check_record(ours, np.load(path))
        assert not bad, (name, bad)
        print("wrote", path, os.path.getsize(path), "bytes;", ties, "threshold ties in n_contrib", flush=True)


if __name__ == "__main__":
    argv = sys.argv[1:]
    out = argv.pop(0) if argv and argv[0] not in CASES else os.path.join(HERE, "golden", "records")
    main(out, argv or list(CASES))
