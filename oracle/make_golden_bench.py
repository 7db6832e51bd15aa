"""TEST INFRASTRUCTURE ONLY -- tests/golden/bench_gradients.npz: the frames the UNMODIFIED reference script
scripts/gradients.py (gradients.im_function, :117-140) draws for bench.py's config-2 clip (346x260, 30 fps).

    python oracle/make_golden_bench.py        # needs the reference tree (oracle/ref_shim.py)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
H, W, N, FPS = 260, 346, 8, 30.0


def main():
    ref_shim.load_reference()
    sys.path.insert(0, os.path.join(ref_shim.REFERENCE_ROOT, "scripts"))
    import gradients as g
    m = g.gradients.__new__(g.gradients)          # im_function only needs these attributes (gradients.py:117-140)
    m.bg, m.contrast, m.bump_width, m.w, m.h, m.speed_pps = 127, 2.0, 0.5, W, H, 300.0
    frames = np.stack([m.im_function(np.arange(H)[:, None], np.arange(W)[None, :], k / FPS) for k in range(N)])
    np.savez_compressed(os.path.join(OUT, "bench_gradients.npz"), frames=frames, fps=np.array(FPS))
    print("bench_gradients.npz written")


if __name__ == "__main__":
    main()
