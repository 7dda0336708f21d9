"""Generate tests/golden/ref_cv2_*.npz by RUNNING THE REFERENCE'S OWN dataset-generation functions (cv2 + NumPy):

    TCL_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden_cv2.py

The generator scripts import ``imageio`` (absent here), so their def blocks -- warp_image / warp_flow / fb_check,
methods/learning-based/dataset-generation/coco-generation.py:66-113 and hollywood2-generation.py:63-111 -- are executed
from the source files where they lie under TCL_REFERENCE_ROOT (never copied).  cv2 4.13.0, numpy 2.3.
"""
import os
import sys

import cv2
import numpy as np

REF = os.environ["TCL_REFERENCE_ROOT"]
GEN = os.path.join(REF, "methods", "learning-based", "dataset-generation")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))


def defs(fname, first, last):
    src = "".join(open(os.path.join(GEN, fname)).readlines()[first - 1:last])
    ns = {"np": np, "cv2": cv2}
    exec(compile(src, fname, "exec"), ns)
    return ns


def main():
    from test_cv2_compat import flows
    coco, holly = defs("coco-generation.py", 66, 113), defs("hollywood2-generation.py", 63, 111)
    for name, (H, W, amp, seed) in {"small": (24, 40, 0.6, 11), "odd": (19, 23, 3.0, 12), "large_disp": (48, 64, 6.0, 13)}.items():
        ff, bf, img = flows(H, W, amp, seed)
        wf = coco["warp_flow"](ff, bf)
        np.savez_compressed(os.path.join(HERE, f"ref_cv2_{name}.npz"), ff=ff, bf=bf, img=img, warped_flow=wf,
                            warped_img=coco["warp_image"](img, bf), mask_occ=coco["fb_check"](wf, bf),
                            mask_both=holly["fb_check"](wf, bf))
        print(name, "keep occ-only %.3f both %.3f" % (coco["fb_check"](wf, bf).mean(), holly["fb_check"](wf, bf).mean()))


if __name__ == "__main__":
    main()
