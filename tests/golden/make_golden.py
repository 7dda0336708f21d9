"""Generate tests/golden/ref_cpu_*.npz by RUNNING THE REFERENCE'S OWN FUNCTIONS (imported by path,
never copied) on small seeded inputs, with TCL_REFERENCE_ROOT naming a checkout of the reference repository:

    TCL_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py

The reference hard-codes ``.cuda()`` (utils/flowtools.py:25) and ``device="cuda"``; on a CPU-only
machine the former is neutralised by patching ``torch.Tensor.cuda`` to the identity and the latter
by passing ``device="cpu"`` -- the arithmetic then runs in ATen's CPU kernels (torch 2.11.0).
The CUDA-flavour vectors (``ref_cuda_*.npz``) are produced on a B200 by tests/golden/make_golden_cuda.py with
oracle/torch_port.py, which tests/test_oracle_pinning.py proves bit-identical to these functions on CPU.
"""
import os
import sys

import numpy as np
import torch

REF = os.environ["TCL_REFERENCE_ROOT"]
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def load_reference():
    torch.Tensor.cuda = lambda self, *a, **k: self
    sys.path.insert(0, os.path.join(REF, "utils"))
    sys.path.insert(0, os.path.join(REF, "methods", "learning-based"))
    import flowtools
    import fs_lib
    return flowtools, fs_lib


def cases():
    import tcl_b200
    synth = tcl_b200.synth
    out = {}
    # (name, B, H, W, flow kwargs, frame kind)
    specs = [("smooth", 2, 24, 40, dict(max_shift=5.0, max_rot_deg=4.0, n_rects=3, rect_shift=3.0), "smooth"),
             ("white_odd", 2, 19, 23, dict(max_shift=6.0, max_rot_deg=2.0, n_rects=1, rect_shift=2.5), "white"),
             ("large_disp", 1, 32, 48, dict(max_shift=30.0, max_rot_deg=3.0, n_rects=2, rect_shift=12.0), "white")]
    for i, (name, B, H, W, kw, kind) in enumerate(specs):
        ff, bf = synth.make_flows(B, H, W, seed=100 + i, **kw)
        prev, cur = synth.make_frames(B, 3, H, W, seed=100 + i, kind=kind)
        out[name] = (ff, bf, prev, cur)
    return out


def main():
    flowtools, fs_lib = load_reference()
    for name, (ff, bf, prev, cur) in cases().items():
        with torch.no_grad():
            warped = flowtools.warp(prev, bf)
            mask = flowtools.fbcCheckTorch(ff, bf, device="cpu")
            grad_u = flowtools.gradient(bf[:, 0, :, :])
            fsw = fs_lib.warp(prev, bf)
            rmse = ((mask * (cur - warped)) ** 2).mean() ** 0.5                # utils/sintel_eval.py:110
            rmse_ps = ((mask * (cur - warped)) ** 2).mean(dim=(1, 2, 3)) ** 0.5  # utils/metrics/eval.py:138
            l2 = ((mask * (cur - warped)) ** 2).mean()                         # solver.py:444
            l1 = (mask * torch.abs(warped - cur)).mean()                       # MoGAN cycle_gan_model.py:281
        # autograd through the reference warp (what g_loss.backward() sees, solver.py:181)
        p = prev.clone().requires_grad_(True)
        f = bf.clone().requires_grad_(True)
        c = cur.clone().requires_grad_(True)
        loss = ((mask * (c - flowtools.warp(p, f))) ** 2).mean()
        loss.backward()
        np.savez_compressed(
            os.path.join(HERE, f"ref_cpu_{name}.npz"),
            ff=ff.numpy(), bf=bf.numpy(), prev=prev.numpy(), cur=cur.numpy(),
            warp=warped.numpy(), mask=mask.numpy(), grad_u=grad_u.numpy(), fs_warp=fsw.numpy(),
            rmse=rmse.numpy(), rmse_per_sample=rmse_ps.numpy(), l2=l2.numpy(), l1=l1.numpy(),
            grad_prev=p.grad.numpy(), grad_flow=f.grad.numpy(), grad_cur=c.grad.numpy(),
            torch_version=np.array(torch.__version__))
        print(name, "keep", float(mask.mean()), "rmse", float(rmse))


if __name__ == "__main__":
    main()
