"""Build tuning variants of the CUDA library into gpurun_out-independent tools/_sweep/ (travels to the GPU box)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gan-based-video-style-transfer_b200", "csrc")
OUT = os.path.join(ROOT, "tools", "_sweep")
VARIANTS = {
    "hot": {"TCL_HOT_ONLY": 1},
    "hot_w16": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16},
    "hot_w16_s1": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_SCANNERS": 1},
    "hot_w16_s3": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_SCANNERS": 3},
    "hot_s1": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 8, "TCL_SCANNERS": 1},
    "hot_s3": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 8, "TCL_SCANNERS": 3},
    "hot_w8": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 8},
    "hot_bw76": {"TCL_HOT_ONLY": 1, "TCL_BW": 76},
    "hot_w16_bw76": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_BW": 76},
    "hot_w12": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 12, "TCL_TH": 24, "TCL_BH": 32},
    "diag1_w16": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_DIAG": 1},
    "diag3_ns2_nb4": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_DIAG": 3},
    "diag3_ns2_nb2": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_DIAG": 3, "TCL_NB": 2, "TCL_BH": 36},
    "diag3_ns3_nb2": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_DIAG": 3, "TCL_NB": 2, "TCL_NS": 3, "TCL_BH": 36},
    "diag3_ns2_nb3": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_DIAG": 3, "TCL_NB": 3, "TCL_BH": 36},
    "w8_th16_ns3": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 8, "TCL_NS": 3, "TCL_NB": 5, "TCL_BH": 22, "TCL_BW": 76, "TCL_TH": 16},
    "w8_th16_ns4": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 8, "TCL_NS": 4, "TCL_NB": 6, "TCL_BH": 22, "TCL_BW": 76, "TCL_TH": 16},
    "w8_th16_ns2": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 8, "TCL_NS": 2, "TCL_NB": 4, "TCL_BH": 22, "TCL_BW": 76, "TCL_TH": 16},
    "full_w16": {"TCL_CWARPS": 16},
    "full_w8": {"TCL_CWARPS": 8},
    "hot_s1": {"TCL_HOT_ONLY": 1, "TCL_SCANNERS": 1},
    "hot_hint1000": {"TCL_HOT_ONLY": 1, "TCL_CONS_HINT_NS": 1000},
    "hot_s3x": {"TCL_HOT_ONLY": 1, "TCL_SCANNERS": 3},
    "hot_s4x": {"TCL_HOT_ONLY": 1, "TCL_SCANNERS": 4},
    "hot_bh42": {"TCL_HOT_ONLY": 1, "TCL_BH": 42},
    "hot_bh44": {"TCL_HOT_ONLY": 1, "TCL_BH": 44},
    "hot_nb3_bh44": {"TCL_HOT_ONLY": 1, "TCL_BH": 44, "TCL_NB": 3},
    "hot_nb3_bh48": {"TCL_HOT_ONLY": 1, "TCL_BH": 48, "TCL_NB": 3},
    "hot_nb3_bh49_s3": {"TCL_HOT_ONLY": 1, "TCL_BH": 49, "TCL_NB": 3, "TCL_SCANNERS": 3},
    "hot_s3_bh44": {"TCL_HOT_ONLY": 1, "TCL_SCANNERS": 3, "TCL_BH": 44},
    "hot_w16_bh42": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16, "TCL_BH": 42},
    "hot_w16": {"TCL_HOT_ONLY": 1, "TCL_CWARPS": 16},
    "hot_s3_bh42": {"TCL_HOT_ONLY": 1, "TCL_SCANNERS": 3, "TCL_BH": 42},
    "hot_bh38": {"TCL_HOT_ONLY": 1, "TCL_BH": 38},
    "hot_bh36": {"TCL_HOT_ONLY": 1, "TCL_BH": 36},
    "trace": {"TCL_TRACE": 1, "TCL_HOT_ONLY": 1},
    "bf16_bh42": {"TCL_HOT_ONLY": 2, "TCL_BH16": 42},
    "bf16_bh48": {"TCL_HOT_ONLY": 2, "TCL_BH16": 48},
    "bf16_bh54": {"TCL_HOT_ONLY": 2, "TCL_BH16": 54},
    "bf16_bh60": {"TCL_HOT_ONLY": 2, "TCL_BH16": 60},
}
# the rest of the library (host entry, cv2 flavour, aggregation) is linked in from the regular build's objects
OTHER_OBJS = [os.path.join(CSRC, o) for o in ("tcl_host.o", "tcl_cv2.o", "tcl_agg.o", "tcl_chain.o")]
if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    names = sys.argv[1:] or list(VARIANTS)
    procs = []
    for n in names:
        defs = [f"-D{k}={v}" for k, v in VARIANTS[n].items()]
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
               "-shared", "-Xptxas", "-v"] + defs + ["-o", os.path.join(OUT, f"lib_{n}.so"), os.path.join(CSRC, "tcl_kernels.cu")] + OTHER_OBJS
        procs.append((n, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for n, pr in procs:
        out = pr.communicate()[0]
        lines = out.splitlines()
        # ptxas -v report of computeTCL's kernel: fused_forward_ws_kernel<float or bf16, MASK_COMPUTED, true, 3, kVarL2, ...>
        hot = [i for i, l in enumerate(lines) if ("ws_kernelIfLi2ELb1ELi3ELi1E" in l or "ws_kernelI13__nv_bfloat16Li2ELb1ELi3ELi1E" in l) and "Compiling" in l]
        info = " | ".join(l.strip() for l in lines[hot[0] + 1:hot[0] + 4]) if hot else "?"
        print(n, "rc", pr.returncode, info[:230])
