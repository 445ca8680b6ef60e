"""Worker of tests/test_gpu_tc_backward.py::test_attn_bwd_img_launch_variants.  The attention-backward launch settings
(LSTUR_ATTN_NBUF, LSTUR_ATTN_CTAS_PER_SM) are read once per process, so a variant runs in a process of its own: this
script runs the real forward over a compacted title list and lstur_attn_pool_bwd_img (dropout 0.2, img_scale 2^10),
writes the kernel's inputs and outputs to the .npz named by argv[1] and exits; the test checks them against the float64
reference.  Usage: tc_backward_worker.py OUT.npz N L F FP16"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, 'tests'))
from mnexp_b200 import _lib                 # noqa: E402
import test_gpu_tc_backward as tb           # noqa: E402


def main():
    out, N, L, F, fp16 = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5])
    lib = _lib.load()
    st = tb.encoder_state(lib, N, L, 64, F, fp16, p=0.2, case_seed=N + L + F)
    dp = tb.make_d_pooled(st, F + 24)
    o = tb.run_attn(lib, st, dp, 2.0 ** 10)
    np_ = lambda t: t.cpu().numpy()
    np.savez(out, grid=lib.lstur_attn_bwd_grid(N), p=st.p, nl=st.nl, idx=np_(st.idx), aw=np_(st.aw),
             c16=np_(st.c16.view(torch.int16)), a=np_(st.a), w=np_(st.w), dp=np_(dp), img=np_(o.img),
             d_att_w=np_(o.d_att_w), d_conv_b=np_(o.d_conv_b), d_att_b=np_(o.d_att_b), scale=o.scale)


if __name__ == '__main__':
    main()
