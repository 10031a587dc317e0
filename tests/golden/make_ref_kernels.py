#!/usr/bin/env python3
"""Generate tests/golden/ref_kernels/*.npz = outputs of the REFERENCE's own CUDA kernels (oracle/_ref, rebuilt for
sm_100a by oracle/build_ref.py) on the seeded inputs of test_gpu_parity.py's comparisons against them
(format: tests/ref_golden.py).  Needs a GPU and oracle/_ref:

    python tests/golden/make_ref_kernels.py [OUT_DIR]      # default: tests/golden/ref_kernels
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import ref_golden as rg  # noqa: E402
from oracle import ref as oref  # noqa: E402


def main(out_dir):
    corr = oref.load_extension("correlation_cuda")
    rs = oref.load_extension("resample2d_cuda")
    cn = oref.load_extension("channelnorm_cuda")
    assert corr and rs and cn, "oracle/_ref is not built"
    for shape in ((1, 256, 48, 64), (2, 20, 13, 36)):
        a, b = rg.correlation_inputs(shape)
        ad, bd = a.cuda(), b.cuda()
        out = ad.new_empty(0)
        corr.forward(ad, bd, ad.new_empty(0), ad.new_empty(0), out, 20, 1, 20, 1, 2, 1)
        go = rg.correlation_grad_output(tuple(out.shape))
        g1, g2 = ad.new_empty(0), ad.new_empty(0)
        corr.backward(ad, bd, ad.new_empty(0), ad.new_empty(0), go.cuda(), g1, g2, 20, 1, 20, 1, 2, 1)
        print(rg.save(rg.case_name("correlation", shape), dict(input1=a, input2=b, grad_output=go),
                      dict(output=out, grad_input1=g1, grad_input2=g2), out_dir))

    img, flow, go, x, gon = (t.cuda() for t in rg.resample_channelnorm_inputs())
    rout = torch.zeros_like(img)
    rs.forward(img, flow, rout, 1, True)
    rg1, rg2 = torch.zeros_like(img), torch.zeros_like(flow)
    rs.backward(img, flow, go, rg1, rg2, 1, True)
    ro = torch.zeros(2, 1, 32, 48, device="cuda")
    cn.forward(x, ro, 2)
    rgi = torch.zeros_like(x)
    cn.backward(x, ro, gon, rgi, 2)
    print(rg.save("resample2d_channelnorm", dict(img=img, flow=flow, grad_output=go, x=x, grad_norm=gon),
                  dict(resample2d_output=rout, resample2d_grad_input1=rg1, resample2d_grad_input2=rg2,
                       channelnorm_output=ro, channelnorm_grad_input1=rgi), out_dir))

    for shape in ((2, 3, 16, 24), (1, 2, 7, 9), (2, 3, 64, 128)):
        x, go = rg.channelnorm_half_inputs(shape)
        xd, god = x.cuda(), go.cuda()
        ro = torch.zeros(go.shape, device="cuda", dtype=torch.float16)
        cn.forward(xd, ro, 2)
        rgi = torch.zeros_like(xd)
        cn.backward(xd, ro, god, rgi, 2)
        print(rg.save(rg.case_name("channelnorm_half", shape), dict(input1=x, grad_output=go),
                      dict(output=ro, grad_input1=rgi), out_dir))
    torch.cuda.synchronize()


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else rg.DIR)
