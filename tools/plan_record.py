"""Record what a build computes and schedules, for comparing two builds of the library on one GPU (no output is written
to the tree; everything goes to --out).

    cd TREE && python /path/to/tools/plan_record.py --out DIR     # for each of the two trees, then compare the DIRs

  * calls.json: the recorded call lists (C function name and every argument that is not a device pointer) of the
    module-path plans (`net(x)`) and the DataParallelTrainer plans of ResNet-18, DenseNet-18 and ResNet-50 cnn_linear in
    train(), frozen BatchNorm and eval(), fp32 and bf16, at B = 2;
  * stem_bwd.pt: dards_stem_bwd's dW / dgamma / dbeta partial rows for fixed inputs, groups of 20 (fused, with and
    without the staged gradient) and 300 (chunked), max and avg pool, fp32 and bf16 gradients.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.getcwd())   # the build under comparison: run from its tree

import torch  # noqa: E402

import deepards_b200 as D  # noqa: E402
from deepards_b200 import _lib, kernels as K  # noqa: E402
from deepards_b200.data_parallel import DataParallelTrainer  # noqa: E402


def _scalars(args):
    return [a if not isinstance(a, float) else repr(a) for a in args
            if not (isinstance(a, int) and abs(a) >= 1 << 32) and (a is None or isinstance(a, (int, float)))]


def calls():
    out = {}
    for backbone in ("resnet18", "densenet18", "resnet50"):
        for state in ("train", "frozen", "eval"):
            if backbone == "densenet18" and state == "frozen":
                continue
            for precision in ("fp32", "bf16"):
                torch.manual_seed(0)
                bb = getattr(D, backbone)(**({"drop_rate": 0.0} if backbone == "densenet18" else {"initial_planes": 16}))
                net = D.CNNLinearNetwork(bb, 20, 0).cuda()
                net.precision = precision
                if state == "eval":
                    net.eval()
                elif state == "frozen":
                    for m in net.modules():
                        if isinstance(m, torch.nn.BatchNorm1d):
                            m.eval()
                x = torch.randn(2, 20, 1, 224, device="cuda")
                with torch.no_grad():
                    net(x)
                tag = "%s/%s/%s" % (backbone, state, precision)
                for key, plan in net._dards_plans.items():
                    out["module/%s/%s" % (tag, key)] = [[n] + _scalars(a) for rec in (plan.fwd, plan.bwd)
                                                        for n, _, a in rec.calls]
                if state != "eval":
                    tr = DataParallelTrainer(net)
                    plan = tr.plan_for(x)
                    out["trainer/%s" % tag] = [[n] + _scalars(a) for rec in (plan.fwd, plan.bwd) for n, _, a in rec.calls]
    return out


def stem_bwd():
    res = {}
    g = torch.Generator().manual_seed(7)
    for group, ng in ((20, 3), (300, 1)):
        n = group * ng
        x = torch.randn(n, 224, generator=g).cuda()
        w = (0.4 * torch.randn(64, 1, 7, generator=g)).cuda()
        gamma = (1 + 0.3 * torch.randn(64, generator=g)).cuda()
        beta = (0.2 * torch.randn(64, generator=g)).cuda()
        for pool in (0, 1):
            for dtype in (torch.float32, torch.bfloat16):
                _, mean, rstd = K.stem_fwd(x, w, gamma, beta, group, pool, dtype)
                dout = (0.1 * torch.randn(n, 56, 64, generator=g)).cuda().to(dtype)
                for strided in (False, True):   # strided: a row stride that rules out the staged gradient slice
                    d = dout
                    if strided:
                        d = torch.zeros(n, 56, 65, dtype=dtype, device="cuda")[..., :64]
                        d.copy_(dout)
                    gg = n // group
                    dwp = torch.empty((gg, 64 * 7), device="cuda")
                    dgp = torch.empty((gg, 64), device="cuda")
                    dbp = torch.empty((gg, 64), device="cuda")
                    nb = _lib.fn("dards_stem_workspace_bytes")(gg, group, 64, 1)
                    ws = torch.empty(((nb + 3) // 4,), device="cuda") if nb else None
                    _lib.call("dards_stem_bwd", d.data_ptr(), x.data_ptr(), w.data_ptr(), gamma.data_ptr(),
                              beta.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dwp.data_ptr(), dgp.data_ptr(),
                              dbp.data_ptr(), gg, group, 64, d.stride(1), pool, ws.data_ptr() if ws is not None else None,
                              nb, _lib.BF16 if dtype == torch.bfloat16 else _lib.F32,
                              torch.cuda.current_stream().cuda_stream)
                    res["g%d/p%d/%s/%s" % (group, pool, dtype, "strided" if strided else "dense")] = \
                        torch.cat([dwp.flatten(), dgp.flatten(), dbp.flatten()]).cpu()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    json.dump(calls(), open(os.path.join(a.out, "calls.json"), "w"))
    torch.save(stem_bwd(), os.path.join(a.out, "stem_bwd.pt"))
    print("recorded", a.out)


if __name__ == "__main__":
    main()
