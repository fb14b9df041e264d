"""Record flash-attn's varlen attention at other head dimensions for
tests/test_attn_hd_gpu.py::test_attention_hd_vs_flash_attn, so that the comparison with the library the reference's
cgpt encoder runs on does not need flash-attn installed where the tests run.

    python tests/golden/make_golden_flash_attn_hd.py [--head-dims 32,128] [OUT_DIR]
        (on a B200 with flash-attn 2 installed; default: every case the test defines, written to tests/golden)

Writes attn_flash_varlen_hd<hd>.npz per head dimension, in the layout of attn_flash_varlen.npz
(tests/golden/make_golden_flash_attn.py): flash-attn's bf16 forward output [R, H * hd] and qkv gradient [R, 3, H, hd]
(raw bf16 bits as uint16) on R token rows -- a fixed, seeded sample plus the first and last row of every sequence -- and
strided probes of the inputs, which the test regenerates from their seed.
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import attention as OA  # noqa: E402
from test_attn_hd_gpu import FLASH_HD_CASES, FLASH_HD_PROBE, flash_attn_hd_case  # noqa: E402

N_SAMPLE = 64


def record(out_dir, hd):
    import flash_attn as fa
    starts, lens, H, qkv, dout = flash_attn_hd_case(hd)
    T = qkv.shape[0]
    slopes = torch.tensor(OA.alibi_slopes(H), dtype=torch.float32, device="cuda")
    cu = torch.tensor(np.concatenate(([0], np.cumsum(lens))), dtype=torch.int32, device="cuda")
    a = qkv.cuda().to(torch.bfloat16).requires_grad_()
    ref = fa.flash_attn_varlen_qkvpacked_func(a, cu, max(lens), 0.0, softmax_scale=1.0 / math.sqrt(hd), causal=True,
                                              alibi_slopes=slopes)
    ref.backward(dout.cuda().view(T, H, hd).to(torch.bfloat16))
    ends = [s + n - 1 for s, n in zip(starts, lens)]
    rows = np.unique(np.concatenate((np.random.RandomState(0).choice(T, N_SAMPLE, replace=False), starts, ends))).astype(np.int64)
    bits = lambda t: t.detach().cpu()[torch.from_numpy(rows)].contiguous().view(torch.int16).numpy().view(np.uint16)
    meta = dict(flash_attn=fa.__version__, torch=torch.__version__, gpu=torch.cuda.get_device_name(0))
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"attn_flash_varlen_hd{hd}.npz")
    np.savez_compressed(path, rows=rows, out_bf16=bits(ref.reshape(T, H * hd)), dqkv_bf16=bits(a.grad),
                        qkv_probe=qkv.reshape(-1)[::FLASH_HD_PROBE].numpy(), dout_probe=dout.reshape(-1)[::FLASH_HD_PROBE].numpy(),
                        meta=np.array(json.dumps(meta)))
    print("wrote", path, os.path.getsize(path) // 1024, "KiB,", len(rows), "rows,", meta)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir", nargs="?", default=HERE)
    ap.add_argument("--head-dims", default=",".join(str(h) for h in FLASH_HD_CASES),
                    help="comma-separated head dimensions, each one of the test's cases")
    args = ap.parse_args()
    for hd in (int(h) for h in args.head_dims.split(",") if h):
        record(args.out_dir, hd)
