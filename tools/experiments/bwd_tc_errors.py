"""Diagnostic: per-output error of the tensor-core L-TAE backward against the fp32 CUDA-core kernel (ops.ltae_backward)."""
import sys, os
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import crop2seg_b200 as c2s
from crop2seg_b200 import _lib, ops
from c2s_testlib import randomise, synth_inputs, to_dev, bf16_round

def case(c_in, lengths, hw=(4, 4), keep=True, seed=3):
    rng = np.random.RandomState(seed)
    m = c2s.LTAE(in_channels=c_in, n_head=16, d_k=4, mlp=[256, 64], d_model=256)
    randomise(m, rng); m = m.cuda()
    b, t = len(lengths), max(lengths)
    h, w = hw
    x, pos, pad = synth_inputs(rng, b, t, c_in, h, w, lengths)
    x = bf16_round(x + 0.3 * rng.standard_normal(x.shape).astype(np.float32) * (~pad)[:, :, None, None, None])
    n = b * h * w
    go = rng.standard_normal((n, 256)).astype(np.float32)
    ga = rng.standard_normal((16, b, t, h, w)).astype(np.float32)
    ak = (rng.uniform(size=(16, b, t, h, w)) >= 0.1).astype(np.uint8) if keep else None
    params = m._params(torch.device("cuda"))
    spec = ops.LtaeSpec(n_head=16, d_k=4, d_model=256, has_inconv=True, c_out=64, pe_mode=m._pe_mode(), zero_padded=True,
                        attn_drop_p=0.1 if keep else 0.0)
    out = {}
    for name, opt in (("tc", 0), ("tc2", 0), ("gen", 1)):
        with _lib.option(_lib.OPT_LTAE_BWD_KERNEL, opt):
            r = ops.ltae_backward(to_dev(x, dtype=torch.bfloat16), to_dev(pos), to_dev(pad), params, to_dev(go), to_dev(ga),
                                  spec, attn_keep=None if ak is None else to_dev(ak))
            torch.cuda.synchronize()
            out[name] = ({k: v.float().cpu().numpy() for k, v in r.items() if torch.is_tensor(v)}, _lib.last_kernel())
    print(f"C={c_in} lengths={lengths} hw={hw} keep={keep}: kernels {out['tc'][1]} / {out['gen'][1]}")
    for k in out["gen"][0]:
        a, b_ = out["tc"][0][k], out["tc2"][0][k]
        if not np.array_equal(a, b_):
            print(f"   run-to-run {k:10s} max|diff| {np.abs(a - b_).max():10.4g} rel {np.abs(a - b_).max() / max(np.abs(b_).max(), 1e-30):8.2e}")
    for k in out["gen"][0]:
        a, b_ = out["tc"][0][k], out["gen"][0][k]
        print(f"   {k:10s} max|ref| {np.abs(b_).max():10.4g}  max|diff| {np.abs(a - b_).max():10.4g}  rel {np.abs(a - b_).max() / max(np.abs(b_).max(), 1e-30):8.2e}  finite {np.isfinite(a).all()}")

if __name__ == "__main__":
    case(128, [61, 27, 5]); case(64, [61, 33, 0]); case(64, [61, 33, 9]); case(64, [61, 33, 9], keep=False); case(128, [16, 8], hw=(8, 8))
    case(64, [64, 64, 1]); case(128, [3, 1])
    case(128, [61, 40, 27], hw=(32, 16)); case(64, [61, 40, 27, 50], hw=(32, 16))
