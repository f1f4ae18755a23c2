"""Float64 torch reference of U-TAE's skip convolution with its BatchNorm normalising by batch statistics (training mode):
``relu(BatchNorm2d_train(Conv2d_1x1(skip)))`` on the aggregated skip map, differentiable, with the bf16 roundings of the
fused kernels (the skip map s and the pre-BatchNorm z are stored as bf16) as identity-gradient steps.  TEST
INFRASTRUCTURE ONLY; checked against ``nn.BatchNorm2d`` in training mode in tests/test_cpu_skipconv_bstats.py."""
import torch


def bf16_value(t):
    """t rounded to bfloat16 in value, identity in gradient."""
    return t + (t.detach().float().to(torch.bfloat16).to(t.dtype) - t).detach()


def skip_conv_bstats(s, conv_weight, conv_bias, bn_weight, bn_bias, eps=1e-5, round_z=False, relu_mask=None,
                     z_value=None):
    """s[B,C,H,W] float64 -> dict(out, pre, z, mean, var): z = W s + b (bf16-valued with ``round_z``; the values of
    ``z_value`` with z's gradient when given), the batch mean and biased variance of z over B*H*W, pre = the BatchNorm
    output, out = relu(pre) or pre * relu_mask."""
    z = torch.nn.functional.conv2d(s, conv_weight, conv_bias)
    if round_z:
        z = bf16_value(z)
    if z_value is not None:
        z = z + (z_value.to(z.dtype) - z).detach()
    mean = z.mean(dim=(0, 2, 3))
    var = z.var(dim=(0, 2, 3), unbiased=False)
    pre = (z - mean[None, :, None, None]) / torch.sqrt(var[None, :, None, None] + eps)
    if bn_weight is not None:
        pre = pre * bn_weight[None, :, None, None]
    if bn_bias is not None:
        pre = pre + bn_bias[None, :, None, None]
    out = torch.relu(pre) if relu_mask is None else pre * relu_mask
    return {"out": out, "pre": pre, "z": z, "mean": mean, "var": var}


@torch.no_grad()
def running_update(running_mean, running_var, num_batches_tracked, mean, var, n, momentum):
    """nn.BatchNorm2d's train-mode update from the batch mean / biased variance over n values per channel."""
    num_batches_tracked += 1
    m = momentum if momentum is not None else 1.0 / float(num_batches_tracked)
    running_mean.mul_(1 - m).add_(m * mean)
    running_var.mul_(1 - m).add_(m * var * n / (n - 1))
    return num_batches_tracked
