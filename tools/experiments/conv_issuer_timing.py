import torch, sys
sys.path.insert(0, "/root/repo")
from crop2seg_b200 import conv as cc
for w in (128, 64, 32):
    x = torch.randn((1024, 64, w, w), device="cuda").to(torch.bfloat16)
    conv = torch.nn.Conv2d(64, 64, 3, padding=1, padding_mode="reflect").cuda()
    for _ in range(2):
        cc.conv2d_reflect_forward(x, conv.weight, conv.bias)
    torch.cuda.synchronize()
for w in (128, 64, 32):
    x = torch.randn((1024, 64, w, w), device="cuda").to(torch.bfloat16)
    conv = torch.nn.Conv2d(64, 64, 4, stride=2, padding=1, padding_mode="reflect").cuda()
    for _ in range(2):
        cc.conv2d_reflect_forward(x, conv.weight, conv.bias, kernel=4, stride=2, padding=1)
    torch.cuda.synchronize()
for c_in, c_out in ((64, 128), (128, 128)):
    x = torch.randn((1024, c_in, 16, 16), device="cuda").to(torch.bfloat16)
    conv = torch.nn.Conv2d(c_in, c_out, 3, padding=1, padding_mode="reflect").cuda()
    for _ in range(2):
        cc.conv2d_reflect_forward(x, conv.weight, conv.bias)
    torch.cuda.synchronize()
