"""Time the tcgen05 attention kernel alone (B x 901 tokens, 6 heads)."""
import importlib, sys
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
_lib = importlib.import_module("deep-spectral-segmentation_b200._lib")
lib = _lib.load()
dev = torch.device("cuda:0")
B, T, heads = int(sys.argv[1]) if len(sys.argv) > 1 else 256, 901, 6
d = heads * 64
qkv = (torch.randn(B, T, 3 * d, device=dev) * 1.5).half()
out = torch.empty(B, T, d, device=dev, dtype=torch.float16)
def call():
    _lib.check(lib.dss_op_attention_tc_f16(qkv.data_ptr(), out.data_ptr(), B, T, heads, _lib.stream_ptr()))
for _ in range(3): call()
torch.cuda.synchronize()
ts = []
for _ in range(10):
    s, e = torch.cuda.Event(True), torch.cuda.Event(True)
    s.record(); call(); e.record(); torch.cuda.synchronize(); ts.append(s.elapsed_time(e))
ts.sort()
t = ts[len(ts) // 2]
flops = 4.0 * B * heads * T * T * 64
print(f"B={B}: {t:.3f} ms  ({t / B * 1024 * 12:.1f} ms per 1024 images x 12 blocks)  {flops / t / 1e9:.0f} TFLOP/s")
