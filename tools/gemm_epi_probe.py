"""Times dss_op_gemm_f16 (the product launch path, all epilogues) on the ViT-S shapes of the 256/296-image step."""
import importlib, os, sys
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
_lib = importlib.import_module("deep-spectral-segmentation_b200._lib")
lib = _lib.load()
dev = torch.device("cuda:0")
M = int(os.environ.get("PROBE_IMAGES", "296")) * 901
EPI = {"bias_f16": 0, "gelu_f16": 1, "resid_f32": 2}
def run(name, N, K, epi, iters=12):
    A = torch.randn(M, K, device=dev).half(); W = (torch.randn(N, K, device=dev) * 0.05).half()
    bias = torch.randn(N, device=dev) * 0.1
    out = torch.zeros(M, N, device=dev, dtype=torch.float32 if epi == "resid_f32" else torch.float16)
    flush = torch.empty(64 * 1024 * 1024, device=dev)
    def call():
        _lib.check(lib.dss_op_gemm_f16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, EPI[epi], None, 0, 0, _lib.stream_ptr()))
    for _ in range(3): call()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.zero_()
        s, e = torch.cuda.Event(True), torch.cuda.Event(True)
        s.record(); call(); e.record(); torch.cuda.synchronize(); ts.append(s.elapsed_time(e))
    ts.sort(); t = ts[len(ts)//2]
    out.zero_(); call(); torch.cuda.synchronize()
    ref = A[:512].float() @ W.float().T + bias
    if epi == "gelu_f16": ref = torch.nn.functional.gelu(ref)
    err = (out[:512].float() - ref).abs().max().item()
    print(f"{name:5s} N={N:5d} K={K:5d} {epi:9s}: {t*1e3:8.1f} us  {2*M*N*K/t/1e9:8.1f} TFLOP/s  err {err:.2e}", flush=True)
print("M =", M)
run("qkv", 1152, 384, "bias_f16"); run("fc1", 1536, 384, "gelu_f16"); run("fc2", 384, 1536, "resid_f32"); run("proj", 384, 384, "resid_f32")
