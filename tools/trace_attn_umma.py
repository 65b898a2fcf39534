"""Debug helper: phase timeline of the tcgen05 attention-forward tile kernel (needs a build with -DRL_TRACE, e.g.
tools/build_variant.sh trace -DRL_TRACE, selected with RALENET_B200_LIB=build/variants/trace.so).  Runs the forward
op at the s3 / s4 shape (B = 256) in training mode and prints, per phase, the median / max SM-clock delta over the
CTAs, next to the back-to-back launch time of the tile kernel and of the one-window kernel it replaces."""
import ctypes, sys, os
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ecg_denoise_b200 import _lib
from ecg_denoise_b200.ops import pos_table

C = int(sys.argv[1]) if len(sys.argv) > 1 else 128
B = int(sys.argv[2]) if len(sys.argv) > 2 else 256
SAVE = int(sys.argv[3]) if len(sys.argv) > 3 else 1          # 0: inference mode (no q, k, v, o, lse saves)
L, H = 2048 // C, C // 4
W = 4 if C == 64 else 0
dev = torch.device("cuda:0")
g = torch.Generator(device="cpu").manual_seed(0)
x = torch.randn(B, L, C, generator=g).to(dev)
p = dict(ln_w=torch.ones(C), ln_b=torch.zeros(C), wq=torch.randn(C, C, generator=g) * C ** -0.5, bq=torch.zeros(C),
         wkv=torch.randn(2 * C, C, generator=g) * C ** -0.5, bkv=torch.zeros(2 * C),
         wp=torch.randn(C, C, generator=g) * C ** -0.5, bp=torch.zeros(C), table=torch.randn(max(2 * W - 1, 1), H, generator=g))
p = {k: v.to(dev).contiguous() for k, v in p.items()}
pe = pos_table(L, C, dev)
lib = _lib.load()
A = _lib.STRUCTS["rl_attn_fwd_args"]()
y, q, k, v, o = (torch.empty_like(x) for _ in range(5))
lse = torch.empty(B, H, L, device=dev)
A.B, A.L, A.C, A.H, A.W, A.c0, A.flags = B, L, C, H, W, (L - W) // 2 if W else 0, 3
for name, t in dict(x=x, pe=pe, ln_w=p["ln_w"], ln_b=p["ln_b"], wq=p["wq"], bq=p["bq"], wkv=p["wkv"], bkv=p["bkv"],
                    wp=p["wp"], bp=p["bp"], y=y).items():
    setattr(A, name, t.data_ptr())
if SAVE:
    for name, t in dict(q=q, k=k, v=v, o=o, lse=lse).items():
        setattr(A, name, t.data_ptr())
if W:
    A.table = p["table"].data_ptr()
st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def timed(n=20):
    for _ in range(5):
        rc = lib.ralenet_attn_fwd(ctypes.byref(A), st)
        assert rc == 0, lib.ralenet_last_error()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        lib.ralenet_attn_fwd(ctypes.byref(A), st)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / n


_lib.set_attn_umma(0)
print(f"C={C} B={B} save={SAVE}: one-window mma.sync kernel {timed():.2f} us per launch (back to back)")
_lib.set_attn_umma(2)
print(f"C={C} B={B} save={SAVE}: tcgen05 tile kernel       {timed():.2f} us per launch (back to back)")
if not hasattr(lib, "ralenet_debug_trace_read_attn_umma"):
    sys.exit(0)
ncta = ((B * L + 127) // 128) * (C // 32)
buf = (ctypes.c_longlong * (ncta * 16))()
lib.ralenet_debug_trace_read_attn_umma.argtypes = [ctypes.POINTER(ctypes.c_longlong), ctypes.c_int]
print("read rc", lib.ralenet_debug_trace_read_attn_umma(buf, ncta * 16))
full = np.array(buf[:], dtype=np.int64).reshape(ncta, 16)
t = full[:, :13]
d = np.diff(t, axis=1)
names = ["prefetch->pdl", "pdl->alloc/init/table", "PE+LN tile", "qkv stage+issue", "wait qkv", "epilogue1 (q,k,v)",
         "attention core", "o/Wp stage+proj MMA", "epilogue2 ld", "cluster.sync", "reduce+store", "cluster.sync2+dealloc"]
for i, n in enumerate(names):
    print(f"{n:24s} median {np.median(d[:, i]):8.0f}  max {d[:, i].max():8.0f} cycles")
tot = t[:, 12] - t[:, 0]
print("total median", np.median(tot), "max", tot.max(), "cycles; /1.965 GHz =", np.median(tot) / 1965, "us")
