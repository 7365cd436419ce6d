import sys, numpy as np, ctypes as C
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1] / 'cutter-vad_b200'))
from real_time_vad.engine import capi
L = capi.dev_lib()
def bf16_bits(x):
    u = x.astype(np.float32).view(np.uint32); r = ((u >> 16) & 1) + 0x7FFF
    return ((u + r) >> 16).astype(np.uint16)
def bf16_val(b): return (b.astype(np.uint32) << 16).view(np.float32)
def split3(x):
    parts=[]; r = x.astype(np.float32)
    for i in range(3):
        b = bf16_bits(r); parts.append(b); r = (r - bf16_val(b)).astype(np.float32)
    return parts
def probe(a,b):
    D = np.zeros((128,32), np.float32)
    rc = L.cvad_tc_probe(0, a.ctypes.data, b.ctypes.data, D.ctypes.data); assert rc==0
    return D
rng = np.random.default_rng(1)
for trial,(sa,sb) in enumerate([(1,1),(1,1),(0.05,0.3)]):
    A = (sa*rng.standard_normal((128,256))).astype(np.float32); B = (sb*rng.standard_normal((32,256))).astype(np.float32)
    if trial==1: A=np.abs(A); B=np.abs(B)   # all-positive: worst case for truncation bias
    a = bf16_bits(A); b = bf16_bits(B)
    D = probe(a,b); want = bf16_val(a).astype(np.float64) @ bf16_val(b).astype(np.float64).T
    f32 = (bf16_val(a) @ bf16_val(b).T)
    print('single pass: max rel err (vs |want|max)', np.abs(D-want).max()/np.abs(want).max(), 'numpy f32:', np.abs(f32-want).max()/np.abs(want).max(), 'mean signed', ((D-want)/np.abs(want).max()).mean())
    As = split3(A); Bs = split3(B)
    exact = A.astype(np.float64) @ B.astype(np.float64).T
    acc = np.zeros((128,32), np.float32); acc64 = np.zeros((128,32))
    for (i,j) in [(2,0),(0,2),(1,1),(1,0),(0,1),(0,0)]:
        d = probe(As[i],Bs[j]); acc = (acc + d).astype(np.float32); acc64 += d
    print('  6-pass: f32-sum', np.abs(acc-exact).max()/np.abs(exact).max(), ' f64-sum', np.abs(acc64-exact).max()/np.abs(exact).max(), ' plain f32 matmul', np.abs((A@B.T)-exact).max()/np.abs(exact).max())
