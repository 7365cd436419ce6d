import sys, numpy as np
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT / "cutter-vad_b200", ROOT / "oracle", ROOT / "tests"): sys.path.insert(0, str(p))
from conftest import synth_streams, V5_ONNX
from real_time_vad.engine.stream_engine import StreamEngine
from vad_oracle import RefLib, RefV5, v5_blob
ref = RefV5(v5_blob(str(V5_ONNX)), RefLib())
T = 30
rng = np.random.default_rng(3)
base = synth_streams(8, 512*T, seed=9)
cases = {
 "zeros": np.zeros((4, 512*T), np.float32),
 "tiny 1e-6": (1e-6*rng.standard_normal((4,512*T))).astype(np.float32),
 "denormal 1e-40": np.full((4,512*T), 1e-40, np.float32),
 "loud x30": (30*base[:4]).astype(np.float32),
 "int16-scale x32768": (32768*base[:4]).astype(np.float32),
 "huge 1e8": (1e8*base[:4]).astype(np.float32),
 "square full scale": np.sign(np.sin(2*np.pi*200*np.arange(512*T)/16000))[None,:].repeat(4,0).astype(np.float32),
 "dc 0.5": np.full((4,512*T), 0.5, np.float32),
 "impulses": (rng.random((4,512*T))>0.999).astype(np.float32),
}
for math in ("tc","fp32"):
    eng = StreamEngine(max_streams=8, math=math)
    for name, x in cases.items():
        for dn in (False, True):
            eng.reset(); eng.configure(enable_denoising=dn)
            want,_,_ = ref.run(x, T, denoise=dn)
            one = eng.step(x).probs
            eng.reset()
            steps = np.stack([eng.step(x[:, j*512:(j+1)*512]).probs[:,0] for j in range(T)],1)
            print(f"{math:5s} {name:22s} dn={int(dn)} max|dp| one-call {np.abs(one-want).max():.2e} per-frame {np.abs(steps-want).max():.2e}  p range [{want.min():.3f},{want.max():.3f}] finite={np.isfinite(one).all() and np.isfinite(steps).all()}")
