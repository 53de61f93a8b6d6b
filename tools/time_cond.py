"""Times the cond GEMM stage (cwg_cond) at BASELINE config-2 size."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cookietts_b200 import WaveGlow, _cabi
from cookietts_b200.synthetic import ModelConfig, synthetic_state_dict
import bench
B, TM = 16, 861
sd = synthetic_state_dict(ModelConfig(), 1234)
lib = _cabi.load()
for prec in sys.argv[1:] or ["bf16x3", "f16f8", "bf16"]:
    m = WaveGlow(precision=prec, **bench.MODEL_KW); m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}); m = m.cuda().eval(); m._ensure_packed()
    mode = _cabi.MODES[prec]
    mel = (torch.randn(B, 80, TM, device="cuda") * 2 - 5).clamp(-11.5, 2)
    bias = m._cond_bias(B, None)
    n = lib.cwg_workspace_bytes(m._ccfg, mode, B, TM)
    ws = torch.zeros(n + 1024, dtype=torch.uint8, device="cuda"); ptr = (ws.data_ptr() + 1023) // 1024 * 1024
    out = torch.zeros(B * TM * 32 * 256 * 4, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    run = lambda: _cabi.check(lib.cwg_cond(m._ccfg, m._cw, mode, 3, mel.data_ptr(), bias.data_ptr(), out.data_ptr(), ptr, n, B, TM, st))
    for _ in range(3): run()
    ts = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); run(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    print(prec, "cond stage median %.1f us (incl. im2col)" % (np.median(ts) * 1e3), "sum", float(out[:1000].float().sum()))
