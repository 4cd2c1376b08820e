"""Time the critic kernels alone: python tools/critic_bench.py [envs] [lstm_hidden] [mlp_hidden,comma] [iters] [seq_len] [lstm_layers]"""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, taco_b200
n = int(sys.argv[1]) if len(sys.argv) > 1 else 262144
hid = int(sys.argv[2]) if len(sys.argv) > 2 else 64
mlp = [int(x) for x in (sys.argv[3] if len(sys.argv) > 3 else "256,256,256").split(",")]
iters = int(sys.argv[4]) if len(sys.argv) > 4 else 30
T, IN = (int(sys.argv[5]) if len(sys.argv) > 5 else 5), 26
L = int(sys.argv[6]) if len(sys.argv) > 6 else 1
gen = torch.Generator().manual_seed(1)
lstm = [(torch.randn(4 * hid, IN if l == 0 else hid, generator=gen) * 0.2, torch.randn(4 * hid, hid, generator=gen) * 0.15,
         torch.randn(4 * hid, generator=gen) * 0.1, torch.randn(4 * hid, generator=gen) * 0.1) for l in range(L)]
sizes = [hid] + mlp + [1]
ws = [torch.randn(sizes[l + 1], sizes[l], generator=gen) * (1.0 / sizes[l] ** 0.5) for l in range(len(sizes) - 1)]
bs = [torch.randn(sizes[l + 1], generator=gen) * 0.1 for l in range(len(sizes) - 1)]
c = taco_b200.CriticLSTM(IN, T, hid, mlp, lstm_layers=L)
c.load(lstm, ws, bs)
states = torch.randn(n, T, IN, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
out = torch.empty(n, 1, device="cuda")
def t(fn, it):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(it): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / it
ms_tc = t(lambda: c.forward(states, tensor_cores=True, out=out), iters)
ms_fp = t(lambda: c.forward(states, tensor_cores=False, out=out), max(iters // 10, 2))
# algorithmic FLOPs per env: T LSTM steps of 2 (in + H) 4H in the bottom layer and of 2 (H + H) 4H in each layer above, then the MLP
flops = (T * 2.0 * (IN + hid) * 4 * hid + (L - 1) * T * 2.0 * (hid + hid) * 4 * hid
         + 2.0 * sum(sizes[i] * sizes[i + 1] for i in range(len(sizes) - 1))) * n
ref = c.forward(states[:4096], tensor_cores=False)
got = c.forward(states[:4096], tensor_cores=True)
print(json.dumps({"envs": n, "lstm_hidden": hid, "lstm_layers": L, "mlp": sizes, "tc_ms": ms_tc, "fp32_ms": ms_fp, "tflops": flops / ms_tc / 1e9,
                  "flops_per_env": flops / n, "max_abs_diff_vs_fp32_kernel": float((ref - got).abs().max())}))
