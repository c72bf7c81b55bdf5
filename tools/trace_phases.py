"""Per-phase clock64 trace of the GEMM kernels (CTA (0,1)) for the decode-step shapes."""
import ctypes as C, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import torch
from novic_b200 import synth, default_decoder, _abi
lib = _abi.lib()
dims = synth.DecoderDims(num_layers=1)
model = default_decoder(dims, synth.synth_state_dict(dims, seed=1), num_layers=1).to("cuda:0")
B = 4096
e = synth.synth_embeddings(B, seed=1234).cuda()
tgt = torch.zeros(B, 1, dtype=torch.int64, device="cuda")
names = {0: "entry", 1: "setup done", 2: "first TMA issued", 3: "last TMA issued", 4: "first stage landed", 5: "last MMA committed", 11: "epi: residual prefetched",
         6: "epi: accumulator ready", 13: "epi: hidden tile written (gelu)", 12: "mma: second GEMM committed", 7: "epi: stats written",
         8: "epi: after sync1 / epilogue done", 9: "epi: stores issued", 10: "exit sync passed"}
with torch.inference_mode():
    st = model._state(torch.device("cuda:0"))
    _abi.check(lib.novic_set_use_graphs(st["handle"], 0))
    model.generate(e, False, True, 1.0, 0.0, None, None, False)
    # GEMM launches of a 1-layer greedy decode: prefix, qkv, block, logits (prefill), then qkv, block, logits per step (the block kernels have
    # their own tools: trace_fused.py, trace_blockrows.py)
    kinds = {4: "qkv (decode, M=4096)", 6: "logits (decode)"}
    for target, label in kinds.items():
        _abi.check(lib.novic_debug_trace(None, 1 + target))
        model.generate(e, False, True, 1.0, 0.0, None, None, False)
        buf = (C.c_int64 * 32)()
        _abi.check(lib.novic_debug_trace(buf, 0))
        t0 = buf[0]
        print(label)
        for i in sorted(names, key=lambda k: buf[k]):
            if buf[i]:
                print(f"   {names[i]:36s} +{buf[i] - t0:7d} cycles")
        for i in range(8):   # persistent kernels: per-tile epilogue spans of CTA 0
            if buf[16 + 2 * i]:
                print(f"   tile {i}: accumulator ready +{buf[16 + 2 * i] - t0:7d}, epilogue done +{buf[17 + 2 * i] - t0:7d}")
