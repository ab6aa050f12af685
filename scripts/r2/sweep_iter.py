"""Round-2 A/B of the thread-per-chain iteration kernel on the headline workload (funnel, HMC nSteps=5, parity math):
ms per launch of rn_k_iter for register caps x CTA sizes; the sample tensors of all variants must be bit-identical."""
import hashlib, json, os, sys, time
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
import numpy as np
import torch
from rainier_b200 import abi, api

ROOT = os.path.join(os.path.dirname(__file__), "..", "..")
C_, I_ = 151552, 100
rir = open(os.path.join(ROOT, "rainier_b200", "models", sys.argv[1] if len(sys.argv) > 1 else "funnel10.rir"), "rb").read()
caps = [int(x) for x in os.environ.get("SWEEP_CAPS", "128,96").split(",")]
blocks = [int(x) for x in os.environ.get("SWEEP_BLOCKS", "128").split(",")]
defsets = os.environ.get("SWEEP_DEFS", "").split("|")
math = abi.RN_MATH_FAST if os.environ.get("SWEEP_FAST") else abi.RN_MATH_PARITY
ref = None
for defs in defsets:
  for cap in caps:
    for block in blocks:
        # tokens ENV:NAME=VALUE set an environment switch of the runtime / emitter for this variant instead of a -D
        for tok in defs.split():
            if tok.startswith("ENV:"):
                os.environ[tok[4:].split("=")[0]] = tok.split("=", 1)[1]
        os.environ["RN_MAXRREGCOUNT"] = str(cap)
        os.environ["RN_BLOCK"] = str(block)
        model = api.CudaModel(rir, [], device=0)
        n = model.nVars
        cfg = api.make_config(iterations=I_, warmupIterations=0, sampler=api.HMCSampler(5), stepSizeTuner=api.StaticStepSize(0.1),
                              massMatrixTuner=api.IdentityMassMatrixTuner(), mathMode=math, launchIterations=I_)
        smp = api.CudaSampler(model, cfg, seeds=np.arange(C_, dtype=np.int64) + 1000)
        smp.warmup(-1)
        stream = torch.cuda.ExternalStream(smp.stream)
        d = torch.empty((I_, n, C_), dtype=torch.float64, device="cuda")
        smp.run(I_, d.data_ptr()); smp.sync()
        h = hashlib.sha1(d[:, :, :4096].cpu().numpy().tobytes()).hexdigest()[:12]
        if ref is None: ref = h
        for _ in range(2): smp.run(I_, d.data_ptr())
        smp.sync()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
        for a, b in ev:
            a.record(stream); smp.run(I_, d.data_ptr()); b.record(stream)
        smp.sync(); torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in ev)
        print(json.dumps({"defs": defs, "cap": cap, "block": block, "ms_min": ms[0], "ms_med": ms[2], "rate": C_ * I_ * 5 / (ms[2] * 1e-3),
                          "same_bits": h == ref, "hash": h}), flush=True)
        smp.close(); model.close()
        for tok in defs.split():
            if tok.startswith("ENV:"):
                os.environ.pop(tok[4:].split("=")[0], None)
