"""Cost of token log-probabilities on the GPU, in one run:

  1. sample_kernel at 64 x 128 256 fp32 logits (the decode step's sampler shape; 33 MB, so the rows are read from L2
     after the first launch, as they are in the engine right after the LM head), CUDA events over many launches:
     logprobs off (the -1 path the engine runs when nobody asks), N = 0 and N = 20, greedy and sampled rows;
  2. the full-size Llama-3-8B decode step at 64 slots (bench_trace.py trace, CUDA graphs + PDL, decode_ms over
     decode_steps from the worker's CUDA-event timing) with no request asking and with all 64 asking N = 5, alternated.

    python tools/logprobs_bench.py [--out FILE] [--reps R]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ollamamq_b200 as mq  # noqa: E402


def P(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def kernel_times(n_launch):
    rows, V = 64, 128256
    g = torch.Generator(device="cuda").manual_seed(0)
    logits = torch.randn(rows, V, device="cuda", generator=g) * 3
    out = torch.zeros(rows, dtype=torch.int32, device="cuda")
    recs = torch.zeros(rows, 41, dtype=torch.float32, device="cuda")
    i32 = lambda v: torch.full((rows,), v, dtype=torch.int32, device="cuda")
    f32 = lambda v: torch.full((rows,), v, dtype=torch.float32, device="cuda")
    seed, cnt = torch.zeros(rows, dtype=torch.int64, device="cuda"), i32(0)

    def launcher(temp, k, p, ntop):
        t, kk, pp = f32(temp), i32(k), f32(p)
        nt = i32(ntop)
        return lambda: mq.lib.mq_debug_sample_logprobs(P(logits), rows, V, V, P(out), P(t), P(kk), P(pp), P(seed), P(cnt),
                                                       P(nt), P(recs))

    cases = [("greedy, logprobs off (-1)", launcher(0.0, 0, 0.0, -1)), ("greedy, N = 0", launcher(0.0, 0, 0.0, 0)),
             ("greedy, N = 20", launcher(0.0, 0, 0.0, 20)),
             ("T 0.8 top_k 40, logprobs off (-1)", launcher(0.8, 40, 0.0, -1)),
             ("T 0.8 top_k 40, N = 20", launcher(0.8, 40, 0.0, 20))]
    res = {name: [] for name, _ in cases}
    for _ in range(3):                      # alternate the cases: the spread of a case is over its three windows
        for name, fn in cases:
            for _ in range(10):
                assert fn() == 0, mq.last_error()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n_launch):
                fn()
            b.record()
            torch.cuda.synchronize()
            res[name].append(a.elapsed_time(b) / n_launch * 1000.0)
    return res


def decode_times(reps):
    from oracle import llama_ref as R
    import bench_trace as BT
    cfg = R.LLAMA3_8B
    prompts = BT.prompts()
    out = {"off": [], "N = 5, all 64 users": []}
    sums = {}
    with mq.Worker(0, mq.model_cfg(cfg, max_batch=BT.USERS, max_seq=BT.PROMPT_LEN + BT.GEN_LEN + 16, max_prefill_tokens=4736,
                                   use_graphs=1, use_pdl=1, model_name="llama-3-8b-random-init")) as wk:
        wk.init_random(seed=0, std=0.02)
        wk.set_timing(True)
        d = mq.Dispatcher([wk], capacity=BT.USERS)
        try:
            for rep in range(reps + 1):          # rep 0 warms up both modes (graph capture, GEMM plans)
                for mode, lp in (("off", False), ("N = 5, all 64 users", True)):
                    wk.reset_stats()
                    ss = [d.submit("user%02d" % u, prompt_tokens=prompts[u], max_new_tokens=BT.GEN_LEN, stream=1,
                                   logprobs=lp, top_logprobs=5) for u in range(BT.USERS)]
                    for s in ss:
                        s.wait(600)
                        assert s.rc == 0, s.err
                    st = wk.stats()
                    sums[mode] = BT.token_checksum([s.tokens() for s in ss])
                    if rep:
                        out[mode].append((st["decode_ms"] / st["decode_steps"], st["decode_steps"],
                                          st["kernel_launches"]))
        finally:
            d.close()
    return out, sums


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=500)
    a = ap.parse_args()
    lines = ["# tools/logprobs_bench.py", "card (name, power limit, max SM clock): %s" % card(), "",
             "## sample_kernel, 64 rows x 128 256 fp32 logits, CUDA events over %d launches; three alternated windows"
             % a.launches, "%-36s %10s %22s" % ("rows", "us/launch", "windows")]
    for name, v in kernel_times(a.launches).items():
        lines.append("%-36s %10.2f %22s" % (name, float(np.median(v)), " ".join("%.2f" % x for x in v)))
    out, sums = decode_times(a.reps)
    lines += ["", "## Llama-3-8B decode step, 64 slots (bench_trace: 64 x 512-token prompts, 128 greedy tokens), "
              "decode_ms / decode_steps; modes alternated, %d runs each" % a.reps,
              "%-24s %12s %28s %14s" % ("mode", "ms/step", "runs", "token checksum")]
    for mode, v in out.items():
        lines.append("%-24s %12.4f %28s %14s" % (mode, float(np.median([x[0] for x in v])),
                                                 " ".join("%.4f(%d)" % (x[0], x[1]) for x in v), sums[mode]))
    lines.append("(ms/step = median; runs = per-run ms/step with its decode step count; both modes launch the same "
                 "kernels: %s kernel launches per run)" % sorted({x[2] for v in out.values() for x in v}))
    txt = "\n".join(lines) + "\n"
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
