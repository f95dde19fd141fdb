"""N-best situation decode on one GPU: FCGGNN.nbest_situations_from_features at D = 2048 on the synthetic 504 / 190 /
2001 vocabulary with imSitu's role histogram, B in {768, 6144}, verb beam kv = 5, n in {5, 16}, eager and replayed
from a CUDA graph.

The reference point is the top-k decode situations_from_features(k = kv) on the same features: both calls run the
verb path and the role graphs of the same B*kv (image, verb) pairs, so the ratio is the cost of the n-best search
(the k = n row pass and the merge kernel) on top of the top-k decode.  The two calls are timed in the same run, in
alternating rounds, and each ratio is the median over the rounds.  The k = n row pass is timed by CUDA events through
srg_topk_logsoftmax on B*kv*R noun-logit-sized rows.  The merge kernel `k_situation_nbest` has no entry point of its
own, so its device time is read from torch.profiler's kernel records in a separate, untimed pass.  The card's name,
power limit and SM clock are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import situation_recognition_b200 as S  # noqa: E402
from situation_recognition_b200 import _lib  # noqa: E402
from situation_recognition_b200.synthetic import make_batch, make_train_json  # noqa: E402
from bench import ClockSampler  # noqa: E402
from bench_situations import card_info, graphed, preheat, timed, topk_kernel  # noqa: E402


def kernel_ms(fn, names, calls):
    """Mean device time per call of the kernels whose names contain each of `names`, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {n: 0.0 for n in names}
    for ev in prof.events():
        for n in names:
            if n in ev.name and ev.device_type == torch.autograd.DeviceType.CUDA:
                out[n] += ev.device_time / 1e3
    return {n: t / calls for n, t in out.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--D", type=int, default=2048)
    ap.add_argument("--batches", default="768,6144")
    ap.add_argument("--ns", default="5,16")
    ap.add_argument("--kv", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds of the two calls per configuration")
    ap.add_argument("--preheat", type=float, default=3.0, help="seconds of untimed calls before each timed region")
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_nbest.py needs a B200: the decode has no CPU path")
    torch.manual_seed(0)
    enc = S.imsitu_encoder(make_train_json(seed=0), verbose=False)
    m = S.FCGGNN(enc, args.D, backbone=None, precision="bf16").cuda().eval()
    lib = _lib.load()
    R, L = enc.get_max_role_count(), enc.get_num_labels()
    Lpad = (L + 255) // 256 * 256
    kv = args.kv
    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    results = []
    for B in [int(x) for x in args.batches.split(",")]:
        fv, fn, _, _ = make_batch(enc, B, args.D, seed=1234, device="cuda")
        topk = lambda: m.situations_from_features(fv, fn, k=kv)                                  # noqa: E731
        for n in [int(x) for x in args.ns.split(",")]:
            nbest = lambda: m.nbest_situations_from_features(fv, fn, n=n, verb_beam=kv)          # noqa: E731
            res = {"B": B, "kv": kv, "n": n}
            for mode in ("eager", "graph"):
                fa, fb = (topk, nbest) if mode == "eager" else (graphed(topk).replay, graphed(nbest).replay)
                preheat(lambda: (fa(), fb()), args.preheat)
                ta, tb = [], []
                for _ in range(args.rounds):
                    ta.append(timed(fa, args.iters))
                    tb.append(timed(fb, args.iters))
                res["ms_topk_" + mode] = statistics.median(ta)
                res["ms_nbest_" + mode] = statistics.median(tb)
                res["nbest_over_topk_" + mode] = statistics.median(b / a for a, b in zip(ta, tb))
                res["situations_per_s_" + mode] = B * n / statistics.median(tb) * 1e3
            res["row_pass_k_n"] = topk_kernel(lib, B * kv * R, L, Lpad, n, args.iters)
            prof = kernel_ms(nbest, ["k_situation_nbest", "k_row_topk_logsoftmax"], args.iters)
            res["ms_merge_kernel_profiler"] = prof["k_situation_nbest"]
            res["ms_row_kernels_profiler"] = prof["k_row_topk_logsoftmax"]
            res["merge_share_of_topk_call"] = prof["k_situation_nbest"] / res["ms_topk_eager"]
            results.append(res)
            torch.cuda.empty_cache()
    clk = clocks.stop()
    line = {"metric": "nbest_situations_decode", "D": args.D, "precision": "bf16", "card": card_info(), "clocks": clk,
            "preheat_s": args.preheat, "iters": args.iters, "rounds": args.rounds, "results": results}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
