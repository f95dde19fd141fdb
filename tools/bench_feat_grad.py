"""Cost of the feature gradients (dL/dfeat) of the fused paths on one GPU, D = 2048.

  * The training step as the launcher runs it on features: forward_features + verb_loss + nouns_loss + backward, train
    mode (Philox dropout), flat gradient / parameter buffers, at each B, with and without requires_grad on both feature
    tensors.  The two variants alternate within one run (`--reps` rounds of `--iters` timed steps each, CUDA events);
    the result is the median round, the ratio of the medians, and each variant's spread (max - min) / median.
  * In a separate torch.profiler pass, the kernels that produce dL/dfeat: the three variants of k_node_init_bwd
    (embedding gradients only -- what runs without feature gradients --, embeddings + dfeat, and dfeat only with frozen
    embeddings) on a predict_nouns + nouns_loss backward at the gt verbs, and k_node_init_verb_bwd on predict_verb +
    verb_loss.  Algorithmic bytes: dh0 (4 B) and the bf16 initial state (2 B) per node element, verb_emb (4 B) per image
    element, feat (4 B, embedding gradients only) and the dfeat store (4 B) per image element; the ~190 role_emb rows and
    the embedding-gradient atomics stay in L2 and are not counted.  GB/s over the 6550 GB/s copy bandwidth DESIGN.md
    uses.
The card's name, power limit and SM clock are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import situation_recognition_b200 as S  # noqa: E402
from situation_recognition_b200 import parallel  # noqa: E402
from situation_recognition_b200.synthetic import make_batch, make_train_json  # noqa: E402
from bench import ClockSampler  # noqa: E402
from bench_situations import COPY_GBPS, card_info, preheat, timed  # noqa: E402

KERNELS = {"emb": "k_node_init_bwd<true, false>", "emb_dfeat": "k_node_init_bwd<true, true>",
           "dfeat": "k_node_init_bwd<false, true>", "verb": "k_node_init_verb_bwd"}


def kernel_us(fn, name, calls=5):
    """Mean device time (µs) of one launch of kernel `name` in `calls` calls of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    total, n = 0.0, 0
    for k in prof.key_averages():
        if name in k.key:
            total += getattr(k, "device_time_total", None) or k.cuda_time_total
            n += k.count
    if n != calls:
        raise RuntimeError("%d launches of %s in %d calls" % (n, name, calls))
    return total / n


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--D", type=int, default=2048)
    ap.add_argument("--batches", default="768,6144")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5, help="alternating rounds of each variant")
    ap.add_argument("--preheat", type=float, default=2.0, help="seconds of untimed steps before the timed rounds")
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_feat_grad.py needs a B200: the GGNN stage has no CPU path")
    torch.manual_seed(0)
    D = args.D
    enc = S.imsitu_encoder(make_train_json(seed=0), verbose=False)
    dev = torch.device("cuda", torch.cuda.current_device())

    def model(frozen_emb=False, flat=True):
        m = S.FCGGNN(enc, D, backbone=None, precision="bf16").to(dev)
        if frozen_emb:
            m.role_emb.weight.requires_grad_(False)
            m.verb_emb.weight.requires_grad_(False)
        return m, (parallel.attach(m, flat_params=True) if flat else None)

    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    steps, kernels = [], []
    for B in [int(x) for x in args.batches.split(",")]:
        fv0, fn0, gt_verb, gt_nouns = make_batch(enc, B, D, seed=1234, device="cuda")
        fv0, fn0 = fv0 - 0.4, fn0 - 0.4
        m, flat = model()
        m.train()
        feats = {False: (fv0, fn0), True: (fv0.clone().requires_grad_(True), fn0.clone().requires_grad_(True))}

        def step(want):
            fv, fn = feats[want]
            fv.grad = fn.grad = None
            flat.zero()
            pv, pn, _ = m.forward_features(fv, fn, gt_verb)
            (m.verb_loss(pv, gt_verb) + m.nouns_loss(pn, gt_nouns)).backward()

        for want in (False, True):
            preheat(lambda: step(want), args.preheat)
        rounds = {False: [], True: []}
        for _ in range(args.reps):
            for want in (False, True):
                rounds[want].append(timed(lambda: step(want), args.iters))
        med = {w: statistics.median(r) for w, r in rounds.items()}
        steps.append({"B": B, "ms_step": med[False], "ms_step_feat_grad": med[True], "ratio": med[True] / med[False],
                      "spread": {"no_feat_grad": (max(rounds[False]) - min(rounds[False])) / med[False],
                                 "feat_grad": (max(rounds[True]) - min(rounds[True])) / med[True]},
                      "rounds_ms": {"no_feat_grad": rounds[False], "feat_grad": rounds[True]}})
        del m, flat

        # kernel pass: eval mode (no dropout), one path per call, the gt verbs
        rows = sum(enc.get_role_count(int(v)) for v in gt_verb.tolist())
        per_tensor, _ = model(flat=False)
        frozen, _ = model(frozen_emb=True)
        per_tensor.eval()
        frozen.eval()
        res = {"B": B, "node_rows": rows}

        def nouns(mm, want):
            fn = feats[want][1]
            fn.grad = None
            mm.nouns_loss(mm.predict_nouns(fn, gt_verb, B), gt_nouns).backward()

        def verb():
            fv = feats[True][0]
            fv.grad = None
            per_tensor.verb_loss(per_tensor.predict_verb(fv, B), gt_verb).backward()

        node = rows * D * (4 + 2) + B * D * 4            # dh0 + bf16 h0 per node element, verb_emb per image element
        for key, fn_, nbytes in (("emb", lambda: nouns(per_tensor, False), node + B * D * 4),
                                 ("emb_dfeat", lambda: nouns(per_tensor, True), node + B * D * 8),
                                 ("dfeat", lambda: nouns(frozen, True), node + B * D * 4),
                                 ("verb", verb, B * D * (4 + 2 + 4))):
            fn_()
            us = kernel_us(fn_, KERNELS[key])
            res[key] = {"kernel": KERNELS[key], "us": us, "bytes": nbytes, "gb_per_s": nbytes / us / 1e3,
                        "of_copy_bw": nbytes / us / 1e3 / COPY_GBPS, "l2_resident": nbytes < 126e6}
        res["emb_dfeat_vs_emb"] = res["emb_dfeat"]["us"] / res["emb"]["us"]
        kernels.append(res)
        del per_tensor, frozen, feats
        torch.cuda.empty_cache()
    clk = clocks.stop()
    line = {"metric": "feature_gradients", "D": D, "precision": "bf16", "card": card_info(), "clocks": clk,
            "preheat_s": args.preheat, "iters": args.iters, "reps": args.reps, "steps": steps, "kernels": kernels}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
