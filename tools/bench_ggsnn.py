"""GGSNN.forward + its backward on caller-supplied node states (model.ggsnn) on one GPU, D = 2048, against the fused
noun path that runs the same role graphs.

Per batch B (images; the role graph has B*R dense rows):
  * noun mode with the encoder's mask (FCGGNN.gather_mask of synthetic verb ids), forward + backward with and without
    mask.requires_grad; the verb node at the largest B;
  * the baseline: predict_nouns + nouns_loss, forward + backward, eval mode, with one row per role slot
    (set_compact_rows(0)) so that it propagates the same B*R rows -- it also runs the node init, the classifier and
    the classifier's backward, i.e. strictly more work;
  * ms per call (CUDA events around back-to-back calls after a timed warm-up), and the achieved GB/s of the
    aggregation backward `k_aggregate_t` from its algorithmic bytes (da, e and ada, plus h_t with the mask gradient,
    at 2 D bytes per row each, plus the R*R fp32 mask per image) over its kernel time, taken with torch.profiler in a
    separate pass and compared with the 6550 GB/s copy bandwidth DESIGN.md uses.
The card's name, power limit and SM clock are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import situation_recognition_b200 as S  # noqa: E402
from situation_recognition_b200.synthetic import make_batch, make_train_json  # noqa: E402
from bench import ClockSampler  # noqa: E402
from bench_situations import COPY_GBPS, card_info, preheat, timed  # noqa: E402


def agg_t_kernel_ms(fn, dmask, calls=5):
    """Mean device time (ms) of one k_aggregate_t launch in `calls` calls of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    want = "k_aggregate_t<%s>" % ("true" if dmask else "false")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    total, n = 0.0, 0
    for k in prof.key_averages():
        if want in k.key:
            total += getattr(k, "device_time_total", None) or k.cuda_time_total
            n += k.count
    if n == 0:
        raise RuntimeError("no %s launch in the profile" % want)
    return total / n / 1e3, n // calls


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--D", type=int, default=2048)
    ap.add_argument("--batches", default="768,6144")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--preheat", type=float, default=2.0, help="seconds of untimed calls before each timed region")
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ggsnn.py needs a B200: the GGNN stage has no CPU path")
    torch.manual_seed(0)
    enc = S.imsitu_encoder(make_train_json(seed=0), verbose=False)
    m = S.FCGGNN(enc, args.D, backbone=None, precision="bf16").cuda().eval()
    m._engine_for(torch.device("cuda", torch.cuda.current_device())).set_compact_rows(0)
    R, D = enc.get_max_role_count(), args.D
    params = list(m.parameters())
    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    results = []
    batches = [int(x) for x in args.batches.split(",")]
    for B in batches:
        _, fn, gt_verb, gt_nouns = make_batch(enc, B, D, seed=1234, device="cuda")
        mask = m.gather_mask(gt_verb)[1]
        gen = torch.Generator(device="cuda").manual_seed(B)
        hidden = torch.randn(B * R, D, device="cuda", generator=gen).relu_().requires_grad_(True)
        G = torch.randn(B * R, D, device="cuda", generator=gen)

        def zero():
            for p in params + [hidden, mask]:
                p.grad = None

        def ggsnn_step(mask_grad):
            mk = mask.requires_grad_(mask_grad)
            zero()
            m.ggsnn(hidden, mask=mk).backward(G)

        def fused_step():
            zero()
            m.nouns_loss(m.predict_nouns(fn, gt_verb, B), gt_nouns).backward()

        res = {"B": B, "rows": B * R}
        for key, fn_ in (("ms_fused_nouns", fused_step), ("ms_ggsnn", lambda: ggsnn_step(False)),
                         ("ms_ggsnn_dmask", lambda: ggsnn_step(True))):
            preheat(fn_, args.preheat)
            res[key] = timed(fn_, args.iters)
        res["ggsnn_vs_fused"] = res["ms_ggsnn"] / res["ms_fused_nouns"]
        res["ggsnn_dmask_vs_fused"] = res["ms_ggsnn_dmask"] / res["ms_fused_nouns"]
        for dm in (False, True):
            ms, per_call = agg_t_kernel_ms(lambda: ggsnn_step(dm), dm)
            nbytes = B * R * 2 * D * (4 if dm else 3) + B * R * R * 4
            res["k_aggregate_t_dmask" if dm else "k_aggregate_t"] = {
                "ms": ms, "launches_per_call": per_call, "gb_per_s": nbytes / ms / 1e6,
                "of_copy_bw": nbytes / ms / 1e6 / COPY_GBPS, "l2_resident": nbytes < 126e6}
        mask.requires_grad_(False)
        results.append(res)
        del hidden, G, mask
        torch.cuda.empty_cache()
    Bv = max(batches)
    hv = torch.randn(Bv, D, device="cuda").relu_().requires_grad_(True)
    Gv = torch.randn(Bv, D, device="cuda")

    def verb_step():
        for p in params + [hv]:
            p.grad = None
        m.ggsnn(hv, verb=True).backward(Gv)

    preheat(verb_step, args.preheat)
    verb = {"B": Bv, "ms_ggsnn_verb": timed(verb_step, args.iters)}
    clk = clocks.stop()
    line = {"metric": "ggsnn_forward_backward", "D": D, "R": R, "precision": "bf16", "card": card_info(),
            "clocks": clk, "preheat_s": args.preheat, "iters": args.iters, "nouns": results, "verb": verb}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
