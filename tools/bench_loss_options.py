"""Cost of the loss options (label smoothing, class weights) in the training step on one GPU, D = 2048, B = 6144.

The step is sr.py's: forward (verb path + both noun paths, train mode, Philox dropout), verb_loss + nouns_loss of the
predicted-verb path and the logged gt-verb nouns_loss, backward, and the fused clip + Adamax over flat buffers.  Four
settings of the objective:
  * defaults     : the reference's plain losses (the default-option kernels; the step bench.py times);
  * eps          : label_smoothing = 0.1 on both losses;
  * eps_weights  : label_smoothing = 0.1 and class weights on the nouns (the option kernels with the stats route);
  * torch_composed: the eps_weights objective composed from F.cross_entropy on the returned logits (a user's
                    workaround without the options: fp32 autograd, no side channel, no softmax statistics).
The settings alternate within one run (`--reps` rounds of `--iters` timed steps each, CUDA events); the result is the
median round per setting, its overhead over the defaults and each setting's spread (max - min) / median.  The card's
name, power limit and SM clock are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import situation_recognition_b200 as S  # noqa: E402
from situation_recognition_b200 import parallel  # noqa: E402
from situation_recognition_b200.synthetic import make_batch, make_train_json  # noqa: E402
from bench import ClockSampler  # noqa: E402
from bench_situations import card_info, preheat, timed  # noqa: E402

SETTINGS = ("defaults", "eps", "eps_weights", "torch_composed")


def composed_nouns_loss(pn, gt, weight, eps, L):
    """The reference's nouns_loss (sum over the 3 annotations) written with F.cross_entropy and the options."""
    z = pn.reshape(-1, L)
    return sum(F.cross_entropy(z, gt[:, a].reshape(-1), weight=weight, ignore_index=L, label_smoothing=eps)
               for a in range(3))


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--D", type=int, default=2048)
    ap.add_argument("--batch", type=int, default=6144)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5, help="alternating rounds of each setting")
    ap.add_argument("--preheat", type=float, default=2.0, help="seconds of untimed steps per setting before timing")
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_loss_options.py needs a B200: the GGNN stage has no CPU path")
    torch.manual_seed(0)
    D, B = args.D, args.batch
    enc = S.imsitu_encoder(make_train_json(seed=0), verbose=False)
    L = enc.get_num_labels()
    dev = torch.device("cuda", torch.cuda.current_device())
    fv, fn, gt_verb, gt_nouns = make_batch(enc, B, D, seed=1234, device="cuda")
    wn = (torch.rand(L, generator=torch.Generator().manual_seed(1)) + 0.5).to(dev)
    m = S.FCGGNN(enc, D, backbone=None, precision="bf16").to(dev).train()
    flat = parallel.attach(m, flat_params=True)
    opt = parallel.FlatAdamax(flat, lr=0.002, max_norm=1.0)
    objective = {"defaults": ({}, {}),
                 "eps": ({"label_smoothing": 0.1}, {"label_smoothing": 0.1}),
                 "eps_weights": ({"label_smoothing": 0.1}, {"label_smoothing": 0.1, "weight": wn})}

    def step(setting):
        flat.zero()
        pv, pn, gpn = m(fv, gt_verb, img_nouns=fn)
        if setting == "torch_composed":
            vl = F.cross_entropy(pv, gt_verb, label_smoothing=0.1)
            nl = composed_nouns_loss(pn, gt_nouns, wn, 0.1, L)
            gl = composed_nouns_loss(gpn, gt_nouns, wn, 0.1, L)
        else:
            vkw, nkw = objective[setting]
            vl, nl, gl = m.verb_loss(pv, gt_verb, **vkw), m.nouns_loss(pn, gt_nouns, **nkw), \
                m.nouns_loss(gpn, gt_nouns, **nkw)
        (vl + nl).backward()
        opt.step()
        return gl

    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    for s in SETTINGS:
        preheat(lambda: step(s), args.preheat)
    rounds = {s: [] for s in SETTINGS}
    for _ in range(args.reps):
        for s in SETTINGS:
            rounds[s].append(timed(lambda: step(s), args.iters))
    clk = clocks.stop()
    med = {s: statistics.median(r) for s, r in rounds.items()}
    res = {s: {"ms_step": med[s], "overhead_vs_defaults": med[s] / med["defaults"] - 1.0,
               "spread": (max(rounds[s]) - min(rounds[s])) / med[s], "rounds_ms": rounds[s]} for s in SETTINGS}
    line = {"metric": "loss_options_step", "D": D, "B": B, "precision": "bf16", "mode": "train, eager, FlatAdamax",
            "card": card_info(), "clocks": clk, "preheat_s": args.preheat, "iters": args.iters, "reps": args.reps,
            "settings": res}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
