"""Class weights for `sr.py --class_weights FILE` from a training json.

    python tools/make_class_weights.py --train_json imSitu/train.json --out weights.pt [--power 0.5]

A class seen k times in the training json gets the weight k^-power; the weights are then normalised to mean 1 over the
classes that were seen.  A class never seen as a target gets weight 1 (it only enters the label-smoothing term).  The
counts go through the encoder's `encode`, i.e. the verb and label ids the loader feeds to the losses: the verbs once
per image, the labels once per (annotation, role) target, the padding slots (ignore_index) not at all.  The encoder is
built from `--encoder_json` (default: the training json), as sr.py builds it from train.json.

The output is a torch.save'd dict {"verb": fp32 [n_verbs], "nouns": fp32 [n_labels]}.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from situation_recognition_b200.imsitu_encoder import imsitu_encoder  # noqa: E402


def class_counts(train_json, encoder):
    """(verb counts [n_verbs], label counts [n_labels]) as int64, counted through encoder.encode."""
    V, L = encoder.get_num_verbs(), encoder.get_num_labels()
    verbs = torch.zeros(V, dtype=torch.int64)
    labels = torch.zeros(L + 1, dtype=torch.int64)       # the last bin collects the padding slots
    for item in train_json.values():
        verb, lab = encoder.encode(item)
        verbs[verb] += 1
        labels += torch.bincount(torch.as_tensor(lab).reshape(-1), minlength=L + 1)
    return verbs, labels[:L]


def weights_from_counts(counts, power):
    """counts^-power on the seen classes, normalised to mean 1 there; 1 on the unseen ones."""
    seen = counts > 0
    w = torch.ones(counts.shape, dtype=torch.float64)
    if seen.any():
        ws = counts[seen].double() ** (-power)
        w[seen] = ws / ws.mean()
    return w.float()


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--train_json", required=True, help="training annotations whose class frequencies are counted")
    ap.add_argument("--encoder_json", default="", help="json the encoder is built from (default: --train_json)")
    ap.add_argument("--power", type=float, default=0.5, help="weight = frequency^-power (0: all ones)")
    ap.add_argument("--out", required=True, help="output file for sr.py --class_weights")
    args = ap.parse_args(argv)
    if args.power < 0:
        ap.error("--power must be >= 0")
    with open(args.train_json) as f:
        train = json.load(f)
    enc_src = train
    if args.encoder_json:
        with open(args.encoder_json) as f:
            enc_src = json.load(f)
    encoder = imsitu_encoder(enc_src, verbose=False)
    verbs, labels = class_counts(train, encoder)
    out = {"verb": weights_from_counts(verbs, args.power), "nouns": weights_from_counts(labels, args.power)}
    torch.save(out, args.out)
    print("wrote %s: %d verbs (%d seen), %d labels (%d seen), power %g" %
          (args.out, verbs.numel(), int((verbs > 0).sum()), labels.numel(), int((labels > 0).sum()), args.power))


if __name__ == "__main__":
    main()
