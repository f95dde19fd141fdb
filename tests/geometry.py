"""Vocabularies of any shape the library accepts: max role count R in [1, 8] (and beyond, for the refusal), any numbers
of verbs, roles and labels, for the geometry tests (tests/test_geometry.py on the CPU, tests/test_geometry_gpu.py on a
B200).  synthetic.make_train_json fixes imSitu's shape (504 / 190 / 2001, R = 6, no verb without roles); the kernels
whose shapes depend on R, on the hidden size D or on the vocabulary sizes need the others.

Plain helper module (no tests).
"""
import numpy as np
import torch

import situation_recognition_b200 as S
from situation_recognition_b200 import synthetic


def role_counts(R, n_verbs, seed):
    """Roles per verb: every count 0..R at least once (so the histogram reaches R exactly and has 0-role verbs), the
    rest drawn from 1..R, shuffled."""
    if n_verbs < R + 1:
        raise ValueError("%d verbs cannot hold every role count 0..%d" % (n_verbs, R))
    rng = np.random.RandomState(seed)
    counts = np.concatenate([np.arange(R + 1), rng.randint(1, R + 1, size=n_verbs - R - 1)])
    rng.shuffle(counts)
    return counts


def make_geometry(R, n_verbs, n_roles, n_labels, seed=0):
    """(imSitu-format training json, its imsitu_encoder) with max role count R, exactly n_verbs verbs, n_roles roles and
    n_labels labels.  Every count 0..R occurs (role_counts); a 0-role verb's frames are empty.  Roles are dealt
    round-robin so that each one is used, labels in order until each one is used, then at random."""
    counts = role_counts(R, n_verbs, seed)
    if n_roles < R or counts.sum() < n_roles:
        raise ValueError("%d roles do not fit role counts up to %d summing to %d" % (n_roles, R, counts.sum()))
    rng = np.random.RandomState(seed + 1)
    role_names = ["role%03d" % i for i in range(n_roles)]
    labels = ["n%05d" % i for i in range(n_labels)]
    cursor = 0
    verb_roles = []
    for n in counts:
        roles = []
        while len(roles) < n:
            cand = role_names[cursor] if cursor < n_roles else role_names[rng.randint(n_roles)]
            cursor += 1
            if cand not in roles:
                roles.append(cand)
        verb_roles.append(roles)
    # enough images per verb that the frames' slots hold every label at least once
    images = max(1, -(-n_labels // (3 * int(counts.sum()))))
    train, label_cursor = {}, 0
    for vi, roles in enumerate(verb_roles):
        for k in range(images):
            frames = []
            for _ in range(3):
                frame = {}
                for r in roles:
                    if label_cursor < n_labels:
                        frame[r] = labels[label_cursor]
                        label_cursor += 1
                    else:
                        frame[r] = labels[rng.randint(n_labels)]
                frames.append(frame)
            train["verb%03d_%d.jpg" % (vi, k)] = {"verb": "verb%03d" % vi, "frames": frames}
    return train, S.imsitu_encoder(train, verbose=False)


def verb_counts(enc):
    return np.array([enc.get_role_count(v) for v in range(enc.get_num_verbs())])


def verbs_with_count(enc, n):
    return [v for v, c in enumerate(verb_counts(enc)) if c == n]


def compact_rows(counts):
    """(first row of each image, rows incl. the shared pad row) of the compact role-node layout (k_prep_rows): image b
    owns rows [off[b], off[b] + n_b), the shared pad row follows the last image."""
    off = np.concatenate([[0], np.cumsum(counts)])
    return off[:-1], int(off[-1]) + 1


def straddles(counts, tile=256):
    """Images whose compact rows lie on both sides of a multiple of `tile`."""
    off, _ = compact_rows(counts)
    return [b for b, (o, n) in enumerate(zip(off, counts)) if n and o // tile != (o + n - 1) // tile]


def crossing_verbs(enc, tile=256):
    """gt verbs of the smallest batch that starts with one verb of every role count 0..R and then repeats verbs with R
    roles until an image's compact rows straddle a `tile`-row boundary.  At R = 1 no image owns two rows: the batch then
    ends where its row count (shared pad row included) first exceeds `tile`."""
    R = enc.get_max_role_count()
    by_count = {n: verbs_with_count(enc, n) for n in range(R + 1)}
    verbs = [by_count[n][0] for n in range(R + 1)]
    k = 0
    while True:
        counts = verb_counts(enc)[verbs]
        if (R > 1 and straddles(counts, tile)) or (R == 1 and compact_rows(counts)[1] > tile):
            return torch.tensor(verbs, dtype=torch.int64)
        full = by_count[R]
        verbs.append(full[k % len(full)])
        k += 1


def make_batch(enc, B, D, seed, gt_verb=None):
    """synthetic.make_batch's features and targets, with the gt verbs given (their noun targets re-derived: random
    labels on the real slots, the ignore label n_labels on the pad slots)."""
    fv, fn, gv, gn = synthetic.make_batch(enc, B, D, seed=seed)
    if gt_verb is None:
        return fv, fn, gv, gn
    L, R = enc.get_num_labels(), enc.get_max_role_count()
    counts = torch.from_numpy(verb_counts(enc))[gt_verb]
    pad = (torch.arange(R)[None, None, :] >= counts[:, None, None]).expand(B, 3, R)
    lab = torch.randint(0, L, (B, 3, R), generator=torch.Generator().manual_seed(seed + 1))
    return fv, fn, gt_verb.clone(), torch.where(pad, torch.full_like(lab, L), lab)
