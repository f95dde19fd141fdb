"""`sr.py`-compatible launcher on the B200-native GGNN stage.

Same command line as the reference's `sr.py` (sr.py:384-420) and the same five modes -- train, --evaluate_dev,
--evaluate_test, --test_img [--verb], --subset N -- with the same console output and the same checkpoint dict
(`epoch`, six history lists, `model_state_dict`, `optimizer_state_dict`; sr.py:145-162), so checkpoints move both
ways.  Differences, all forced by the B200-first design:
  * one process per GPU (`torchrun --nproc-per-node G -m situation_recognition_b200.sr ...`) instead of
    `nn.DataParallel`; `--batch_size` stays the GLOBAL batch and is split contiguously over the ranks;
  * no `GradScaler`/autocast: the stage computes in bf16 with fp32 accumulation and needs no loss scaling;
  * the scorer is the vectorised one (identical numbers); rank 0 prints and writes checkpoints;
  * clip_grad_norm_ + Adamax (sr.py:80-83) run as the fused `parallel.FlatAdamax` step over flat parameter / gradient
    buffers, sharded over the ranks (reduce-scatter, 1/N update, all-gather); its `state_dict()` has torch.optim.Adamax's
    format, so checkpoints load into the reference's optimizer and vice versa;
  * the features of the frozen backbones on the dev / test images are cached across epochs (`features.FeatureCache`):
    the per-epoch validation (sr.py:123) runs the backbones once, not once per epoch;
  * `--no_pretrained` (extra flag) skips the ImageNet weights when there is no network; `--no_feature_cache` disables
    the cache;
  * `--topk_situations K` (extra flag, default 0 = off) adds the standard imSitu top-k situation metrics
    (`situations.SituationScorer`) to --evaluate_dev / --evaluate_test, and K situations per image to --test_img;
  * `--finetune_backbone` (extra flag) trains both ResNet-152 backbones with the GGNN stage (bf16 only; the dev
    feature cache is off, and a checkpoint resumes only under the setting it was trained with).
"""
import os
from argparse import ArgumentParser
from json import load as jload
from os.path import isfile as pisfile, join as pjoin
from pathlib import Path
from random import randrange

import torch
import torch.distributed as dist

from . import parallel
from .features import FeatureCache
from .imsitu_encoder import imsitu_encoder
from .imsitu_loader import ShardedBatchSampler, imsitu_loader
from .imsitu_scorer import imsitu_scorer
from .model import FCGGNN
from .situations import SituationScorer
from .utils import format_dict, load_net


def _rank_world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def _print0(*a, **k):
    if _rank_world()[0] == 0:
        print(*a, **k)


def _all_sum(t):
    if _rank_world()[1] > 1:
        dist.all_reduce(t)
    return t


def _merge_scorer(s):
    """Sum the per-rank score cards so every rank reports the global averages."""
    if _rank_world()[1] > 1 and s._sums is not None:
        packed = torch.cat([s._sums, torch.tensor([float(s._count)], dtype=s._sums.dtype, device=s._sums.device)])
        dist.all_reduce(packed)
        s._sums, s._count = packed[:-1], int(packed[-1].item())
    return s


def _avg_score(top1_a, top5_a):
    score = top1_a['verb'] + top1_a['value'] + top1_a['value-all'] + top5_a['verb'] + top5_a['value'] + \
        top5_a['value-all'] + top1_a['gt-value'] + top1_a['gt-value-all']
    return score / 8 * 100


def _print_scores(prefix, losses, top1_a, top5_a, avg_score, tail):
    _print0(prefix.format(*losses))
    gt = {key: top1_a[key] for key in ['gt-value', 'gt-value-all']}
    one_val = {key: top1_a[key] for key in ['verb', 'value', 'value-all']}
    _print0('{}\n{}\n{}, mean = {:.2f}\n{}'.format(format_dict(one_val, '{:.2f}', '1-'), format_dict(top5_a, '{:.2f}', '5-'),
                                                   format_dict(gt, '{:.2f}', ''), avg_score, tail))


def _global_sizes(loader):
    sampler = getattr(loader, "batch_sampler", None)
    return sampler.global_sizes() if hasattr(sampler, "global_sizes") else None


def train(model, train_loader, dev_loader, optimizer, max_epoch, encoder, model_saving_name, folder, checkpoint=None,
          flat=None, plot=True, dev_cache=None):
    """sr.py:15-162."""
    model.train()
    hist = {k: [] for k in ('avg_scores', 'verb_losses', 'nouns_losses', 'val_avg_scores', 'val_verb_losses',
                            'val_nouns_losses')}
    epoch = 0
    if checkpoint is not None:
        epoch = checkpoint['epoch']
        for k in hist:
            hist[k] = checkpoint[k]
        model.load_state_dict(checkpoint['model_state_dict'])
        saved = sum(len(g['params']) for g in checkpoint['optimizer_state_dict']['param_groups'])
        now = sum(len(g['params']) for g in optimizer.param_groups)
        if saved != now:
            raise SystemExit("cannot resume: the checkpoint's optimizer state covers %d trainable tensors, this run trains "
                             "%d -- resume with the same --finetune_backbone setting the checkpoint was trained with"
                             % (saved, now))
        optimizer.load_state_dict(checkpoint['optimizer_state_dict'])
    if flat is None:
        flat = parallel.attach(model)
    params = [p for p in model.parameters() if p.requires_grad]
    dev = next(model.parameters()).device
    fused = getattr(optimizer, "fused_clip", False)          # parallel.FlatAdamax: clip (+ gradient exchange) inside step()
    sharded = getattr(optimizer, "world", 1) > 1

    for e in range(epoch, max_epoch):
        sums = torch.zeros(3, device=dev)
        _print0('Epoch-{}, lr: {:.4f}'.format(e, optimizer.param_groups[0]['lr']))
        top1, top5 = imsitu_scorer(encoder, 1, 3), imsitu_scorer(encoder, 5, 3)
        if hasattr(train_loader.batch_sampler, 'set_epoch'):
            train_loader.batch_sampler.set_epoch(e)
        sizes = _global_sizes(train_loader)
        for step, (_, img, verb, nouns) in enumerate(train_loader):
            img, verb, nouns = img.to(dev, non_blocking=True), verb.to(dev), nouns.to(dev)
            model.global_batch = sizes[step] if sizes is not None else None
            flat.zero()
            pred_verb, pred_nouns, pred_gt_nouns = model(img, verb)
            verb_loss = model.verb_loss(pred_verb, verb)
            nouns_loss = model.nouns_loss(pred_nouns, nouns)
            gt_nouns_loss = model.nouns_loss(pred_gt_nouns, nouns)
            (verb_loss + nouns_loss).backward()
            if not sharded:
                flat.all_reduce()
            if not fused:
                torch.nn.utils.clip_grad_norm_(params, 1)
            optimizer.step()
            top1.add_point_both(pred_verb, verb, pred_nouns, nouns, pred_gt_nouns)
            top5.add_point_both(pred_verb, verb, pred_nouns, nouns, pred_gt_nouns)
            sums += torch.stack([verb_loss.detach(), nouns_loss.detach(), gt_nouns_loss.detach()])
        # per-rank losses are partial sums of the global-batch means (model.loss_group): add them up
        means = (_all_sum(sums) / len(train_loader)).tolist()
        top1_a, top5_a = _merge_scorer(top1).get_average_results_both(), _merge_scorer(top5).get_average_results_both()
        avg_score = _avg_score(top1_a, top5_a)
        hist['avg_scores'].append(avg_score)
        hist['verb_losses'].append(means[0])
        hist['nouns_losses'].append(means[1])
        _print_scores('training losses = [v: {:.2f}, n: {:.2f}, gt: {:.2f}]', means, top1_a, top5_a, avg_score, '-' * 50)

        top1, top5, val_losses, val_avg_score = eval(model, dev_loader, encoder, logging=True, cache=dev_cache)
        model.train()
        hist['val_avg_scores'].append(val_avg_score)
        hist['val_verb_losses'].append(val_losses['verb_loss'])
        hist['val_nouns_losses'].append(val_losses['nouns_loss'])

        opt_state = optimizer.state_dict()          # a collective when the optimizer state is sharded: every rank calls it
        if _rank_world()[0] == 0:
            if plot:
                _plot(hist, pjoin(folder, model_saving_name + '.png'))
            ckpt = {'epoch': e + 1, **hist, 'model_state_dict': model.state_dict(),
                    'optimizer_state_dict': opt_state}
            torch.save(ckpt, pjoin(folder, model_saving_name))


def _plot(hist, path):
    try:
        import matplotlib
        matplotlib.use('Agg')
        import matplotlib.pyplot as plt
    except Exception:
        return
    plt.plot(hist['verb_losses'], label='verb losses')
    plt.plot(hist['nouns_losses'], label='nouns losses')
    plt.plot(hist['avg_scores'], label='accuracy mean')
    plt.plot(hist['val_verb_losses'], '-.', label='val verb losses')
    plt.plot(hist['val_nouns_losses'], '-.', label='val nouns losses')
    plt.plot(hist['val_avg_scores'], '-.', label='val accuracy mean')
    plt.grid()
    plt.legend()
    plt.savefig(path)
    plt.clf()


def eval(model, loader, encoder, logging=False, cache=None, topk_situations=0):
    """sr.py:165-232.  cache (FeatureCache, optional): the frozen backbones' features of this loader's images are kept
    across calls; once every image is cached the loader stops decoding images altogether.
    topk_situations K > 0: also decode the top-K situations of every image (and the gt-verb situation) from the same
    backbone features and print the standard imSitu top-1 / top-K metrics after the existing lines."""
    model.eval()
    dev = next(model.parameters()).device
    sums = torch.zeros(3, device=dev)
    top1, top5 = imsitu_scorer(encoder, 1, 3), imsitu_scorer(encoder, 5, 3)
    sit = SituationScorer(encoder, (1, topk_situations)) if topk_situations > 0 else None
    dataset = getattr(loader, "dataset", None)
    if cache is not None and dataset is not None and hasattr(dataset, "skip_images"):
        dataset.skip_images = cache.has(dataset.imgs_names)       # read by the workers this iteration starts
    sizes = _global_sizes(loader)
    with torch.no_grad():
        for step, (names, img, verb, nouns) in enumerate(loader):
            verb, nouns = verb.to(dev), nouns.to(dev)
            model.global_batch = sizes[step] if sizes is not None else None
            if cache is not None:
                fv, fn = cache.features(model, list(names), img.to(dev, non_blocking=True) if img.numel() else None)
                pred_verb, pred_nouns, pred_gt_nouns = model.forward_features(fv, fn, verb)
            elif sit is not None:      # the backbones run once for both decodes
                fv, fn = model.extract_features(img.to(dev, non_blocking=True))
                pred_verb, pred_nouns, pred_gt_nouns = model.forward_features(fv, fn, verb)
            else:
                pred_verb, pred_nouns, pred_gt_nouns = model(img.to(dev, non_blocking=True), verb)
            if sit is not None:
                sit.add_point(model.situations_from_features(fv, fn, k=topk_situations), verb, nouns,
                              model.situations_from_features(None, fn, verbs=verb[:, None]))
            top1.add_point_both(pred_verb, verb, pred_nouns, nouns, pred_gt_nouns)
            top5.add_point_both(pred_verb, verb, pred_nouns, nouns, pred_gt_nouns)
            sums += torch.stack([model.verb_loss(pred_verb, verb), model.nouns_loss(pred_nouns, nouns),
                                 model.nouns_loss(pred_gt_nouns, nouns)])
    if dataset is not None and hasattr(dataset, "skip_images"):
        dataset.skip_images = False
    v, n, g = (_all_sum(sums) / len(loader)).tolist()
    val_losses = {'verb_loss': v, 'nouns_loss': n, 'gt_loss': g}
    avg_score = 0
    _merge_scorer(top1)
    _merge_scorer(top5)
    if logging is True:
        top1_a, top5_a = top1.get_average_results_both(), top5.get_average_results_both()
        avg_score = _avg_score(top1_a, top5_a)
        _print_scores('val losses = [v: {:.2f}, n: {:.2f}, gt: {:.2f}]', (v, n, g), top1_a, top5_a, avg_score, '')
    if sit is not None:
        _print_situation_scores(_merge_scorer(sit))
    return top1, top5, val_losses, avg_score


def _print_situation_scores(sit):
    """The standard imSitu block: top-1 / top-K verb, value, value-all, then gt-value, gt-value-all and the mean."""
    a = {key: 100 * x for key, x in sit.get_average_results().items()}
    _print0('top-k situations (imSitu definitions):')
    for k in sit.ks:
        _print0('top-{}: verb: {:.2f}, value: {:.2f}, value-all: {:.2f}'.format(
            k, a['verb@%d' % k], a['value@%d' % k], a['value-all@%d' % k]))
    _print0('gt-value: {:.2f}, gt-value-all: {:.2f}, mean = {:.2f}'.format(a['gt-value'], a['gt-value-all'], a['mean']))


def _spaces(dataset_folder):
    with open(pjoin(dataset_folder, 'imsitu_space.json'), 'r') as f:
        space = jload(f)
    return space["nouns"], space["verbs"]


def _gloss(encoder, nouns_space, idx):
    label = encoder.label_list[idx]
    return '-' if label in ('', 'UNK') else nouns_space[label]['gloss'][0]


def _predict_one(model, img, encoder, verb_tensor=None):
    """predict_verb -> argmax -> predict_nouns on a batch of one (sr.py:255-268, 316-327); keeps the reference's
    softmax over dim 0 (roles) for the reported label probabilities."""
    dev = next(model.parameters()).device
    img = img.to(dev)
    verb_prob = 100
    if verb_tensor is None:
        logits = model.predict_verb(img, 1)
        verb_tensor = torch.argmax(logits, 1)
        verb_prob = torch.max(torch.nn.functional.softmax(logits, dim=1)).item() * 100
    logits = model.predict_nouns(img, verb_tensor.to(dev), 1).squeeze(0)
    nouns_tensor = torch.argmax(logits, 1)
    probabilities = torch.max(torch.nn.functional.softmax(logits, dim=0), 1)
    return verb_tensor, verb_prob, nouns_tensor, [p.item() * 100 for p in probabilities[0]]


def results(model, image, encoder, gt_verb, dataset_folder="imSitu"):
    """sr.py:235-281."""
    from PIL import Image
    model.eval()
    nouns_space, verbs_space = _spaces(dataset_folder)
    img = encoder.dev_transform(Image.open(image).convert('RGB')).unsqueeze(0)
    verb_tensor = None
    if gt_verb and encoder.verb_list.count(gt_verb):
        verb_tensor = torch.tensor([encoder.verb_list.index(gt_verb)])
    else:
        print("No ground truth verb found, calculating by myself...")
    with torch.no_grad():
        verb_tensor, verb_prob, nouns_tensor, labels_prob = _predict_one(model, img, encoder, verb_tensor)
    verb_name = encoder.verb_list[int(verb_tensor)]
    roles = list(verbs_space[verb_name]["roles"].keys())
    labels = {roles[c]: _gloss(encoder, nouns_space, int(i)) for c, i in enumerate(nouns_tensor[:len(roles)])}
    return verb_name, verb_prob, labels, labels_prob


def results_topk(model, image, encoder, k, gt_verb="", dataset_folder="imSitu"):
    """The k best situations of one image: [(verb, verb probability % or None, score, {role: (gloss, label
    probability %)})].  With a known `gt_verb` only that verb's situation.  Probabilities are softmaxes over the
    verbs / over the labels."""
    from PIL import Image
    model.eval()
    dev = next(model.parameters()).device
    nouns_space, verbs_space = _spaces(dataset_folder)
    img = encoder.dev_transform(Image.open(image).convert('RGB')).unsqueeze(0).to(dev)
    fv, fn = model.extract_features(img)
    if gt_verb and encoder.verb_list.count(gt_verb):
        s = model.situations_from_features(fv, fn, verbs=torch.tensor([[encoder.verb_list.index(gt_verb)]], device=dev))
    else:
        s = model.situations_from_features(fv, fn, k=k)
    verbs, labels, label_logp, score = s.verbs[0].tolist(), s.labels[0].tolist(), s.label_logp[0].exp().tolist(), \
        s.score[0].tolist()
    verb_p = s.verb_logp[0].exp().tolist() if s.verb_logp is not None else [None] * len(verbs)
    out = []
    for j, v in enumerate(verbs):
        name = encoder.verb_list[v]
        roles = list(verbs_space[name]["roles"].keys())
        out.append((name, None if verb_p[j] is None else 100 * verb_p[j], score[j],
                    {roles[r]: (_gloss(encoder, nouns_space, labels[j][r]), 100 * label_logp[j][r])
                     for r in range(len(roles))}))
    return out


def _print_situations(sits):
    for j, (verb, verb_p, score, roles) in enumerate(sits):
        vp = 'given' if verb_p is None else '{:.2f}%'.format(verb_p)
        print('situation {} ({}): {}, log-score = {:.4f}'.format(j + 1, vp, verb, score))
        for role, (gloss, p) in roles.items():
            print('  {} ({:.2f}%): {}'.format(role, p, gloss))


def analize_subset(model, dev_set, encoder, size, dataset_folder="imSitu", imgset_dir="resized_256"):
    """sr.py:284-380."""
    model.eval()
    nouns_space, verbs_space = _spaces(dataset_folder)
    subset = torch.utils.data.Subset(dev_set, [randrange(0, len(dev_set)) for _ in range(size)])
    batch = next(iter(torch.utils.data.DataLoader(subset, batch_size=size, num_workers=0, shuffle=False)))
    imgs_name, imgs, gt_verbs, gt_nouns = batch
    num_labels = encoder.get_num_labels()
    for el in range(size):
        with torch.no_grad():
            verb_tensor, verb_prob, labels_tensor, labels_prob = _predict_one(model, imgs[el].unsqueeze(0), encoder)
        verb_name = encoder.verb_list[int(verb_tensor)]
        gt_verb_name = encoder.verb_list[int(gt_verbs[el])]
        roles = list(verbs_space[verb_name]["roles"].keys())
        labels = {roles[c]: _gloss(encoder, nouns_space, int(i)) for c, i in enumerate(labels_tensor[:len(roles)])}
        gt_roles = list(verbs_space[gt_verb_name]["roles"].keys())
        gt_labels = {}
        for c, row in enumerate(gt_nouns[el].transpose(0, 1)[:len(gt_roles)]):
            gt_labels[gt_roles[c]] = tuple('-' if int(i) == num_labels else _gloss(encoder, nouns_space, int(i))
                                           for i in row[:3])
        print('&' * 35)
        print('Analizing: ', imgs_name[el])
        _display(pjoin(imgset_dir, imgs_name[el]))
        print('action ({:.2f}%): {}'.format(verb_prob, verb_name))
        for c, (k, v) in enumerate(labels.items()):
            print('{} ({:.2f}%): {}'.format(k, labels_prob[c], v))
        print('---- Ground truth ----')
        print('action: {}'.format(gt_verb_name))
        for k, v in gt_labels.items():
            print('{} = [{}, {}, {}]'.format(k, v[0], v[1], v[2]))


def _display(path):
    try:
        from IPython.display import display
        from PIL import Image
        display(Image.open(path, 'r'))
    except Exception:
        pass


# (flag, type, default, help) -- the reference's command line (sr.py:384-420), flag for flag
_STR_FLAGS = [("resume_model", "", "checkpoint to resume from / evaluate"),
              ("test_img", "", "run the single-image mode on this file"),
              ("verb", "", "ground-truth verb for --test_img"),
              ("model_saving_name", "sr", "file name of the checkpoint"),
              ("saving_folder", "checkpoints", "where checkpoints and the cached encoder live"),
              ("imgset_dir", "resized_256", "directory of the images"),
              ("dataset_folder", "imSitu", "directory of the annotation json files"),
              ("train_file", "train.json", "training annotations"),
              ("dev_file", "dev.json", "dev annotations"),
              ("test_file", "test.json", "test annotations")]
_NUM_FLAGS = [("subset", int, 0, "analyse a random dev subset of this size"),
              ("batch_size", int, 6144, "GLOBAL batch size (split over the ranks)"),
              ("num_workers", int, 10, "DataLoader workers"),
              ("epochs", int, 1000, "training epochs"),
              ("lr", float, 0.002, "Adamax learning rate")]


def build_parser():
    parser = ArgumentParser(description="Situation recognition with GNN (B200-native GGNN stage).")
    for name, default, text in _STR_FLAGS:
        parser.add_argument("--" + name, type=str, default=default, help=text)
    for name, kind, default, text in _NUM_FLAGS:
        parser.add_argument("--" + name, type=kind, default=default, help=text)
    for name in ("evaluate_dev", "evaluate_test"):
        parser.add_argument("--" + name, action="store_true", help="only evaluate on that split")
    # extensions (not in the reference)
    parser.add_argument("--no_pretrained", action="store_true", help="random-init backbones (no network access)")
    parser.add_argument("--precision", type=str, default="bf16", choices=["bf16", "fp32"])
    parser.add_argument("--no_feature_cache", action="store_true",
                        help="recompute the frozen backbones on the dev set at every epoch, like the reference")
    parser.add_argument("--torch_optimizer", action="store_true",
                        help="torch.optim.Adamax + clip_grad_norm_ + gradient all-reduce instead of the fused sharded step")
    parser.add_argument("--finetune_backbone", action="store_true",
                        help="train both ResNet-152 backbones with the GGNN stage (turns the dev feature cache off)")
    parser.add_argument("--topk_situations", type=int, default=0,
                        help="K > 0: with --evaluate_dev / --evaluate_test also report the standard imSitu top-1 / top-K "
                             "situation metrics (2 <= K <= 16); with --test_img print the K best situations (K <= 16)")
    return parser


def _loader(dataset, batch_size, shuffle, num_workers):
    rank, world = _rank_world()
    sampler = ShardedBatchSampler(len(dataset), batch_size, rank, world, shuffle=shuffle)
    return torch.utils.data.DataLoader(dataset, batch_sampler=sampler, pin_memory=True, num_workers=num_workers)


def main(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    if not 0 <= args.topk_situations <= 16:
        parser.error("--topk_situations must be in [0, 16], got %d" % args.topk_situations)
    if args.topk_situations == 1 and (args.evaluate_dev or args.evaluate_test):
        # the block reports top-1 and top-K and the mean of those 8 numbers; K = 1 would print a different mean
        parser.error("--topk_situations with --evaluate_dev / --evaluate_test needs K >= 2 (top-1 is always reported)")
    if args.finetune_backbone and args.precision == "fp32":
        parser.error("--finetune_backbone needs --precision bf16 (precision fp32 is a forward-only parity mode)")
    if not torch.cuda.is_available():
        raise SystemExit("situation_recognition_b200.sr needs a B200 GPU: the GGNN stage has no CPU path")
    if "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # one process per GPU; SRG_DIST_BACKEND=gloo lets several ranks share one GPU (tests on a single-GPU box: NCCL
        # refuses two ranks on the same device)
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count())
        dist.init_process_group(os.environ.get("SRG_DIST_BACKEND", "nccl"))
    rank, world = _rank_world()
    dev = torch.device("cuda", torch.cuda.current_device())
    Path(args.saving_folder).mkdir(exist_ok=True)
    checkpoint = None

    def load_json(name):
        with open(pjoin(args.dataset_folder, name), 'r') as f:
            return jload(f)

    encoder_json = load_json('train.json')          # the encoder is always built from train.json (sr.py:429-430)
    train_json, dev_json, test_json = load_json(args.train_file), load_json(args.dev_file), load_json(args.test_file)
    enc_path = pjoin(args.saving_folder, 'encoder')
    if not pisfile(enc_path):
        encoder = imsitu_encoder(encoder_json, verbose=(rank == 0))
        if rank == 0:
            torch.save(encoder, enc_path)
    else:
        _print0("Loading encoder file")
        encoder = torch.load(enc_path, weights_only=False)

    train_set = imsitu_loader(args.imgset_dir, train_json, encoder, encoder.train_transform)
    dev_set = imsitu_loader(args.imgset_dir, dev_json, encoder, encoder.dev_transform)
    test_set = imsitu_loader(args.imgset_dir, test_json, encoder, encoder.dev_transform)
    train_loader = _loader(train_set, args.batch_size, True, args.num_workers)
    dev_loader = _loader(dev_set, args.batch_size, False, args.num_workers)
    test_loader = _loader(test_set, args.batch_size, True, args.num_workers)

    seed = os.environ.get("SRG_SEED")            # extension: repeatable initial weights / dropout (tests)
    if seed is not None:
        torch.manual_seed(int(seed))
    model = FCGGNN(encoder, D_hidden_state=2048, precision=args.precision,
                   pretrained=False if args.no_pretrained else None).to(dev)
    if args.finetune_backbone:      # before attach(): the flat buffers and the optimizer cover what requires grad
        model.convnet_verbs.requires_grad_(True)
        model.convnet_nouns.requires_grad_(True)
    parallel.broadcast_model(model)              # every rank built its own random init: rank 0's becomes everyone's
    if seed is not None:
        torch.manual_seed(int(seed) + 1000 * rank)      # per-rank dropout streams from here on
    _print0('Using', world, 'GPUs!')
    if args.torch_optimizer:
        flat = parallel.attach(model)
        optimizer = torch.optim.Adamax(filter(lambda p: p.requires_grad, model.parameters()), lr=args.lr)
    else:   # sr.py:80-83,472-473 as one fused kernel over flat buffers, sharded over the ranks
        flat = parallel.attach(model, flat_params=True)
        optimizer = parallel.FlatAdamax(flat, lr=args.lr, max_norm=1.0, group=dist.group.WORLD if world > 1 else None)
    # the cache holds frozen backbones' features: a fine-tuned backbone changes them at every step
    dev_cache = None if (args.no_feature_cache or args.finetune_backbone) else FeatureCache(len(dev_set), 2048, dev)
    torch.backends.cudnn.benchmark = True

    if len(args.resume_model) > 1:
        _print0('Resume training from: {}'.format(args.resume_model))
        path_to_model = pjoin(args.saving_folder, args.resume_model)
        checkpoint = torch.load(path_to_model, map_location=dev, weights_only=False)
        load_net(path_to_model, [model])
        args.model_saving_name = args.resume_model

    if args.evaluate_dev:
        _print0('=> evaluating model with dev-set...')
        eval(model, dev_loader, encoder, logging=True, topk_situations=args.topk_situations)
    elif args.evaluate_test:
        _print0('=> evaluating model with test-set...')
        eval(model, test_loader, encoder, logging=True, topk_situations=args.topk_situations)
    elif args.test_img:
        verb, verb_prob, labels, labels_prob = results(model, args.test_img, encoder, args.verb, args.dataset_folder)
        print('&' * 50)
        print('Analizing: ', args.test_img)
        _display(args.test_img)
        print('&' * 50)
        print('action ({:.2f}%): {}'.format(verb_prob, verb))
        for c, (k, v) in enumerate(labels.items()):
            print('{} ({:.2f}%): {}'.format(k, labels_prob[c], v))
        if args.topk_situations > 0:
            with torch.no_grad():
                sits = results_topk(model, args.test_img, encoder, args.topk_situations, args.verb, args.dataset_folder)
            print('&' * 50)
            _print_situations(sits)
    elif args.subset > 0:
        analize_subset(model, dev_set, encoder, args.subset, args.dataset_folder, args.imgset_dir)
    else:
        _print0('Model training started!')
        train(model, train_loader, dev_loader, optimizer, args.epochs, encoder, args.model_saving_name,
              folder=args.saving_folder, checkpoint=checkpoint, flat=flat, dev_cache=dev_cache)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
