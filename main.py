# -*- coding: utf-8 -*-
"""Command line of the reference (main.py:10-76), driving the B200 hot path.

Same flags and defaults, same loop over the three (Step, Ne, Nc, Ner, Ncr) presets; every flag
given on the command line overrides ALL presets, as in the reference.  Extra flags: --variant
(1-4 = model_1..model_4, default 2 = the model main.py imports), --root (directory holding
Adjset/ and dataset/), --seed, --no_q2 (feed each batch its own entity->hunk maps instead of the
reference's first-Mini_batch slice, model_2.py:376-381).  Extra value --Type untangle: the hunk groups the trained model
predicts for every test commit (graph2graph.untangle), scored against the labelled groups over each commit's real hunks
(pair precision / recall / F1, Rand and adjusted Rand index, purity).  With --Type untangle, --grouping average forms the
groups by average-linkage clustering of the relation probabilities instead of connected components of the arg-max relations:
two groups merge only while their mean relation probability is > --threshold (default 0.5).  --sweep 0.3,0.4,... (with
--grouping average only) scores those thresholds as well, and the cut at each commit's labelled number of groups, from one
dendrogram per batch, so a threshold can be chosen from the scores; the groups written stay those at --threshold.
Multi-GPU: launch with `python -m torch.distributed.run --nproc-per-node N main.py ...`.
"""
import argparse
import os

import torch


def _thresholds(text):
    """'0.3,0.4' -> [0.3, 0.4]: 1 to 63 thresholds, none NaN (one hdgnn_linkage_cut call takes --threshold and 63 more)."""
    try:
        ts = [float(t) for t in text.split(',')]
    except ValueError:
        raise argparse.ArgumentTypeError(f'not a comma-separated list of numbers: {text!r}')
    if not 1 <= len(ts) <= 63 or any(t != t for t in ts):
        raise argparse.ArgumentTypeError(f'1 to 63 thresholds, none NaN: {text!r}')
    return ts


def main(argv=None):
    steps = [2, 3, 5]
    entity_nodes = [200, 250, 250]
    hunk_nodes = [74, 114, 150]
    entity_edges = [39800, 62250, 62250]
    hunk_edges = [5402, 12882, 22350]
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not torch.distributed.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        torch.distributed.init_process_group("nccl")
    from hdgnn_b200.model import graph2graph

    results = []
    for step, entity_node, hunk_node, entity_edge, hunk_edge in zip(steps, entity_nodes, hunk_nodes, entity_edges, hunk_edges):
        print(step, entity_node, hunk_node, entity_edge, hunk_edge)
        parser = argparse.ArgumentParser(description='')
        parser.add_argument('--epoch', type=int, default=50, help='number of training epochs')
        parser.add_argument('--Ds', type=int, default=1, help='The State Dimention')
        parser.add_argument('--Ds_inter', type=int, default=1, help='The State Dimention of inter state')
        parser.add_argument('--Dr', type=int, default=2, help='The Relationship Dimension')
        parser.add_argument('--Dr_inter', type=int, default=2, help='The Relationship Dimension of inter state')
        parser.add_argument('--De_e', type=int, default=20, help='The Effect Dimension on entity')
        parser.add_argument('--De_er', type=int, default=20, help='The Effect Dimension on entity Relations')
        parser.add_argument('--Mini_batch', type=int, default=50, help='The training mini_batch')
        parser.add_argument('--checkpoint_dir', dest='checkpoint_dir', default='./checkpoint40/', help='models are saved here')
        parser.add_argument('--Ne', type=int, default=entity_node, help='The Number of entities')
        parser.add_argument('--Nc', type=int, default=hunk_node, help='The Number of code changes')
        parser.add_argument('--Ner', type=int, default=entity_edge, help='The Number of entity Relations')
        parser.add_argument('--Ncr', type=int, default=hunk_edge, help='The Number of code change Relations')
        parser.add_argument('--Step', type=int, default=step, help='the number of commits/groups')
        parser.add_argument('--Repo', type=str, default='glide', help='the name of repository')
        parser.add_argument('--Type', dest='Type', default='train', help='train or test')
        # additions (no reference flag renamed or removed)
        parser.add_argument('--variant', type=int, default=2, help='1..4 = model_1..model_4 (reference imports model_2)')
        parser.add_argument('--root', type=str, default='.', help='directory holding Adjset/ and dataset/')
        parser.add_argument('--seed', type=int, default=None, help='weight-init seed (the reference is unseeded)')
        parser.add_argument('--no_q2', action='store_true', help='per-batch entity->hunk maps (fixes model_2.py:376-381)')
        parser.add_argument('--grouping', choices=['components', 'average'], default='components',
                            help='untangle: hunk groups as connected components of the arg-max relations, or by average '
                                 'linkage of the relation probabilities')
        parser.add_argument('--threshold', type=float, default=0.5,
                            help='untangle --grouping average: merge two groups while their mean relation probability is above it')
        parser.add_argument('--sweep', type=_thresholds, default=None,
                            help='untangle --grouping average: comma-separated thresholds to score beside --threshold')
        args = parser.parse_args(argv)
        if args.sweep is not None and (args.Type != 'untangle' or args.grouping != 'average'):
            parser.error('--sweep needs --Type untangle --grouping average')

        ck = args.checkpoint_dir if os.path.isabs(args.checkpoint_dir) else os.path.join(args.root, args.checkpoint_dir)
        if not os.path.exists(ck):
            os.makedirs(ck, exist_ok=True)
        model = graph2graph(None,
                            Ds=args.Ds,
                            Ne=args.Ne, Nc=args.Nc,
                            Ner=args.Ner, Ncr=args.Ncr,
                            Dr=args.Dr,
                            De_e=args.De_e, De_er=args.De_er,
                            Mini_batch=args.Mini_batch,
                            checkpoint_dir=args.checkpoint_dir,
                            epoch=args.epoch,
                            Ds_inter=args.Ds_inter, Dr_inter=args.Dr_inter,
                            Step=args.Step,
                            Repo=args.Repo,
                            variant=args.variant, seed=args.seed)
        if args.Type == 'train':
            results.append(model.train(args, root=args.root, quirk_q2=not args.no_q2))
        if args.Type == 'test':
            results.append(model.test(args, root=args.root, quirk_q2=not args.no_q2))
        if args.Type == 'untangle':
            results.append(model.untangle(args, root=args.root, quirk_q2=not args.no_q2, grouping=args.grouping,
                                          threshold=args.threshold, sweep=args.sweep))
        model.engine.close()
    return results


if __name__ == '__main__':
    main()
