"""The ``--tables`` sweeps of the three CLIs (mr_gan.py:236-341, mr_nn.py:121-168, mr_svm.py:118-165): the
fold-training jobs of every table, the arguments the CLIs share and one driver that runs a CLI's tables and prints them in
the reference's layout.  Tables 2 and 4 are defined once, so the NN and SVM columns of a table train on the same jobs."""
import argparse
import sys

import numpy as np
from sklearn.model_selection import StratifiedKFold

from . import checkpoint, results, sweep, synthetic

MODALITIES = ['Force', 'Temperature', 'Force and Temperature', 'Contact mic', 'Temperature and Contact Mic',
              'Force, Temperature, and Contact Mic', 'Force and Contact Mic']      # mr_gan.py:237
LABELED = [1, 2, 4, 8, 16, 50, 100]                 # labeled % of tables 1 and 2 (mr_gan.py:246)
LOO_LABELED = [1, 4, 16, 50, 100]                   # labeled % of tables 3 and 4 (mr_gan.py:269)


def kfold_jobs(X, y, seed, **kw):
    """mr_gan.py:255-257 as index jobs: the split is expressed as row indices into the shared X."""
    skf = StratifiedKFold(n_splits=6, shuffle=True, random_state=seed)            # mr_gan.py:255
    return [dict(X=X, y=y, train_idx=tr, test_idx=te, **kw) for tr, te in skf.split(X, y)]


def stack_objects(objects):
    """Leave-one-object-out data as one matrix + per-object row ranges (mr_gan.py:274-278 concatenates per fold)."""
    names = list(objects)
    X = np.concatenate([np.asarray(objects[n]['x']) for n in names])
    y = np.concatenate([np.asarray(objects[n]['y']) for n in names])
    ends = np.cumsum([len(objects[n]['y']) for n in names])
    return X, y, {n: (e - len(objects[n]['y']), e) for n, e in zip(names, ends)}


def loo_jobs(objects, **kw):
    """mr_gan.py:274-279: one job per held-out object."""
    X, y, spans = stack_objects(objects)
    rows = np.arange(len(y))
    jobs = []
    for name, (a, b) in spans.items():
        jobs.append(dict(X=X, y=y, train_idx=np.concatenate([rows[:a], rows[b:]]), test_idx=rows[a:b], name=name, **kw))
    return jobs


def job_rows(j):
    """(n_train, n_test) of a job in either format."""
    if 'train_idx' in j:
        return len(j['train_idx']), len(j['test_idx'])
    return len(j['trainTestSets'][0]), len(j['trainTestSets'][1])


def job_width(j):
    return j['X'].shape[1] if 'train_idx' in j else j['trainTestSets'][0].shape[1]


def argument_parser(description, group, nets=True):
    """The arguments of every CLI; nets: the GAN and NN CLIs' --epochs, --precision and --saliency."""
    parser = argparse.ArgumentParser(description=description)
    parser.add_argument('-t', '--tables', nargs='+', help='[Required] Tables to recompute', required=True)
    parser.add_argument('-v', '--verbose', help='Verbose', action='store_true')
    # additive flags (defaults reproduce the reference's behaviour)
    parser.add_argument('--seed', type=int, default=None, help='seed for splits, initial weights, permutations and noise')
    if nets:
        parser.add_argument('--epochs', type=int, default=100)
        parser.add_argument('--precision', choices=['fp32', 'tf32', 'f16'], default='f16',
                            help='arithmetic of the dense layers: f16 = fp16 operand copies, fp32 accumulation and master weights '
                                 '(default; per-step losses within 1e-3 of the oracle, 43 k step-pairs/s per B200); tf32; '
                                 'fp32 = FFMA parity mode (1e-7, 9.8 k)')
    parser.add_argument('--group', type=int, default=group,
                        help='largest number of folds trained side by side per handle (results do not depend on it)')
    parser.add_argument('--data-dir', default='data_processed')
    parser.add_argument('--synthetic', action='store_true', help='synthetic data of the MREO shape instead of the processed pickles')
    results.add_arguments(parser, saliency=nets)
    if nets:
        parser.add_argument('--checkpoint', metavar='DIR', default=None,
                            help='write each fold-training\'s final state to DIR/<tool>_job<id>.npz; on a rerun, take finished '
                                 'jobs from their files and resume unfinished ones (a file of another run is an error)')
        parser.add_argument('--checkpoint-every', metavar='E', type=int, default=0,
                            help='with --checkpoint, also write the state every E epochs')
    return parser


def _chunks(seq, n):
    return [seq[a:a + n] for a in range(0, len(seq), n)]


def run(args, tool, train, key, cost, tables, checkpoint_fields=None):
    """Run and print the CLI's ``tables`` that ``args.tables`` asks for.  train(jobs, device, seed, report) trains one
    group of jobs; key and cost group and deal the jobs (sweep.run_sharded).  Job ids count up in printed order over the
    whole invocation, so a job's streams depend only on the tables asked for and the seed.  With ``--checkpoint``
    (checkpoint.Sweep), train also takes ``start_states`` and ``on_epoch``, and checkpoint_fields are the fingerprint fields
    the CLI fixes (model, shared_t, batch, perm)."""
    from .mr_gan import dataset      # the reference's dataset() lives in mr_gan.py, which imports this module
    rank = sweep.dist_env()[0]
    seed = sweep.shared_seed(args.seed)          # one seed for every rank: same dataset, same splits, same job streams
    say = print if rank == 0 else (lambda *a, **k: None)
    if rank == 0:
        sys.stderr.write('seed: %d%s\n' % (seed, '   [SYNTHETIC data of the MREO shape: not the paper\'s dataset]' if args.synthetic else ''))
    nets = dict(precision=args.precision, epochs=args.epochs) if hasattr(args, 'epochs') else {}
    rep = results.Report(args, tool, rank, say, seed=seed, **nets)
    want = [t for t in tables if t in args.tables]
    next_id = [0]
    ck = None
    if getattr(args, 'checkpoint_every', 0) and not args.checkpoint:
        raise SystemExit('--checkpoint-every needs --checkpoint DIR')
    if getattr(args, 'checkpoint', None):
        ck = checkpoint.Sweep(args.checkpoint, tool, seed, args.epochs, args.checkpoint_every,
                              dict(checkpoint_fields, precision=args.precision))

    def data(modality, **kw):
        return dataset(modalities=modality, seed=seed, data_dir=args.data_dir, synthetic_data=args.synthetic, **kw)

    def train_all(jobs):
        for j in jobs:
            j['job_id'] = next_id[0]
            next_id[0] += 1
        if ck is None:
            return sweep.run_sharded(jobs, lambda js, dev: train(js, dev, seed, rep), group_size=args.group, key=key, cost=cost)
        start = {j['job_id']: ck.start(j) for j in jobs}        # folds of a group train in lockstep: group by start epoch too
        return sweep.run_sharded(jobs, lambda js, dev: ck.train(js, dev, rep, train), group_size=args.group,
                                 key=lambda j: (key(j), start[j['job_id']]), cost=cost)

    def title(text):
        say('\n', '-' * 25, text, '-' * 25)
        say('-' * 100)

    def modality_line(modality):
        say('-' * 25, MODALITIES[modality], 'modality', '-' * 25)

    def setting(label, jobs, res, blocks, folds=True, **fields):
        """One setting's lines: its label, one line per fold-training (per held-out object under leave-one-object-out,
        where folds is ignored), the average, then what the --confusion / --results / --saliency flags add."""
        say('-' * 15, label, '-' * 15)
        errors = results.errors(res)
        loo = 'name' in jobs[0]
        for j, e in zip(jobs, errors):
            if loo:
                say(j['name'], 'Test error:', e, 'Test accuracy:', 1.0 - e)
            elif folds:
                say('Test error:', e, 'Test accuracy:', 1.0 - e)
        say('Average leave-one-object-out error:' if loo else 'Average error:', np.mean(errors),
            'Average accuracy:', np.mean(1.0 - np.array(errors)))
        rep.setting(jobs, res, blocks, **fields)
        sys.stdout.flush()

    if '1' in want:                             # mr_gan.py:244-261
        # every (modality, labeled %, fold) training is independent: all 294 are built first, sharded over the GPUs in one
        # go, and the results are printed afterwards in the reference's loop order
        jobs = []
        for modality in range(len(MODALITIES)):
            X, y = data(modality)
            jobs += [j for p in LABELED for j in kfold_jobs(X, y, seed + p, percentlabeled=p)]
        res = train_all(jobs)
        title('Testing various amounts of labeled training data')
        for modality, (mj, mr) in enumerate(zip(_chunks(jobs, 6 * len(LABELED)), _chunks(res, 6 * len(LABELED)))):
            modality_line(modality)
            for p, js, rs in zip(LABELED, _chunks(mj, 6), _chunks(mr, 6)):
                setting('Percentage of training data labeled: %d%%' % p, js, rs, synthetic.block_widths(modality), table=1,
                        modality=MODALITIES[modality])

    if '2' in want:                             # mr_nn.py:129-146
        title('Testing various amounts of labeled training data')
        for modality in [2, 5]:
            modality_line(modality)
            X, y = data(modality)
            jobs = [j for p in LABELED for j in kfold_jobs(X, y, seed + p, percentlabeled=p)]
            res = train_all(jobs)
            for p, js, rs in zip(LABELED, _chunks(jobs, 6), _chunks(res, 6)):
                setting('Percentage of training data labeled: %d%%' % p, js, rs, synthetic.block_widths(modality), folds=False,
                        table=2, modality=MODALITIES[modality])

    for table in [t for t in ('3', '4') if t in want]:     # mr_gan.py:263-283 (GAN), mr_nn.py:148-168 (NN, SVM)
        title('Testing generalization with leave-one-object-out validation')
        for modality in [2, 5]:
            modality_line(modality)
            objects = data(modality, leaveObjectOut=True)
            jobs = [j for p in LOO_LABELED for j in loo_jobs(objects, percentlabeled=p)]
            res = train_all(jobs)
            for p, js, rs in zip(LOO_LABELED, _chunks(jobs, len(objects)), _chunks(res, len(objects))):
                setting('Percentage of training data labeled: %d%%' % p, js, rs, synthetic.block_widths(modality),
                        table=int(table), modality=MODALITIES[modality])

    if '5' in want:                             # mr_gan.py:285-318
        for header_mods, times, is_contact in (([0, 1, 2], [4, 3, 2, 1, 0.5, 0.2, 0.1], False),
                                               ([3], [1, 0.7, 0.5, 0.3, 0.2, 0.1, 0.05], True)):
            title('Testing various lengths of contact time in training data')
            for modality in header_mods:
                modality_line(modality)
                kws = [dict(contactmicTime=tm) if is_contact else dict(forcetempTime=tm) for tm in times]
                jobs = [j for kw in kws for j in kfold_jobs(*data(modality, **kw), seed, percentlabeled=100)]
                res = train_all(jobs)
                for tm, kw, js, rs in zip(times, kws, _chunks(jobs, 6), _chunks(res, 6)):
                    setting('Length of training data: %.1fs' % tm, js, rs, synthetic.block_widths(modality, **kw), table=5,
                            modality=MODALITIES[modality], time=tm)

    if '6' in want:                             # mr_gan.py:320-341
        title('Testing performance as quantity of unlabeled data increases')
        percentlabeled = 4
        unl = [0, 4, 8, 16, 32, 64, 100 - percentlabeled]
        for modality in [2, 5]:
            modality_line(modality)
            X, y = data(modality)
            say('-' * 15, 'Percentage of training data labeled: %d%%' % percentlabeled, '-' * 15)
            jobs = [j for pu in unl for j in kfold_jobs(X, y, seed + pu, percentlabeled=percentlabeled, percentunlabeled=pu)]
            res = train_all(jobs)
            for pu, js, rs in zip(unl, _chunks(jobs, 6), _chunks(res, 6)):
                setting('Percentage of training data unlabeled: %d%%' % pu, js, rs, synthetic.block_widths(modality), table=6,
                        modality=MODALITIES[modality])
    rep.close()
    return 0
