"""Per-fold results of the three CLIs (mr_gan.py, mr_nn.py, mr_svm.py): the JSON Lines record of one fold-training
(``--results FILE``), the printed confusion block (``--confusion``) and, for the GAN / NN CLIs, the saliency profiles
(``--saliency FILE``: an .npz file, and one printed line of block shares per setting).

The trainers return one float per job by default, or with ``details=True`` one dict per job,
``{'error': <the same float>, 'confusion': int [K, K]}`` (rows = true class, columns = predicted class); with
``saliency=True`` the dict also holds ``'saliency'``, float32 [K, D] (mean |d log p(true class) / dx| over the test rows of
each class, x in the fold's scaled input space).  A ``Report`` turns a setting's results into what the flags ask for;
without a flag it prints and writes nothing, so the CLIs' stdout stays the reference's."""
import json

import numpy as np

from .model import MATERIALS


def add_arguments(parser, saliency=False):
    parser.add_argument('--confusion', action='store_true',
                        help="after each setting's average, print its confusion matrix summed over the setting's fold-trainings")
    parser.add_argument('--results', metavar='FILE', default=None,
                        help='write one JSON Lines record per fold-training (rank 0)')
    if saliency:
        parser.add_argument('--saliency', metavar='FILE', default=None,
                            help="write every fold-training's input-gradient saliency profile [K, D] to one .npz file (rank 0) and "
                                 "print each feature block's share of a setting's summed profile after its average")


def errors(results):
    """The test errors of a list of trainer results (floats, or the dicts of details=True)."""
    return [r['error'] if isinstance(r, dict) else r for r in results]


def collect(fg, errors, details=False, saliency=False, extra=None):
    """A trainer's results from its group's test errors: the floats as they are, or with details / saliency one dict per
    fold, ``{'error', 'confusion'}`` from fg.confusion() and with saliency also ``'saliency'`` from fg.saliency(); extra:
    per-fold fields to add (a tuned SVM's selected point), which makes dicts too."""
    if not (details or saliency or extra):
        return errors
    out = [dict(error=e) for e in errors]
    if details or saliency:
        for r, c in zip(out, fg.confusion()):
            r['confusion'] = c
    if saliency:
        for r, p in zip(out, fg.saliency()):
            r['saliency'] = p
    for r, x in zip(out, extra or []):
        r.update(x)
    return out


def confusion_lines(conf, names=MATERIALS):
    """The printed block of one K x K confusion matrix, materials in model.MATERIALS order."""
    conf = np.asarray(conf)
    w = max(max(len(n) for n in names), len(str(int(conf.max()))) if conf.size else 1) + 1
    lines = ['Confusion matrix (rows: true material, columns: predicted material):',
             ' ' * w + ''.join(n.rjust(w) for n in names)]
    for n, row in zip(names, conf):
        lines.append(n.ljust(w) + ''.join(str(int(v)).rjust(w) for v in row))
    return lines


def setting_fields(tool, job, index, **fields):
    """What identifies one fold-training: the given fields, the job's labeled / unlabeled shares, its fold index within the
    setting (k-fold) or held-out object (leave-one-object-out), and its id."""
    rec = dict(tool=tool)
    rec.update(fields)
    rec['percentlabeled'] = job['percentlabeled']
    if job.get('percentunlabeled') is not None:
        rec['percentunlabeled'] = job['percentunlabeled']
    if 'name' in job:
        rec['object'] = job['name']
    else:
        rec['fold'] = index
    rec['job_id'] = job.get('job_id')
    return rec


def record(tool, job, result, index, **fields):
    """The JSON record of one fold-training: its setting_fields, n_test, error and confusion, and for a tuned SVM fold
    (mr_svm.py --tune) the selected C, gamma_D and the cv_accuracy grid [nC][nG]."""
    rec = setting_fields(tool, job, index, **fields)
    conf = np.asarray(result['confusion'])
    rec['n_test'] = int(conf.sum())
    rec['error'] = result['error']
    rec['confusion'] = conf.tolist()
    for k in ('C', 'gamma_D'):
        if k in result:
            rec[k] = float(result[k])
    if 'cv_accuracy' in result:
        rec['cv_accuracy'] = np.asarray(result['cv_accuracy'], dtype=np.float64).tolist()
    return rec


def block_shares(profiles, blocks):
    """Each feature block's share of the summed profiles (over folds, classes and the block's features): a mass share, so
    wider blocks hold more features.  blocks: [(name, width)] in row order."""
    tot = np.sum([np.asarray(p, dtype=np.float64).sum(axis=0) for p in profiles], axis=0)    # [D]
    edges = np.cumsum([0] + [w for _, w in blocks])
    mass = np.array([tot[a:b].sum() for a, b in zip(edges[:-1], edges[1:])])
    return mass / mass.sum()


def share_line(shares, blocks):
    return 'Saliency share: ' + ' '.join('%s %.3f' % (name, v) for (name, _), v in zip(blocks, shares))


class Report:
    """What --confusion, --results and --saliency add to a CLI; inactive (details=False, saliency=False) without them."""

    def __init__(self, args, tool, rank, say, **fields):
        self.show = bool(args.confusion)
        sal = getattr(args, 'saliency', None)
        self.saliency = bool(sal)
        self.details = self.show or bool(args.results)
        self.tool, self.say, self.fields = tool, say, fields
        self.fh = open(args.results, 'w') if args.results and rank == 0 else None
        self.sal_path = sal if sal and rank == 0 else None
        self.sal_arrays, self.sal_index = {}, []

    def setting(self, jobs, results, blocks=None, **fields):
        """Call after a setting's average line, with the setting's jobs and trainer results in printed order; blocks: the
        [(name, width)] feature blocks of the setting's rows (needed with --saliency).  Results of a tuned SVM (mr_svm.py
        --tune) also print the selected C and gamma * D of every fold-training."""
        if self.show:
            for line in confusion_lines(np.sum([np.asarray(r['confusion']) for r in results], axis=0)):
                self.say(line)
        if self.saliency:
            self.say(share_line(block_shares([r['saliency'] for r in results], blocks), blocks))
            for k, (j, r) in enumerate(zip(jobs, results)):
                self.sal_arrays['job_%d' % j['job_id']] = np.asarray(r['saliency'], dtype=np.float32)
                self.sal_index.append(dict(setting_fields(self.tool, j, k, **dict(self.fields, **fields)),
                                           blocks=[[name, int(w)] for name, w in blocks]))
        if results and isinstance(results[0], dict) and 'C' in results[0]:
            self.say('Selected C: ' + ' '.join('%g' % r['C'] for r in results) +
                     ' Selected gamma*D: ' + ' '.join('%g' % r['gamma_D'] for r in results))
        if self.fh:
            for k, (j, r) in enumerate(zip(jobs, results)):
                self.fh.write(json.dumps(record(self.tool, j, r, k, **dict(self.fields, **fields))) + '\n')
            self.fh.flush()

    def close(self):
        if self.fh:
            self.fh.close()
            self.fh = None
        if self.sal_path:
            with open(self.sal_path, 'wb') as f:       # the name as given (np.savez would append .npz to a path)
                np.savez(f, index=np.array(json.dumps(self.sal_index)), **self.sal_arrays)
            self.sal_path = None
