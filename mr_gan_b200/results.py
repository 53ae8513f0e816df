"""Per-fold results of the three CLIs (mr_gan.py, mr_nn.py, mr_svm.py): the JSON Lines record of one fold-training
(``--results FILE``) and the printed confusion block (``--confusion``).

The trainers return one float per job by default, or with ``details=True`` one dict per job,
``{'error': <the same float>, 'confusion': int [K, K]}`` (rows = true class, columns = predicted class).  A ``Report``
turns a setting's results into what the flags ask for; without either flag it prints and writes nothing, so the CLIs'
stdout stays the reference's."""
import json

import numpy as np

from .model import MATERIALS


def add_arguments(parser):
    parser.add_argument('--confusion', action='store_true',
                        help="after each setting's average, print its confusion matrix summed over the setting's fold-trainings")
    parser.add_argument('--results', metavar='FILE', default=None,
                        help='write one JSON Lines record per fold-training (rank 0)')


def errors(results):
    """The test errors of a list of trainer results (floats, or the dicts of details=True)."""
    return [r['error'] if isinstance(r, dict) else r for r in results]


def confusion_lines(conf, names=MATERIALS):
    """The printed block of one K x K confusion matrix, materials in model.MATERIALS order."""
    conf = np.asarray(conf)
    w = max(max(len(n) for n in names), len(str(int(conf.max()))) if conf.size else 1) + 1
    lines = ['Confusion matrix (rows: true material, columns: predicted material):',
             ' ' * w + ''.join(n.rjust(w) for n in names)]
    for n, row in zip(names, conf):
        lines.append(n.ljust(w) + ''.join(str(int(v)).rjust(w) for v in row))
    return lines


def record(tool, job, result, index, **fields):
    """The JSON record of one fold-training: the given fields, the job's labeled / unlabeled shares and id, its fold index
    within the setting (k-fold) or held-out object (leave-one-object-out), n_test, error and confusion."""
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
    conf = np.asarray(result['confusion'])
    rec['n_test'] = int(conf.sum())
    rec['error'] = result['error']
    rec['confusion'] = conf.tolist()
    return rec


class Report:
    """What --confusion and --results add to a CLI; inactive (details=False) when neither flag is given."""

    def __init__(self, args, tool, rank, say, **fields):
        self.show = bool(args.confusion)
        self.details = self.show or bool(args.results)
        self.tool, self.say, self.fields = tool, say, fields
        self.fh = open(args.results, 'w') if args.results and rank == 0 else None

    def setting(self, jobs, results, **fields):
        """Call after a setting's average line, with the setting's jobs and trainer results in printed order."""
        if not self.details:
            return
        if self.show:
            for line in confusion_lines(np.sum([np.asarray(r['confusion']) for r in results], axis=0)):
                self.say(line)
        if self.fh:
            for k, (j, r) in enumerate(zip(jobs, results)):
                self.fh.write(json.dumps(record(self.tool, j, r, k, **dict(self.fields, **fields))) + '\n')
            self.fh.flush()

    def close(self):
        if self.fh:
            self.fh.close()
            self.fh = None
