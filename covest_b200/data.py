"""Histogram files, saved results and the YAML report (reference: covest/data.py).  Formats and
YAML keys are the reference's; the likelihood values in the report come from the device."""
import random
from collections import namedtuple
from os import path

import yaml

from .models import BasicModel, select_model
from .utils import safe_int, verbose_print

REFERENCE_VERSION = '0.5.6'  # the CovEst release whose behaviour this package mirrors


class InvalidFormatException(Exception):
    def __init__(self, fname):
        self.fname = fname

    def __str__(self):
        return 'Unable to parse %s. Unsupported format.' % self.fname


def load_histogram(fname):
    """`<abundance> <count>` lines and `#key:value` comment lines -> (hist, meta)
    (data.py:22-41)."""
    hist, meta = {}, {}
    with open(fname, 'r') as f:
        for line in f:
            if line[0] == '#':
                try:
                    key, value = line[1:].strip().split(':')
                    meta[key] = value
                except (IndexError, ValueError):
                    # the reference only swallows IndexError; a comment without exactly one
                    # colon makes it raise ValueError.  Ignoring the line is the gentler reading.
                    pass
                continue
            fields = line.split()
            try:
                hist[int(fields[0])] = int(fields[1])
            except (ValueError, KeyError):
                raise InvalidFormatException(fname)
    return hist, meta


def save_histogram(hist, fname, meta=None):
    with open(fname, 'w') as f:
        for key, value in (meta or {}).items():
            f.write('#{}:{}\n'.format(key, value))
        for j, h in hist.items():
            f.write('%d %d\n' % (j, h))


def load_reads(fname):
    """(id, sequence) of every read of a FASTA/FASTQ file; needs Biopython (data.py:44-55)."""
    from Bio import SeqIO
    ext = path.splitext(fname)[1]
    fmt = 'fastq' if ext in ('.fq', '.fastq') else 'fasta'
    try:
        with open(fname, 'r') as f:
            for read in SeqIO.parse(f, fmt):
                yield read.id, read.seq
    except FileNotFoundError as exc:
        verbose_print(str(exc))


def sample_reads(src_reads_file, dest_reads_file, factor):
    keep = 1.0 / factor
    with open(dest_reads_file, 'w') as out:
        for read_id, read in load_reads(src_reads_file):
            if random.random() < keep:
                out.write('>{}\n{}\n'.format(read_id, read))


def count_reads_stats(fname):
    total = count = 0
    for _, read in load_reads(fname):
        total += len(read)
        count += 1
    return (round(total / count) if count else 0), total


ParsedData = namedtuple('ParsedData', ('estimated', 'guess', 'model', 'sample_factor'))


def parse_data(f):
    """A previously printed YAML report (data.py:76-91)."""
    data = yaml.safe_load(f)
    try:
        model = select_model(data['model'])
    except KeyError:
        model = BasicModel
    guess = [data.get('guessed_coverage'), data.get('guessed_error_rate')]
    estimated = [data.get(name) for name in model.params]
    return ParsedData(estimated=estimated, guess=guess, model=model,
                      sample_factor=data.get('sample_factor', 1))


def replace_none(dest, src):
    if dest is None or src is None:
        raise ValueError('Invalid arguments.')
    dest = list(dest)
    if len(dest) != len(src):
        raise ValueError('Length of arguments should be equal.')
    return [s if d is None else d for d, s in zip(dest, src)]


def genome_size(hist_orig, model, coverage, sample_factor):
    """The report's genome size at `coverage` (sampled data): k-mers over the corrected coverage of the
    un-sampled data (data.py:152-154).  Decreasing in the coverage."""
    kmers = sum(j * h for j, h in hist_orig.items())
    return safe_int(round(kmers / model.correct_c(coverage * sample_factor)))


def interval_report(hist_orig, model, sample_factor, intervals, level):
    """The report's keys of likelihood-ratio intervals (CoverageEstimator.likelihood_intervals, model
    coordinates): ci_level, <param>_ci = [lo, hi] per parameter (coverage times sample_factor, as the
    estimate), genome_size_ci = [gs(coverage hi), gs(coverage lo)] and ci_flags = the flags set per
    parameter."""
    out = {'ci_level': float(level)}
    for name, iv in intervals.items():
        f = sample_factor if name == 'coverage' else 1
        out['%s_ci' % name] = [float(iv.lo * f), float(iv.hi * f)]
    if 'coverage' in intervals:
        c = intervals['coverage']
        out['genome_size_ci'] = [genome_size(hist_orig, model, c.hi, sample_factor),
                                 genome_size(hist_orig, model, c.lo, sample_factor)]
    out['ci_flags'] = {name: sorted(k for k, v in iv.flags.items() if v) for name, iv in intervals.items()}
    return out


def print_output(hist_orig, model, success, sample_factor, estimated=None, guess=None, orig=None,
                 reads_size=None, silent=False, orig_sample_factor=1, starting_points=1,
                 use_grid_search=False, extra=None):
    """Build (and unless `silent` print) the YAML report; keys and arithmetic as data.py:106-173.
    The up-to-three log-likelihoods it needs are evaluated in one device launch.  `extra`: further
    keys (interval_report), added last."""
    def named(names, values):
        if values is None or names is None:
            return {}
        values = [None if v is None else float(v) for v in values]
        if values[0] is not None and sample_factor is not None:
            values[0] *= sample_factor  # coverage is reported for the un-sampled data
        return {name: v for name, v in zip(names, values) if v is not None}

    out = {
        'model': model.short_name(),
        'hist_size': max(model.hist),
        'sample_factor': sample_factor,
        'orig_sample_factor': orig_sample_factor,
        'success': success,
        'version': REFERENCE_VERSION,
        'starting_points': starting_points,
        'use_grid_search': use_grid_search,
    }
    want = {}
    if guess is not None:
        want['guessed_loglikelihood'] = tuple(guess)
    if estimated is not None:
        want['loglikelihood'] = tuple(estimated)
    if orig is not None and any(orig):
        try:
            want['provided_loglikelihood'] = tuple(replace_none(orig, estimated))
        except ValueError:
            pass
    ll = {}
    if want:  # one launch for all of them
        values = model.loglikelihood_batch(model._rows(list(want.values())))
        ll = {name: float(v) for name, v in zip(want, values)}

    if guess is not None:
        out.update(named(('guessed_coverage', 'guessed_error_rate'), guess))
        out['guessed_loglikelihood'] = ll['guessed_loglikelihood']
    if estimated is not None:
        out.update(named(model.params, estimated))
        out['orig_coverage'] = float(estimated[0] * orig_sample_factor * sample_factor)
        out['loglikelihood'] = ll['loglikelihood']
        out['genome_size'] = genome_size(hist_orig, model, estimated[0], sample_factor)
        if reads_size is not None:
            out['genome_size_reads'] = safe_int(
                round(reads_size / (estimated[0] * sample_factor * orig_sample_factor)))
    if orig is not None and any(orig):
        out.update(named(['provided_%s' % name for name in model.params], orig))
        if 'provided_loglikelihood' in want:
            out['provided_loglikelihood'] = ll['provided_loglikelihood']
    if extra:
        out.update(extra)
    if not silent:
        print(yaml.dump(out, indent=4, default_flow_style=False))
    return out
