# !/usr/bin/env python3
"""DeepGRP prediction with a pretrained model on B200 -- drop-in for ``deepgrp predict``
(reference ``deepgrp/__main__.py``).  Same options (``-b -s -x -l -t --xla -v``, ``predict
--output --no_use_mss``); ``-t`` and ``--xla`` are accepted and ignored (there is no TensorFlow).
The README form ``deepgrp <modelfile> <fastafile>...`` (reference ``README.rst:92-98``) is accepted
as well as the ``predict`` sub-command.  ``train`` trains a GRU model on the GPU (``deepgrp_b200.training``).
"""
from __future__ import annotations

import argparse
import io
import logging
import os
import sys
from typing import Iterator, List, TextIO, Tuple

import numpy as np

from . import model as dgmodel
from . import prediction as dgpred
from . import sequence as dgsequence

logging.basicConfig()
_LOG = logging.getLogger(__name__)


def _read_multi_fasta(filestream: TextIO) -> Iterator[Tuple[str, str]]:
    """(header, sequence) of every record of a multi-FASTA stream, as the reference reads it
    (``deepgrp/__main__.py:20-43``): lines are stripped, ``>`` opens a record whose header is the rest of that
    line, other lines are upper-cased and concatenated.  Its corner cases are kept: a line that is empty after
    stripping raises ``IndexError`` (the reference indexes its first character), text in front of the first
    ``>`` and records whose header is empty are dropped."""
    _LOG.debug("Reading FASTA file.")
    name, pieces = "", []                     # name == "": nothing to emit for what is being collected
    for raw_line in filestream:
        text = raw_line.strip()
        if not text:
            raise IndexError("string index out of range")
        if text.startswith(">"):
            if name:
                yield name, "".join(pieces)
            name, pieces = text[1:], []
        else:
            pieces.append(text.upper())
    if name:
        yield name, "".join(pieces)


def _read_raw(filename: str):
    """Raw FASTA bytes of `filename` ("-" = stdin; ``.gz`` files are decompressed on the host, as the
    reference's preprocessing script does, deepgrp/_scripts/preprocess_sequence.py:19-38).  A regular file is
    memory-mapped, so only the bytes the prediction stream uploads (this rank's records) are ever read."""
    if filename == "-":
        return sys.stdin.buffer.read()
    if filename.endswith(".gz"):
        import gzip
        with gzip.open(filename, "rb") as fh:
            return fh.read()
    import mmap
    with open(filename, "rb") as fh:
        if os.fstat(fh.fileno()).st_size == 0:
            return b""
        return mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ)


class _ByteSink:
    """Adapter for the TSV pieces (bytes-like views): binary streams take them as they are, text streams through
    their ``.buffer`` when they have one (``sys.stdout``), otherwise decoded (an ``io.StringIO`` in tests)."""

    def __init__(self, outstream):
        self.out = outstream
        self.raw = getattr(outstream, "buffer", None)
        self.binary = isinstance(outstream, (io.RawIOBase, io.BufferedIOBase))

    def write(self, view) -> None:
        if self.binary:
            self.out.write(view)
        elif self.raw is not None:
            self.out.flush()
            self.raw.write(view)
        else:
            self.out.write(bytes(view).decode("utf-8", "replace"))


def _predict(dnasequence: str, model: dgmodel.ModelWeights, options: dgmodel.Options,
             step_size: int, use_mss: bool) -> Tuple[np.ndarray, int]:
    """Labels of one sequence and the position of its first non-N base (reference ``deepgrp/__main__.py:46-83``):
    encode, enumerate windows, predict with the max-vote, then MSS or softmax, argmax -- the reference's five
    calls in its order, each through the CUDA path."""
    start_pos, one_hot = dgsequence.one_hot_encode_dna_sequence(dnasequence)
    n_bases = one_hot.shape[1]
    _LOG.debug("Encoded %d bases, first base at %d.", n_bases, start_pos)
    windows = dgpred.fetch_validation_batch(one_hot, step_size, options.batch_size, options.vecsize)
    votes = dgpred.predict(model, windows, (n_bases, model.output_shape[2]), step_size)
    _LOG.debug("Prediction finished, %s.", "applying MSS" if use_mss else "softmax")
    decided = dgpred.apply_mss(votes, options) if use_mss else dgpred.softmax(votes)
    return np.asanyarray(decided.argmax(axis=1)), start_pos


class CommandLineParser:
    """Commandline parser (reference ``deepgrp/__main__.py:86-351``)."""

    def __init__(self, **kwargs):
        kwargs.setdefault("prog", "deepgrp")
        kwargs.setdefault("formatter_class", argparse.ArgumentDefaultsHelpFormatter)
        kwargs.setdefault("description", "DeepGRP - Prediction of repetitive elements")
        self.parser = argparse.ArgumentParser(**kwargs)
        self.args = None
        self.threads = 1
        self.xla = False
        self.verbose = 0
        # the reference's options (deepgrp/__main__.py:101-207), same flags, defaults and destinations
        integer_options = [
            ("--batch_size", "-b", 256, "Batch size (only decides where the reference places the final short batch)"),
            ("--step_size", "-s", 50, "Window step size"),
            ("--xdrop_length", "-x", 50, "XDrop parameter for MSS algorithm, ignored if --no_use_mss, "
                                         "disabled with values<0"),
            ("--min_mss_length", "-l", 50, "Minimal length of maximum scoring segments, ignored if --no_use_mss"),
            ("--threads", "-t", 1, "Accepted for compatibility; ignored (GPU path)"),
        ]
        for long_flag, short_flag, default, text in integer_options:
            self.parser.add_argument(long_flag, short_flag, type=int, default=default, help=text)
        self.parser.add_argument("--xla", action="store_true", help="Accepted for compatibility; ignored")
        self.parser.add_argument("-v", "--verbose", action="count", default=0, help="Increase verbosity")
        commands = self.parser.add_subparsers(help="sub-command help", dest="command")
        sub = {name: commands.add_parser(name=name, description=text,
                                         formatter_class=argparse.ArgumentDefaultsHelpFormatter)
               for name, text in (("predict", "predict using a deepgrp model"),
                                  ("train", "Train a deepgrp model"))}
        sub["predict"].add_argument("model", type=str, help="Keras model in HDF5 format (or .npz weights)")
        sub["predict"].add_argument("FASTA", nargs="+", type=str, help="Fasta input files")
        sub["predict"].add_argument("--output", type=str, default="-", help="Output filename")
        sub["predict"].add_argument("--no_use_mss", "-m", action="store_true",
                                    help="Disable maximum scoring segment algorithm")
        sub["predict"].add_argument("--stepwise", action="store_true",
                                    help="Run the reference's five Python-level calls per record instead of the "
                                         "fused whole-record GPU call")
        for name, text in (("parameter", "TOML file of hyper-parameters (Options)"),
                           ("trainfile", "one-hot .npz of the training chromosome (preprocess_sequence)"),
                           ("validfile", "one-hot .npz of the validation chromosome"),
                           ("bedfile", "repeat annotations: chromosome, begin, end, repeat number")):
            sub["train"].add_argument(name, type=str, help=text)
        sub["train"].add_argument("--logdir", type=str, default=".", help="Directory for best.hdf5 and history.tsv")
        sub["train"].add_argument("--modelfile", type=str, default="model.hdf5", help="Keras HDF5 file to write")

    def parse_args(self, argv=None) -> "CommandLineParser":
        """Parse command line arguments."""
        argv = list(sys.argv[1:] if argv is None else argv)
        # README form: `deepgrp [options] <modelfile> <fasta...>` without the sub-command
        if not any(a in ("predict", "train") for a in argv) and not any(a in ("-h", "--help") for a in argv):
            with_value = {"-b", "--batch_size", "-s", "--step_size", "-x", "--xdrop_length", "-l",
                          "--min_mss_length", "-t", "--threads"}
            i = 0
            while i < len(argv):
                if argv[i] in with_value:
                    i += 2
                elif argv[i].startswith("-") and argv[i] != "-":
                    i += 1
                else:
                    break
            argv.insert(i, "predict")
        args = self.parser.parse_args(argv)
        self.threads = args.threads
        self.verbose = args.verbose
        self.xla = args.xla
        self.args = args
        return self

    def setup_tensorflow(self) -> "CommandLineParser":
        """Kept for call-compatibility with the reference (``:221-233``); nothing to set up."""
        return self

    def set_logging(self) -> "CommandLineParser":
        loglevels = [logging.WARNING, logging.INFO, logging.DEBUG]
        _LOG.setLevel(level=loglevels[min(len(loglevels) - 1, self.verbose)])
        return self

    def run(self):
        """Run the command provided by the user."""
        if self.args.command is None:
            self.parser.error("a sub-command is required")
        options = dgmodel.Options(min_mss_len=self.args.min_mss_length,
                                  batch_size=self.args.batch_size,
                                  xdrop_len=self.args.xdrop_length)
        getattr(self, self.args.command)(self.args, options)

    @staticmethod
    def predict(args: argparse.Namespace, options: dgmodel.Options):
        """Predict with deepgrp (reference ``deepgrp/__main__.py:252-297``)."""
        _LOG.debug("Loading model %s!", args.model)
        model = dgmodel.load_model(args.model)
        options.vecsize = model.input_shape[1]
        _LOG.info("Model loading finished successfully!")
        outstream = sys.stdout if args.output == "-" else open(args.output, "w")
        use_mss = not args.no_use_mss
        for filename in args.FASTA:
            _LOG.info("Processing %s", filename)
            if getattr(args, "stepwise", False):
                if filename == "-":
                    filestream = sys.stdin
                elif filename.endswith(".gz"):
                    import gzip
                    filestream = gzip.open(filename, "rt")
                else:
                    filestream = open(filename, "r")
                try:
                    for header, dnasequence in _read_multi_fasta(filestream):
                        predictions, startpos = _predict(dnasequence, model, options,
                                                         args.step_size, use_mss=use_mss)
                        for segment in dgsequence.yield_segments(predictions, startpos):
                            if segment[2] > 0:
                                outstream.write("{}\t{}\t{}\t{}\t{}\n".format(
                                    filename, header, *segment))
                finally:
                    if filename != "-":
                        filestream.close()
            else:
                # records stream through the GPU pipeline; a record's rows are written as soon as it is done,
                # so an error in a later record leaves the earlier rows in the output, as in the reference
                stats = dgpred.predict_fasta_tsv_stream(
                    model, _read_raw(filename), filename, _ByteSink(outstream), args.step_size,
                    options.batch_size, use_mss, options.min_mss_len, options.xdrop_len)
                _LOG.info("%s: %d records, %d bases, %d rows", filename, stats["records"], stats["bases"],
                          stats["rows"])
        if args.output != "-":
            outstream.close()

    @staticmethod
    def train(args: argparse.Namespace, options: dgmodel.Options):
        """Train a model (reference ``deepgrp/__main__.py:299-351``): TOML hyper-parameters, the two one-hot
        ``.npz`` files, their labels from the annotation table, ``training``, then the Keras HDF5 model file."""
        names = ("parameter", "trainfile", "validfile", "bedfile", "logdir", "modelfile")
        if any(getattr(args, name, None) is None for name in names):
            raise SystemExit("usage: deepgrp train parameter trainfile validfile bedfile [--logdir LOGDIR] "
                             "[--modelfile MODELFILE]")
        from . import hdf5
        from . import preprocessing as dgprep
        from . import training as dgtrain
        options = _train_options(args.parameter, options)
        data = []
        for path in (args.trainfile, args.validfile):
            fwd, _ = dgprep.load_onehot_npz(path)
            dgtrain.onehot_to_codes(fwd)                      # columns must be one-hot (ValueError)
            truelbl = dgprep.preprocess_y(args.bedfile, chromosome_name(path), fwd.shape[1],
                                          options.repeats_to_search)
            data.append(dgprep.Data(*dgprep.drop_start_end_n(fwd, truelbl)))
        model = dgmodel.create_model(options)
        _LOG.info("Training on %s (%d bases), validating on %s (%d bases)", args.trainfile, data[0].fwd.shape[1],
                  args.validfile, data[1].fwd.shape[1])
        dgtrain.training(tuple(data), options, model, args.logdir)
        hdf5.save_keras_model(args.modelfile, model)
        _LOG.info("Model written to %s", args.modelfile)


def chromosome_name(path: str) -> str:
    """The chromosome a one-hot file holds: its base name up to the first ``.`` (``chr1.fa.gz.npz`` -> ``chr1``)."""
    return os.path.basename(path).split(".", 1)[0]


def _train_options(parameter: str, cli_options: dgmodel.Options) -> dgmodel.Options:
    """Options of ``deepgrp train``: the TOML file's keys, and the command line's values for what it lacks."""
    import tomllib
    with open(parameter, "rb") as fh:
        parsed = tomllib.load(fh)
    return dgmodel.Options(**{**cli_options.todict(), **parsed})


def main():
    """Main function."""
    CommandLineParser().parse_args().set_logging().setup_tensorflow().run()


if __name__ == "__main__":
    main()
