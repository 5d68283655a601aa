#!/usr/bin/env python3
"""Command line of the reference (stringdecomposer/main.py:186-252), same arguments and output files, with both
stages on the GPU: the decomposition DP through ``sd_run_files`` (in-process, instead of spawning ``build/bin/dp``)
and the identity rescoring through ``sd_identity``.  Needs neither Biopython nor python-edlib.

    python -m stringdecomposer_b200 reads.fa monomers.fa -o out_dir [--second-best] [-s ins,del,mm,match] ...

``--whole-reads`` sets the segment size (``-b``) to the longest read of the file, so that every read is decomposed as
one segment, with no segment seams for the overlap resolution to patch.

writes ``<out-dir>/<out-file>_raw.tsv``, ``<out-file>.tsv``, ``<out-file>_alt.tsv`` and ``stringdecomposer.log``.

Scoring: the reference's main.py always passes ten arguments to `dp`, which parses the scores only when it gets nine
(main.cpp:380-391), so ``-s`` never reaches the DP there.  That behaviour is kept by default so that outputs match the
reference; export ``SD_HONOR_SCORING=1`` to have ``-s`` applied.
"""
import argparse
import logging
import os
import re
import pathlib
import sys
import time

from . import _lib
from .convert import load_fasta, add_rc_monomers, convert_raw_file_native


def get_logger(filename, logger_name="StringDecomposer"):
    logger = logging.getLogger(logger_name)
    logger.setLevel(logging.INFO)
    logger.handlers.clear()
    fmt = logging.Formatter("%(asctime)s - %(name)s - %(levelname)s - %(message)s")
    for h in (logging.StreamHandler(sys.stdout), logging.FileHandler(filename, mode="w")):
        h.setFormatter(fmt)
        logger.addHandler(h)
    return logger


def honor_scoring():
    """SD_HONOR_SCORING parsed exactly like csrc/dp_main.cpp does (atoi != 0): "0" and "" mean off."""
    m = re.match(r"\s*([+-]?\d+)", os.environ.get("SD_HONOR_SCORING", ""))
    return bool(m) and int(m.group(1)) != 0


def run(sequences, monomers, num_threads, scoring, batch_size, raw_file, ed_thr, overlap, logger, flavour="cuda"):
    """main.py:186-197: run the DP on the two FASTA files and leave its stdout in raw_file.  The reference then reads
    that file back into one string (main.py:195-197); here the rescoring stage streams it in chunks of whole reads."""
    ins, dels, mm, match = (int(x) for x in scoring.split(","))
    if not honor_scoring():
        if (ins, dels, mm, match) != (-1, -1, -1, 1):
            note = ("NOTE: like the reference's dp (main.cpp:380-391), the DP ignores --scoring when it is driven by "
                    "main.py; export SD_HONOR_SCORING=1 to apply it")
            logger.info(note)
            print(note, file=sys.stderr)
        ins, dels, mm, match = -1, -1, -1, 1
    logger.info(" ".join(["Run", _lib.library_path(flavour), "with parameters", sequences, monomers, str(num_threads),
                          str(batch_size), str(overlap), scoring]))
    with open(raw_file, "w") as f:
        f.flush()
        st = _lib.run_files(sequences, monomers, int(num_threads), int(batch_size), int(overlap), (ins, dels, mm, match),
                            int(ed_thr), out_fd=f.fileno(), err_fd=2, flavour=flavour)
    if st != 0:                                       # subprocess.run(..., check=True) raises at main.py:194
        lib = _lib.load_library(flavour)
        raise _lib.SdError(st, "dp failed with status %d: %s" % (st, (lib.sd_last_error(None) or b"").decode()))
    return raw_file


def main(argv=None, flavour="cuda"):
    parser = argparse.ArgumentParser(prog="stringdecomposer_b200", description="Decomposes string into blocks alphabet")
    parser.add_argument("sequences", help="fasta-file with long reads or genomic sequences")
    parser.add_argument("monomers", help="fasta-file with monomers")
    parser.add_argument("-t", "--threads", help="number of threads (accepted; the DP runs on the GPU)", default="1", required=False)
    parser.add_argument("-o", "--out-dir", help="output directory (by default .)", default=".", required=False)
    parser.add_argument("--out-file", help='output tsv-file (by default "final_decomposition")', default="final_decomposition", required=False)
    parser.add_argument("-i", "--min-identity", help="only monomer alignments with percent identity >= MIN_IDENTITY are printed (by default MIN_IDENTITY=0)",
                        type=int, default=0, required=False)
    parser.add_argument("-s", "--scoring", help='scoring scheme "insertion,deletion,mismatch,match" (by default "-1,-1,-1,1")',
                        default="-1,-1,-1,1", required=False)
    parser.add_argument("-b", "--batch-size", help="size of the read segments (by default 5000)", type=str, default="5000", required=False)
    parser.add_argument("--second-best", dest="second_best", help="generate second best monomer and homopolymer scores", action="store_true")
    parser.add_argument("--ed_thr", help="align only monomers with edit distance less then ed_thr for each segment (by default align all monomers)",
                        default=-1, type=int, required=False)
    parser.add_argument("--whole-reads", dest="whole_reads", action="store_true",
                        help="decompose every read as one segment: the segment size becomes the longest read (overrides -b)")
    parser.add_argument("-v", "--overlap", help="size of the segment overlap (by default 500)", type=str, default="500", required=False)
    parser.add_argument("--device", help="CUDA device of the identity stage (by default 0; the DP obeys SD_DEVICES)", type=int, default=0)
    args = parser.parse_args(argv)
    pathlib.Path(args.out_dir).mkdir(parents=True, exist_ok=True)

    logger = get_logger(os.path.join(args.out_dir, "stringdecomposer.log"))
    logger.info("cmd: %s" % (sys.argv if argv is None else list(argv)))

    raw_fn = os.path.join(args.out_dir, args.out_file + "_raw.tsv")
    t0 = time.time()
    reads = None
    batch_size = args.batch_size
    if args.whole_reads:
        reads = load_fasta(args.sequences, "map")
        batch_size = str(max([len(s) for s in reads.values()] + [1]))
        logger.info("--whole-reads: segment size %s (the longest read), every read is one segment" % batch_size)
    run(args.sequences, args.monomers, args.threads, args.scoring, batch_size, raw_fn, args.ed_thr, args.overlap,
              logger, flavour=flavour)
    t1 = time.time()
    logger.info("Saved raw decomposition to " + raw_fn)

    if reads is None:
        reads = load_fasta(args.sequences, "map")
    monomers = add_rc_monomers(load_fasta(args.monomers))
    logger.info("Transforming raw alignments...")
    out_fn = os.path.join(args.out_dir, args.out_file + ".tsv")
    stats = {}
    convert_raw_file_native(raw_fn, reads, monomers, out_fn, int(args.min_identity), not args.second_best, device=args.device,
                            flavour=flavour, stats=stats)
    t2 = time.time()
    if stats.get("hirschberg_pairs"):
        logger.info("NOTE: %d interval/monomer pairs are large enough for edlib to leave its traceback for Hirschberg "
                    "splitting; their identity follows the traceback rule" % stats["hirschberg_pairs"])
    logger.info("Transformation finished. Results can be found in " + out_fn)
    logger.info("decomposition %.2f s, rescoring %.2f s (%d alignments, %.1f ms on the device)" %
                (t1 - t0, t2 - t1, stats.get("pairs", 0), stats.get("kernel_ms", 0.0)))
    logger.info("Thank you for using StringDecomposer!")
    return 0


if __name__ == "__main__":
    sys.exit(main())
