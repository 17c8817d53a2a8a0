"""`kmer histo`: the k-mer multiplicity spectrum of a FASTA file (the histogram of `kmer count`'s count column)."""
import logging

import click

from kman_b200 import alphabet as ab
from kman_b200.io import input_file_exists
from kman_b200.scripts import arguments as args


@click.command(name="histo", context_settings=dict(help_option_names=["--help", "-h"]),
               help="Histogram of k-mer multiplicities of INPUT: one line 'M<TAB>N' per multiplicity M that occurs, "
                    "ascending, where N is the number of distinct k-mers seen exactly M times (the count column of "
                    "`kmer count INPUT OUTPUT K`, without writing the table). The INPUT file can be gzipped.")
@args.input_path()
@args.output_path(file_okay=True)
@args.k()
@args.reverse()
@args.canonical()
def run(input_path: str, output_path: str, k: int, reverse: bool = False, canonical: bool = False) -> None:
    args.check_canonical(canonical, reverse)
    input_file_exists(input_path)
    if k <= 1:
        raise AssertionError(f"k must be >= 1, got {k} instead.")  # the check `kmer count` makes
    from kman_b200.engine import CANONICAL, get_engine

    eng = get_engine()
    d = eng.load_fasta(input_path, ab.default_alphabet(), ab.NATYPES.DNA, with_names=False)
    with open(output_path, "wb") as fh:  # (the file exists even when the spectrum is empty)
        eng.write_histogram(d, k, CANONICAL if canonical else reverse, fh)
    logging.info("That's all! :smiley:")
