"""`kmer uniq` (kmermaid/scripts/kmer_uniq.py:19-108)."""
import logging
import tempfile
from typing import Optional

import click

from kman_b200.batcher import BatcherThreading, FastaBatcher, load_batches
from kman_b200.io import input_file_exists, set_tempdir
from kman_b200.join import KJoinerThreading
from kman_b200.scripts import arguments as args


@click.command(name="uniq", context_settings=dict(help_option_names=["--help", "-h"]),
               help="Extract all k-mers that appear only once in the INPUT fasta file. The INPUT file can be gzipped.")
@args.input_path()
@args.output_path(file_okay=True)
@args.k()
@args.reverse()
@args.canonical()
@args.scan_mode()
@args.batch_size()
@args.batch_mode()
@args.previous_batches()
@args.threads()
@args.tmp()
@args.re_sort()
def run(input_path: str, output_path: str, k: int, reverse: bool = False, scan_mode: str = FastaBatcher.MODE.KMERS.name,
        batch_size: int = 1000000, batch_mode: str = BatcherThreading.FEED_MODE.APPEND.name,
        previous_batches: Optional[str] = None, threads: int = 1, tmp: str = tempfile.gettempdir(),
        re_sort: bool = False, canonical: bool = False) -> None:
    args.check_canonical(canonical, reverse, previous_batches)
    input_file_exists(input_path)
    set_tempdir(tmp)
    if previous_batches is not None:
        batches = load_batches(previous_batches, threads, re_sort)
    else:
        batches = (FastaBatcher(scan_mode=FastaBatcher.MODE[scan_mode], reverse=reverse, size=batch_size, threads=threads,
                                canonical=canonical)
                   .do(input_path, k, BatcherThreading.FEED_MODE[batch_mode]).collection)
    joiner = KJoinerThreading()
    joiner.threads = threads
    joiner.batch_size = max(2, int(len(batches) / threads))
    joiner.join(batches, output_path)
    logging.info("That's all! :smiley:")
