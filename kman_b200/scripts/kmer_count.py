"""`kmer count` (kmermaid/scripts/kmer_count.py:20-144)."""
import logging
import tempfile
from typing import Optional

import click

from kman_b200.batcher import BatcherThreading, FastaBatcher, load_batches
from kman_b200.io import input_file_exists, set_tempdir
from kman_b200.join import KJoiner, KJoinerThreading
from kman_b200.scripts import arguments as args


@click.command(name="count", context_settings=dict(help_option_names=["--help", "-h"]),
               help="Count occurrences of all k-mers from INPUT (SEQ_COUNT: sequence<TAB>count table). The INPUT file can be gzipped.")
@args.input_path()
@args.output_path(file_okay=True)
@args.k()
@args.reverse()
@args.canonical()
@args.scan_mode()
@args.batch_size()
@args.batch_mode()
@args.previous_batches()
@args.count_mode()
@args.memory_mode()
@args.threads()
@args.tmp()
@args.re_sort()
@args.min_count()
@args.max_count()
def run(input_path: str, output_path: str, k: int, reverse: bool = False, scan_mode: str = FastaBatcher.MODE.KMERS.name,
        batch_size: int = 1000000, batch_mode: str = BatcherThreading.FEED_MODE.APPEND.name,
        previous_batches: Optional[str] = None, count_mode: str = KJoiner.MODE.SEQ_COUNT.name,
        memory_mode: str = KJoiner.MEMORY.NORMAL.name, threads: int = 1, tmp: str = tempfile.gettempdir(),
        re_sort: bool = False, min_count: int = 1, max_count: Optional[int] = None, canonical: bool = False) -> None:
    args.check_canonical(canonical, reverse, previous_batches, count_mode)
    input_file_exists(input_path)
    set_tempdir(tmp)
    joiner = KJoinerThreading(KJoiner.MODE[count_mode], KJoiner.MEMORY[memory_mode])
    joiner.count_range = (min_count, max_count)  # (a bad range or a VEC mode fails before any work)
    if previous_batches is not None:
        batches = load_batches(previous_batches, threads, re_sort)
    else:
        batches = (FastaBatcher(scan_mode=FastaBatcher.MODE[scan_mode], reverse=reverse, size=batch_size, threads=threads,
                                canonical=canonical)
                   .do(input_path, k, BatcherThreading.FEED_MODE[batch_mode]).collection)
    prep_joiner(joiner, len(batches), threads).join(batches, output_path)
    logging.info("That's all! :smiley:")


def prep_joiner(joiner: KJoinerThreading, n_batches: int, threads: int = 1) -> KJoinerThreading:
    joiner.threads = threads
    joiner.batch_size = max(2, int(n_batches / threads))
    return joiner
