"""Shared click decorators: the option surface of kmermaid/scripts/arguments.py:14-221."""
import tempfile

import click

from kman_b200.batcher import BatcherThreading, FastaBatcher
from kman_b200.join import KJoiner


def input_path():
    return click.argument("input_path", metavar="INPUT", type=click.Path(exists=True, file_okay=True, readable=True))


def output_path(file_okay=False, dir_okay=False):
    return click.argument("output_path", metavar="OUTPUT",
                          type=click.Path(exists=False, file_okay=file_okay, dir_okay=dir_okay, writable=True))


def k():
    return click.argument("k", type=click.INT)


def reverse():
    return click.option("--reverse", "-r", is_flag=True, help="Include also reverse-complemented sequences")


def canonical():
    # long option only: -C is the reference's --compress
    return click.option("--canonical", is_flag=True,
                        help="Count each k-mer together with its reverse complement, as the smaller of the two "
                             "(canonical k-mers, one per window). Not with -r, -B or the VEC count modes.")


def check_canonical(canonical: bool, reverse: bool = False, previous_batches=None, count_mode: str = "") -> None:
    """AssertionError, before any work, for --canonical with an option it cannot go with."""
    if not canonical:
        return
    if reverse:
        raise AssertionError("--canonical already covers both strands: do not combine it with -r")
    if previous_batches is not None:
        raise AssertionError("--canonical needs the FASTA input: -B batch files fixed their strands when written")
    if count_mode.startswith("VEC_"):
        raise AssertionError(f"--canonical does not apply to {count_mode}: the vectors are per strand")


def scan_mode():
    return click.option("--scan-mode", "-s", type=click.Choice([m.name for m in FastaBatcher.MODE], case_sensitive=True),
                        default=FastaBatcher.MODE.KMERS.name,
                        help=f"Accepted for compatibility; does not change results. Default: {FastaBatcher.MODE.KMERS.name}")


def batch_size():
    return click.option("--batch-size", "-b", type=click.INT, default=1000000,
                        help="Number of k-mers per batch. Default: 1000000")


def batch_mode():
    return click.option("--batch-mode", "-m",
                        type=click.Choice([m.name for m in BatcherThreading.FEED_MODE], case_sensitive=True),
                        default=BatcherThreading.FEED_MODE.APPEND.name,
                        help=f"Default: {BatcherThreading.FEED_MODE.APPEND.name}")


def previous_batches():
    return click.option("--previous-batches", "-B", type=click.Path(exists=True, dir_okay=True, readable=True),
                        help="Path to folder with previously generated batches.")


def count_mode():
    return click.option("--count-mode", "-m",
                        type=click.Choice([m.name for m in KJoiner.MODE if "COUNT" in m.name], case_sensitive=True),
                        default=KJoiner.MODE.SEQ_COUNT.name, help=f'Default: "{KJoiner.MODE.SEQ_COUNT.name}"')


def memory_mode():
    return click.option("--memory-mode", "-M", type=click.Choice([m.name for m in KJoiner.MEMORY], case_sensitive=True),
                        default=KJoiner.MEMORY.NORMAL.name, help=f'Default: "{KJoiner.MEMORY.NORMAL.name}"')


def threads():
    return click.option("--threads", "-t", type=click.INT, default=1, help="Number of threads for parallelization.")


def tmp():
    return click.option("--tmp", "-T", type=click.Path(exists=True), default=tempfile.gettempdir(),
                        help=f'Temporary folder path. Default: "{tempfile.gettempdir()}"')


def compress():
    return click.option("--compress", "-C", is_flag=True, help="Compress output files.")


def re_sort():
    return click.option("--re-sort", "-R", is_flag=True, help="Force batch re-sorting, when loaded with -B.")


def min_count():
    return click.option("--min-count", type=click.INT, default=1,
                        help="Write only the k-mers that occur at least this many times. Default: 1")


def max_count():
    return click.option("--max-count", type=click.INT, default=None,
                        help="Write only the k-mers that occur at most this many times (at most 4294967295). Default: no limit")
