"""`kmer` entry point (kmermaid/scripts/kmer.py:13-32): group with batch, count, uniq, and histo."""
import click

from kman_b200 import __version__
from kman_b200.scripts import kmer_batch, kmer_count, kmer_histo, kmer_uniq


@click.group(name="kmer", context_settings=dict(help_option_names=["--help", "-h"]),
             help=f"Version: {__version__}\n\nK-mer management tools (B200-native engine behind the kmermaid interface).")
@click.version_option(__version__)
def main():
    """Entry point."""


main.add_command(kmer_batch.run)
main.add_command(kmer_count.run)
main.add_command(kmer_uniq.run)
main.add_command(kmer_histo.run)

if __name__ == "__main__":
    main()
