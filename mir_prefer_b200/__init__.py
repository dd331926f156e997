"""mir_prefer_b200 -- B200-native fold stage for miR-PREFeR (libmirfold.so + Python host layer)."""
from ._lib import MirfoldError, LIB_PATH  # noqa: F401
from .fold import MirFold, FoldResult, Genome, parse_rnalfold_input, format_record, convert_sequence  # noqa: F401

from .structures import (structures_from_result, structures_from_result_native, get_structures_next_extendregion, is_stem_loop, filter_ss,  # noqa: F401
                         has_one_good_bifurcation, classify)

from .records import LocusRecord, fold_records, header_line, parse_header, records_from_fasta, write_fasta, get_reverse_complement  # noqa: F401,E501
from .fastaindex import FastaIndex, write_fai  # noqa: F401
from .predict import DuplexTable, check_loci, filter_next_loci, duplex_items  # noqa: F401

__all__ = ["FastaIndex", "write_fai", "LocusRecord", "fold_records", "header_line", "parse_header", "records_from_fasta", "write_fasta", "get_reverse_complement",
           "DuplexTable", "check_loci", "filter_next_loci", "duplex_items",
           "structures_from_result", "structures_from_result_native", "get_structures_next_extendregion", "is_stem_loop", "filter_ss",
           "has_one_good_bifurcation", "classify", "MirFold", "FoldResult", "Genome", "MirfoldError", "parse_rnalfold_input", "format_record", "convert_sequence"]
