"""sufr_b200: B200-native suffix array + LCP array construction behind the `create` interface of
TravisWheelerLab/sufr (libsufr `SufrBuilder` / `SufrBuilderArgs`, `.sufr` v6 byte layout)."""
from .builder import (BuildResult, Context, create_multi, ExtractResult, ExtractSequence, KmerSpectrum, SeedMask, SequenceFileData, SuffixArray, SufrBuilder, SufrIndex,  # noqa: F401
                      SufrBuilderArgs, SufrError, build, default_context, file_info, find_lcp_full_offset,
                      read_sequence_file)
from ._lib import MEM_DEVICE, MEM_HOST  # noqa: F401

__all__ = ["SufrBuilder", "SufrBuilderArgs", "SuffixArray", "SeedMask", "SufrError", "Context", "BuildResult",
           "build", "default_context", "read_sequence_file", "find_lcp_full_offset", "SufrIndex", "ExtractResult",
           "ExtractSequence", "file_info", "MEM_HOST", "MEM_DEVICE"]
