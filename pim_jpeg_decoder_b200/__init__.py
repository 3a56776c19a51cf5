"""B200-native JPEG decode back end: a drop-in for the MCU-decode hot path of jeun-990806/pim-jpeg-decoder.

The product is ``libb200jpeg.so`` (C ABI in ``include/b200jpeg.h``, sm_100a kernels in ``csrc/``).  This Python
package is the host-side mirror of the reference's interface for that path (``Decoder.exec_mcus`` = the DPU
program, ``Decoder.decode`` = decode_Huffman_data + DPU program + BMP pixel gathering, ``decode_files`` = the
``./bin/decoder <jpeg...>`` CLI) used by the tests and the benchmark.  There is no CPU decode path.
"""
from ._lib import (BJ_ERR_ARG, BJ_ERR_CORRUPT_SCAN, BJ_ERR_CUDA, BJ_ERR_INVALID_JPEG, BJ_ERR_UNSUPPORTED, BJ_OK, BJ_OUT_BMP,  # noqa: F401
                   BJ_OUT_REF_MCUS, BJ_OUT_RGB8, BJ_SCAN_RAW, BJ_SCAN_UNSTUFFED, BatchInfo, BjError, ImageDesc, Roi, Size, lib)
from .decoder import (Batch, Decoder, Job, PinnedBuffer, decode_files, lpt_shards, parse_header, resize_plan,  # noqa: F401
                      resized_output_size, roi_output_size, scaled_output_size, shard_by_size)
