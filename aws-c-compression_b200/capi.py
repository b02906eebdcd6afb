"""ctypes bindings for include/aws/compression/*.h. Layouts mirror the C structs one for one."""
import ctypes as C
import os

import numpy as np

from . import build as _build

AWS_OP_SUCCESS = 0
AWS_OP_ERR = -1
AWS_ERROR_SHORT_BUFFER = 4
AWS_ERROR_INVALID_ARGUMENT = 34
AWS_ERROR_COMPRESSION_UNKNOWN_SYMBOL = 3072
AWS_ERROR_COMPRESSION_DEVICE_FAILURE = 3073
AWS_ERROR_COMPRESSION_INVALID_CODE_TABLE = 3074
AWS_ERROR_COMPRESSION_INVALID_PADDING = 3075
HPACK_HUFFMAN_SMALLEST, HPACK_HUFFMAN_NEVER, HPACK_HUFFMAN_ALWAYS = 0, 1, 2
# enum aws_hpack_field_kind
(HPACK_FIELD_INDEXED, HPACK_FIELD_LITERAL_INCREMENTAL, HPACK_FIELD_LITERAL_WITHOUT_INDEXING,
 HPACK_FIELD_LITERAL_NEVER_INDEXED, HPACK_FIELD_TABLE_SIZE_UPDATE, HPACK_FIELD_AUTO) = range(6)
# enum aws_qpack_field_kind
(QPACK_FIELD_INDEXED_STATIC, QPACK_FIELD_INDEXED_DYNAMIC, QPACK_FIELD_INDEXED_POST_BASE, QPACK_FIELD_NAME_REF_STATIC,
 QPACK_FIELD_NAME_REF_DYNAMIC, QPACK_FIELD_NAME_REF_POST_BASE, QPACK_FIELD_LITERAL_NAME, QPACK_FIELD_AUTO) = range(8)
# enum aws_qpack_instruction_stream, enum aws_qpack_instruction_kind
QPACK_ENCODER_STREAM, QPACK_DECODER_STREAM = 0, 1
(QPACK_INSERT_NAME_REF_STATIC, QPACK_INSERT_NAME_REF_DYNAMIC, QPACK_INSERT_LITERAL_NAME, QPACK_DUPLICATE,
 QPACK_SET_CAPACITY, QPACK_SECTION_ACKNOWLEDGMENT, QPACK_STREAM_CANCELLATION, QPACK_INSERT_COUNT_INCREMENT,
 QPACK_INSERT_AUTO) = range(9)


class CodecError(RuntimeError):
    def __init__(self, code, what):
        super().__init__("%s failed: aws error %d" % (what, code))
        self.code = code


class aws_huffman_code(C.Structure):
    _fields_ = [("pattern", C.c_uint32), ("num_bits", C.c_uint8)]


ENCODE_FN = C.CFUNCTYPE(aws_huffman_code, C.c_uint8, C.c_void_p)
DECODE_FN = C.CFUNCTYPE(C.c_uint8, C.c_uint32, C.POINTER(C.c_uint8), C.c_void_p)


# ctypes cannot RETURN a struct from a Python callback. On x86-64 SysV an 8-byte integer-class struct
# comes back in RAX, so a Python encode callback is declared as returning uint64 = pattern | bits << 32.
ENCODE_FN_PY = C.CFUNCTYPE(C.c_uint64, C.c_uint8, C.c_void_p)


class aws_huffman_symbol_coder(C.Structure):
    _fields_ = [("encode", ENCODE_FN), ("decode", DECODE_FN), ("userdata", C.c_void_p)]


class aws_huffman_encoder(C.Structure):
    _fields_ = [("coder", C.POINTER(aws_huffman_symbol_coder)), ("eos_padding", C.c_uint8),
                ("overflow_bits", aws_huffman_code)]


class aws_huffman_decoder(C.Structure):
    _fields_ = [("coder", C.POINTER(aws_huffman_symbol_coder)), ("allow_growth", C.c_bool),
                ("working_bits", C.c_uint64), ("num_bits", C.c_uint8)]


class aws_byte_cursor(C.Structure):
    _fields_ = [("len", C.c_size_t), ("ptr", C.c_void_p)]


class aws_byte_buf(C.Structure):
    _fields_ = [("len", C.c_size_t), ("buffer", C.c_void_p), ("capacity", C.c_size_t), ("allocator", C.c_void_p)]


class aws_huffman_batch(C.Structure):
    _fields_ = [
        ("n", C.c_size_t),
        ("in_", C.c_void_p),
        ("in_offsets", C.c_void_p),
        ("in_size", C.c_uint64),
        ("out", C.c_void_p),
        ("out_capacity", C.c_uint64),
        ("out_offsets", C.c_void_p),
        ("out_caps", C.c_void_p),
        ("out_lens", C.c_void_p),
        ("status", C.c_void_p),
        ("consumed", C.c_void_p),
        ("overflow_pattern", C.c_void_p),
        ("overflow_num_bits", C.c_void_p),
        ("leftover_working_bits", C.c_void_p),
        ("leftover_num_bits", C.c_void_p),
    ]


class aws_hpack_header_lists(C.Structure):
    _fields_ = [
        ("n", C.c_size_t),
        ("field_offsets", C.c_void_p),
        ("field_capacity", C.c_uint64),
        ("field_kind", C.c_void_p),
        ("field_index", C.c_void_p),
        ("never_indexed", C.c_void_p),
        ("strings", C.c_void_p),
        ("strings_capacity", C.c_uint64),
        ("string_offsets", C.c_void_p),
    ]


class aws_qpack_field_sections(C.Structure):
    _fields_ = [
        ("n", C.c_size_t),
        ("encoded_insert_count", C.c_void_p),
        ("base_sign", C.c_void_p),
        ("delta_base", C.c_void_p),
        ("field_offsets", C.c_void_p),
        ("field_capacity", C.c_uint64),
        ("field_kind", C.c_void_p),
        ("field_index", C.c_void_p),
        ("never_indexed", C.c_void_p),
        ("strings", C.c_void_p),
        ("strings_capacity", C.c_uint64),
        ("string_offsets", C.c_void_p),
    ]


class aws_qpack_instructions(C.Structure):
    _fields_ = [
        ("n", C.c_size_t),
        ("instruction_offsets", C.c_void_p),
        ("instruction_capacity", C.c_uint64),
        ("kind", C.c_void_p),
        ("index", C.c_void_p),
        ("strings", C.c_void_p),
        ("strings_capacity", C.c_uint64),
        ("string_offsets", C.c_void_p),
    ]


class aws_huffman_table_coder(C.Structure):
    _fields_ = [("coder", aws_huffman_symbol_coder), ("codes", aws_huffman_code * 256),
                ("lut_entries", C.c_void_p), ("lut_count", C.c_uint32), ("lut_root_bits", C.c_uint8)]


def python_coder(encode, decode=None):
    """A symbol coder backed by Python callables (tests only).
    encode(sym) -> (pattern, num_bits); decode(bits) -> (symbol, num_bits) or None."""
    def enc_cb(sym, _):
        pattern, nbits = encode(sym)
        return (int(pattern) & 0xFFFFFFFF) | (int(nbits) << 32)

    def dec_cb(bits, out_sym, _):
        hit = decode(bits)
        if not hit:
            return 0
        out_sym[0] = hit[0]
        return hit[1]

    enc_c = ENCODE_FN_PY(enc_cb)
    dec_c = DECODE_FN(dec_cb) if decode else C.cast(None, DECODE_FN)
    coder = aws_huffman_symbol_coder(C.cast(enc_c, ENCODE_FN), dec_c, None)
    coder._keepalive = (enc_c, dec_c)
    return coder


assert C.sizeof(aws_huffman_code) == 8 and C.sizeof(aws_huffman_symbol_coder) == 24
assert C.sizeof(aws_huffman_encoder) == 24 and C.sizeof(aws_huffman_decoder) == 32

# every symbol include/aws/compression/*.h declares (tests check the library exports them all)
EXPORTED_SYMBOLS = [
    "aws_compression_library_init", "aws_compression_library_clean_up",
    "aws_huffman_encoder_init", "aws_huffman_encoder_reset", "aws_huffman_decoder_init",
    "aws_huffman_decoder_reset", "aws_huffman_get_encoded_length", "aws_huffman_encode",
    "aws_huffman_decode", "aws_huffman_decoder_allow_growth",
    "huffman_test_transitive", "huffman_test_transitive_chunked",
    "aws_huffman_batch_ctx_new", "aws_huffman_batch_ctx_new_from_code_table", "aws_huffman_batch_ctx_destroy",
    "aws_huffman_encode_batch",
    "aws_huffman_decode_batch", "aws_huffman_encode_batch_device", "aws_huffman_decode_batch_device",
    "aws_huffman_encode_batch_resume", "aws_huffman_decode_batch_resume",
    "aws_huffman_encode_batch_resume_device", "aws_huffman_decode_batch_resume_device",
    "aws_huffman_histogram", "aws_huffman_histogram_device", "aws_huffman_code_lengths_from_counts",
    "aws_huffman_canonical_codes", "aws_huffman_code_table_from_counts", "aws_huffman_code_table_write_def",
    "aws_huffman_table_coder_init", "aws_huffman_table_coder_clean_up",
    "aws_hpack_string_encode_batch", "aws_hpack_string_decode_batch",
    "aws_hpack_string_encode_batch_device", "aws_hpack_string_decode_batch_device",
    "aws_huffman_get_encoded_length_batch", "aws_huffman_get_encoded_length_batch_device",
    "aws_huffman_encode_batch_multi", "aws_huffman_decode_batch_multi", "aws_huffman_batch_ctx_synchronize",
    "aws_huffman_batch_ctx_stream", "aws_huffman_batch_ctx_device", "aws_huffman_batch_ctx_launch_count",
    "aws_huffman_batch_plan_shards", "aws_huffman_batch_concat_offsets",
    "aws_hpack_header_block_decode_batch", "aws_hpack_header_block_encode_batch",
    "aws_hpack_header_block_decode_batch_device", "aws_hpack_header_block_encode_batch_device",
    "aws_hpack_header_block_encode_records_batch", "aws_hpack_header_block_encode_records_batch_device",
    "aws_hpack_string_encode_batch_multi", "aws_hpack_string_decode_batch_multi",
    "aws_hpack_header_block_decode_batch_multi", "aws_hpack_header_block_encode_batch_multi",
    "aws_hpack_header_block_encode_records_batch_multi",
    "aws_qpack_field_section_decode_batch", "aws_qpack_field_section_encode_batch",
    "aws_qpack_field_section_encode_records_batch", "aws_qpack_field_section_decode_batch_device",
    "aws_qpack_field_section_encode_batch_device", "aws_qpack_field_section_encode_records_batch_device",
    "aws_qpack_instruction_decode_batch", "aws_qpack_instruction_encode_batch",
    "aws_qpack_instruction_decode_batch_device", "aws_qpack_instruction_encode_batch_device",
]


def bind_streaming_api(lib):
    """Declares the reference-compatible streaming API on a CDLL (ours or the reference build)."""
    P = C.POINTER
    lib.aws_huffman_encoder_init.argtypes = [P(aws_huffman_encoder), P(aws_huffman_symbol_coder)]
    lib.aws_huffman_encoder_init.restype = None
    lib.aws_huffman_encoder_reset.argtypes = [P(aws_huffman_encoder)]
    lib.aws_huffman_encoder_reset.restype = None
    lib.aws_huffman_decoder_init.argtypes = [P(aws_huffman_decoder), P(aws_huffman_symbol_coder)]
    lib.aws_huffman_decoder_init.restype = None
    lib.aws_huffman_decoder_reset.argtypes = [P(aws_huffman_decoder)]
    lib.aws_huffman_decoder_reset.restype = None
    lib.aws_huffman_decoder_allow_growth.argtypes = [P(aws_huffman_decoder), C.c_bool]
    lib.aws_huffman_decoder_allow_growth.restype = None
    lib.aws_huffman_get_encoded_length.argtypes = [P(aws_huffman_encoder), aws_byte_cursor]
    lib.aws_huffman_get_encoded_length.restype = C.c_size_t
    lib.aws_huffman_encode.argtypes = [P(aws_huffman_encoder), P(aws_byte_cursor), P(aws_byte_buf)]
    lib.aws_huffman_encode.restype = C.c_int
    lib.aws_huffman_decode.argtypes = [P(aws_huffman_decoder), P(aws_byte_cursor), P(aws_byte_buf)]
    lib.aws_huffman_decode.restype = C.c_int
    lib.huffman_test_transitive.argtypes = [P(aws_huffman_symbol_coder), C.c_char_p, C.c_size_t, C.c_size_t,
                                            P(C.c_char_p)]
    lib.huffman_test_transitive.restype = C.c_int
    lib.huffman_test_transitive_chunked.argtypes = [P(aws_huffman_symbol_coder), C.c_char_p, C.c_size_t, C.c_size_t,
                                                    C.c_size_t, P(C.c_char_p)]
    lib.huffman_test_transitive_chunked.restype = C.c_int
    lib.aws_last_error.restype = C.c_int
    lib.aws_reset_error.restype = None
    lib.aws_error_name.argtypes = [C.c_int]
    lib.aws_error_name.restype = C.c_char_p
    lib.aws_compression_library_init.argtypes = [C.c_void_p]
    lib.aws_compression_library_init.restype = None
    lib.aws_compression_library_clean_up.restype = None
    lib.aws_default_allocator.restype = C.c_void_p
    lib.aws_byte_buf_init.argtypes = [P(aws_byte_buf), C.c_void_p, C.c_size_t]
    lib.aws_byte_buf_init.restype = C.c_int
    lib.aws_byte_buf_clean_up.argtypes = [P(aws_byte_buf)]
    lib.aws_byte_buf_clean_up.restype = None
    return lib


class Library:
    """The product library."""

    def __init__(self, path=None):
        # AWS_HUFFMAN_B200_LIB: another build of the same library (kernel A/B runs, tools/build_variant.sh)
        path = path or os.environ.get("AWS_HUFFMAN_B200_LIB") or _build.PRODUCT_LIB
        if not os.path.exists(path):
            raise FileNotFoundError(
                "%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no Python or CPU fallback for the batched codec." % path)
        self.path = path
        self.lib = bind_streaming_api(C.CDLL(path))
        L, P = self.lib, C.POINTER
        L.aws_huffman_batch_ctx_new.argtypes = [P(C.c_void_p), P(aws_huffman_symbol_coder), C.c_uint8, C.c_int]
        L.aws_huffman_batch_ctx_new.restype = C.c_int
        L.aws_huffman_batch_ctx_new_from_code_table.argtypes = [P(C.c_void_p), C.c_void_p, C.c_uint8, C.c_int]
        L.aws_huffman_batch_ctx_new_from_code_table.restype = C.c_int
        L.aws_huffman_batch_ctx_destroy.argtypes = [C.c_void_p]
        L.aws_huffman_batch_ctx_destroy.restype = None
        for name in ("aws_huffman_encode_batch", "aws_huffman_decode_batch",
                     "aws_huffman_encode_batch_resume", "aws_huffman_decode_batch_resume"):
            getattr(L, name).argtypes = [C.c_void_p, P(aws_huffman_batch)]
            getattr(L, name).restype = C.c_int
        for name in ("aws_huffman_encode_batch_device", "aws_huffman_decode_batch_device",
                     "aws_huffman_encode_batch_resume_device", "aws_huffman_decode_batch_resume_device"):
            getattr(L, name).argtypes = [C.c_void_p, P(aws_huffman_batch), C.c_void_p]
            getattr(L, name).restype = C.c_int
        L.aws_huffman_get_encoded_length_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.aws_huffman_get_encoded_length_batch.restype = C.c_int
        L.aws_huffman_get_encoded_length_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                                                 C.c_void_p]
        L.aws_huffman_get_encoded_length_batch_device.restype = C.c_int
        for name in ("aws_huffman_encode_batch_multi", "aws_huffman_decode_batch_multi"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_size_t, P(aws_huffman_batch)]
            getattr(L, name).restype = C.c_int
        L.aws_huffman_batch_ctx_synchronize.argtypes = [C.c_void_p]
        L.aws_huffman_batch_ctx_synchronize.restype = C.c_int
        L.aws_huffman_batch_ctx_stream.argtypes = [C.c_void_p]
        L.aws_huffman_batch_ctx_stream.restype = C.c_void_p
        L.aws_huffman_batch_ctx_device.argtypes = [C.c_void_p]
        L.aws_huffman_batch_ctx_device.restype = C.c_int
        L.aws_huffman_batch_ctx_launch_count.argtypes = [C.c_void_p]
        L.aws_huffman_batch_ctx_launch_count.restype = C.c_uint64
        L.aws_huffman_batch_plan_shards.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p]
        L.aws_huffman_batch_plan_shards.restype = C.c_int
        L.aws_huffman_batch_concat_offsets.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.aws_huffman_batch_concat_offsets.restype = C.c_int
        L.aws_hpack_header_block_decode_batch_device.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64,
                                                                 P(aws_hpack_header_lists), C.c_void_p, C.c_void_p]
        L.aws_hpack_header_block_encode_batch_device.argtypes = [C.c_void_p, P(aws_hpack_header_lists), C.c_uint64,
                                                                 C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p,
                                                                 C.c_void_p]
        L.aws_hpack_header_block_encode_records_batch_device.argtypes = [
            C.c_void_p, P(aws_hpack_header_lists), C.c_uint64, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p,
            C.c_void_p, C.c_void_p]
        for name in ("aws_hpack_header_block_decode_batch_device", "aws_hpack_header_block_encode_batch_device",
                     "aws_hpack_header_block_encode_records_batch_device"):
            getattr(L, name).restype = C.c_int
        # the HPACK host-pointer calls and their _multi forms (ctxs, n_ctx ahead of the same arguments)
        hpack_host = {
            "aws_hpack_string_encode_batch": [C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64,
                                              C.c_void_p],
            "aws_hpack_string_decode_batch": [C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                              C.c_void_p],
            "aws_hpack_header_block_decode_batch": [C.c_size_t, C.c_void_p, C.c_void_p, P(aws_hpack_header_lists),
                                                    C.c_void_p],
            "aws_hpack_header_block_encode_batch": [P(aws_hpack_header_lists), C.c_int, C.c_void_p, C.c_uint64,
                                                    C.c_void_p],
            "aws_hpack_header_block_encode_records_batch": [P(aws_hpack_header_lists), C.c_int, C.c_void_p, C.c_uint64,
                                                            C.c_void_p, C.c_void_p],
        }
        for name, args in hpack_host.items():
            getattr(L, name).argtypes = [C.c_void_p] + args
            getattr(L, name + "_multi").argtypes = [C.c_void_p, C.c_size_t] + args
            getattr(L, name).restype = getattr(L, name + "_multi").restype = C.c_int
        Q = P(aws_qpack_field_sections)
        qpack = {
            "aws_qpack_field_section_decode_batch": [C.c_size_t, C.c_void_p, C.c_void_p, Q, C.c_void_p],
            "aws_qpack_field_section_encode_batch": [Q, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p],
            "aws_qpack_field_section_encode_records_batch": [Q, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p],
            "aws_qpack_field_section_decode_batch_device": [C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64, Q, C.c_void_p,
                                                            C.c_void_p],
            "aws_qpack_field_section_encode_batch_device": [Q, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                                            C.c_void_p, C.c_void_p],
            "aws_qpack_field_section_encode_records_batch_device": [Q, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p,
                                                                    C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p],
            "aws_qpack_instruction_decode_batch": [C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, P(aws_qpack_instructions),
                                                   C.c_void_p, C.c_void_p],
            "aws_qpack_instruction_encode_batch": [C.c_int, P(aws_qpack_instructions), C.c_int, C.c_void_p, C.c_uint64,
                                                   C.c_void_p, C.c_void_p],
            "aws_qpack_instruction_decode_batch_device": [C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64,
                                                          P(aws_qpack_instructions), C.c_void_p, C.c_void_p, C.c_void_p],
            "aws_qpack_instruction_encode_batch_device": [C.c_int, P(aws_qpack_instructions), C.c_uint64, C.c_uint64,
                                                          C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                                          C.c_void_p],
        }
        for name, args in qpack.items():
            getattr(L, name).argtypes = [C.c_void_p] + args
            getattr(L, name).restype = C.c_int

    def last_error(self):
        return self.lib.aws_last_error()

    def plan_shards(self, in_offsets, num_shards):
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        begin = np.zeros(num_shards + 1, dtype=np.uint64)  # size_t
        rc = self.lib.aws_huffman_batch_plan_shards(in_offsets.ctypes.data, n, num_shards, begin.ctypes.data)
        if rc != 0:
            raise CodecError(self.last_error(), "aws_huffman_batch_plan_shards")
        return begin.astype(np.int64)

    def concat_offsets(self, shard_offsets):
        arrays = [np.ascontiguousarray(a, dtype=np.uint64) for a in shard_offsets]
        ptrs = (C.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
        items = np.array([len(a) - 1 for a in arrays], dtype=np.uint64)
        out = np.zeros(int(items.sum()) + 1, dtype=np.uint64)
        rc = self.lib.aws_huffman_batch_concat_offsets(ptrs, items.ctypes.data, len(arrays), out.ctypes.data)
        if rc != 0:
            raise CodecError(self.last_error(), "aws_huffman_batch_concat_offsets")
        return out


_product = None
_coders = None


class TableBuilder:
    """include/aws/compression/huffman_table_builder.h through ctypes (tests and tools)."""

    def __init__(self, library=None):
        self.library = library or product_library()
        L, P = self.library.lib, C.POINTER
        L.aws_huffman_histogram.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]
        L.aws_huffman_histogram_device.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.aws_huffman_code_lengths_from_counts.argtypes = [C.c_void_p, C.c_uint, C.c_bool, C.c_bool, C.c_void_p, P(C.c_uint8)]
        L.aws_huffman_canonical_codes.argtypes = [C.c_void_p, C.c_uint8, C.c_void_p, P(aws_huffman_code)]
        L.aws_huffman_code_table_from_counts.argtypes = [C.c_void_p, C.c_uint, C.c_bool, C.c_bool, C.c_void_p, P(aws_huffman_code)]
        L.aws_huffman_code_table_write_def.argtypes = [C.c_void_p, C.c_char_p]
        L.aws_huffman_table_coder_init.argtypes = [P(aws_huffman_table_coder), C.c_void_p]
        L.aws_huffman_table_coder_clean_up.argtypes = [P(aws_huffman_table_coder)]
        L.aws_huffman_table_coder_clean_up.restype = None

    def _check(self, rc, what):
        if rc != 0:
            raise CodecError(self.library.last_error(), what)

    def histogram(self, data, device=0):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        counts = np.zeros(256, dtype=np.uint64)
        self._check(self.library.lib.aws_huffman_histogram(device, data.ctypes.data, len(data), counts.ctypes.data),
                    "aws_huffman_histogram")
        return counts

    def histogram_device(self, tensor, counts_tensor, stream=None):
        self._check(self.library.lib.aws_huffman_histogram_device(tensor.data_ptr(), tensor.numel(), counts_tensor.data_ptr(),
                                                                  stream or 0), "aws_huffman_histogram_device")

    def lengths(self, counts, max_bits=32, cover_all=True, reserve_eos=False):
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        lens = np.zeros(256, dtype=np.uint8)
        eos = C.c_uint8(0)
        self._check(self.library.lib.aws_huffman_code_lengths_from_counts(counts.ctypes.data, max_bits, cover_all, reserve_eos,
                                                                          lens.ctypes.data, C.byref(eos)),
                    "aws_huffman_code_lengths_from_counts")
        return lens, eos.value

    def codes(self, counts, max_bits=32, cover_all=True, reserve_eos=False):
        """Returns (aws_huffman_code[256] ctypes array, eos aws_huffman_code)."""
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        table = (aws_huffman_code * 256)()
        eos = aws_huffman_code()
        self._check(self.library.lib.aws_huffman_code_table_from_counts(counts.ctypes.data, max_bits, cover_all, reserve_eos,
                                                                        C.cast(table, C.c_void_p), C.byref(eos)),
                    "aws_huffman_code_table_from_counts")
        return table, eos

    def canonical(self, lengths, eos_length=0):
        lengths = np.ascontiguousarray(lengths, dtype=np.uint8)
        table = (aws_huffman_code * 256)()
        eos = aws_huffman_code()
        self._check(self.library.lib.aws_huffman_canonical_codes(lengths.ctypes.data, eos_length, C.cast(table, C.c_void_p),
                                                                 C.byref(eos)), "aws_huffman_canonical_codes")
        return table, eos

    def write_def(self, table, path):
        self._check(self.library.lib.aws_huffman_code_table_write_def(C.cast(table, C.c_void_p), path.encode()),
                    "aws_huffman_code_table_write_def")

    def table_coder(self, table):
        coder = aws_huffman_table_coder()
        self._check(self.library.lib.aws_huffman_table_coder_init(C.byref(coder), C.cast(table, C.c_void_p)),
                    "aws_huffman_table_coder_init")
        return coder

    def table_coder_clean_up(self, coder):
        self.library.lib.aws_huffman_table_coder_clean_up(C.byref(coder))


def product_library():
    global _product
    if _product is None:
        _product = Library()
    return _product


class CodersLibrary:
    """Coders emitted by OUR generator: hpack and (from the golden fixture) the reference test table."""

    def __init__(self, path=None):
        path = path or _build.CODERS_LIB
        if not os.path.exists(path):
            raise FileNotFoundError("%s is missing: run __graft_entry__.build()" % path)
        self.lib = C.CDLL(path)

    def coder(self, name):
        fn = getattr(self.lib, name + "_get_coder")
        fn.restype = C.POINTER(aws_huffman_symbol_coder)
        return fn()

    def code_table_pointer(self, name):
        fn = getattr(self.lib, name + "_get_code_table")
        fn.restype = C.POINTER(aws_huffman_code * 256)
        return fn()

    def code_table(self, name):
        fn = getattr(self.lib, name + "_get_code_table")
        fn.restype = C.POINTER(aws_huffman_code * 256)
        table = fn().contents
        return (np.array([c.pattern for c in table], dtype=np.uint32),
                np.array([c.num_bits for c in table], dtype=np.uint8))


def coders_library():
    global _coders
    if _coders is None:
        _coders = CodersLibrary()
    return _coders


def _ptr(x):
    """Address of a numpy array / torch tensor / None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return x.data_ptr()  # torch tensor (host or device)


class BatchContext:
    """aws_huffman_batch_ctx for one (coder, eos_padding, device)."""

    def __init__(self, coder, eos_padding=0xFF, device=0, library=None, code_table=None):
        """`coder`: a pointer to aws_huffman_symbol_coder, or None with `code_table` = pointer to 256
        aws_huffman_code entries (aws_huffman_batch_ctx_new_from_code_table: no callbacks)."""
        self.library = library or product_library()
        self._keep = coder  # callbacks must stay alive while the C side probes them
        handle = C.c_void_p()
        if code_table is not None:
            rc = self.library.lib.aws_huffman_batch_ctx_new_from_code_table(
                C.byref(handle), C.cast(code_table, C.c_void_p), eos_padding, device)
            if rc != 0:
                raise CodecError(self.library.last_error(), "aws_huffman_batch_ctx_new_from_code_table")
        else:
            coder_ptr = coder if not isinstance(coder, aws_huffman_symbol_coder) else C.pointer(coder)
            rc = self.library.lib.aws_huffman_batch_ctx_new(C.byref(handle), coder_ptr, eos_padding, device)
            if rc != 0:
                raise CodecError(self.library.last_error(), "aws_huffman_batch_ctx_new")
        self.handle = handle
        self.device = device

    def close(self):
        if getattr(self, "handle", None):
            self.library.lib.aws_huffman_batch_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return self.library.lib.aws_huffman_batch_ctx_stream(self.handle)

    @property
    def launch_count(self):
        return int(self.library.lib.aws_huffman_batch_ctx_launch_count(self.handle))

    def synchronize(self):
        if self.library.lib.aws_huffman_batch_ctx_synchronize(self.handle) != 0:
            raise CodecError(self.library.last_error(), "aws_huffman_batch_ctx_synchronize")

    def _call(self, fn_name, n, arrays, out_capacity, stream=None, in_size=0):
        b = aws_huffman_batch()
        b.n = n
        b.in_size = in_size
        b.out_capacity = out_capacity
        for key, value in arrays.items():
            setattr(b, key, _ptr(value))
        fn = getattr(self.library.lib, fn_name)
        rc = fn(self.handle, C.byref(b)) if stream is None else fn(self.handle, C.byref(b), stream)
        if rc != 0:
            raise CodecError(self.library.last_error(), fn_name)

    # ---- host-buffer entry points (numpy in, numpy out) ----
    def _host(self, encode, data, in_offsets, out_capacity, out_offsets=None, out_caps=None, out=None, extras=True,
              state=None):
        """state = (overflow_pattern, overflow_num_bits) resp. (leftover_working_bits, leftover_num_bits) of the
        previous call: the *_resume entry points (the arrays come back updated in the result)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        slotted = out_caps is not None
        res = {
            "out": out if out is not None else np.zeros(max(int(out_capacity), 1), dtype=np.uint8),
            "out_offsets": (np.ascontiguousarray(out_offsets, dtype=np.uint64) if slotted
                            else np.zeros(n + 1, dtype=np.uint64)),
            "out_lens": np.zeros(n, dtype=np.uint64),
            "status": np.zeros(n, dtype=np.int32),
            "consumed": np.zeros(n, dtype=np.uint64),
        }
        if not extras:  # only payload, offsets and status (what a throughput-minded caller asks for)
            del res["out_lens"], res["consumed"]
        elif encode:
            res["overflow_pattern"] = np.zeros(n, dtype=np.uint32)
            res["overflow_num_bits"] = np.zeros(n, dtype=np.uint8)
        else:
            res["leftover_working_bits"] = np.zeros(n, dtype=np.uint64)
            res["leftover_num_bits"] = np.zeros(n, dtype=np.uint8)
        if state is not None:
            if encode:
                res["overflow_pattern"] = np.array(state[0], dtype=np.uint32)
                res["overflow_num_bits"] = np.array(state[1], dtype=np.uint8)
            else:
                res["leftover_working_bits"] = np.array(state[0], dtype=np.uint64)
                res["leftover_num_bits"] = np.array(state[1], dtype=np.uint8)
        arrays = dict(res)
        arrays["in_"] = data
        arrays["in_offsets"] = in_offsets
        if slotted:
            arrays["out_caps"] = np.ascontiguousarray(out_caps, dtype=np.uint64)
        name = "aws_huffman_encode_batch" if encode else "aws_huffman_decode_batch"
        self._call(name + ("_resume" if state is not None else ""), n, arrays, int(out_capacity))
        return res

    # ---- HPACK string literals (hpack_string_batch.h), host buffers ----
    def hpack_encode_strings(self, data, in_offsets, out_capacity, mode=HPACK_HUFFMAN_SMALLEST):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        res = {"out": np.zeros(max(int(out_capacity), 1), dtype=np.uint8), "out_offsets": np.zeros(n + 1, dtype=np.uint64)}
        fn = self.library.lib.aws_hpack_string_encode_batch
        fn.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]
        fn.restype = C.c_int
        rc = fn(self.handle, n, data.ctypes.data, in_offsets.ctypes.data, mode, res["out"].ctypes.data, int(out_capacity),
                res["out_offsets"].ctypes.data)
        if rc != 0:
            err = CodecError(self.library.last_error(), "aws_hpack_string_encode_batch")
            err.result = res
            raise err
        return res

    def hpack_decode_strings(self, data, in_offsets, out_capacity):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        res = {"out": np.zeros(max(int(out_capacity), 1), dtype=np.uint8), "out_offsets": np.zeros(n + 1, dtype=np.uint64),
               "status": np.zeros(n, dtype=np.int32)}
        fn = self.library.lib.aws_hpack_string_decode_batch
        fn.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        fn.restype = C.c_int
        rc = fn(self.handle, n, data.ctypes.data, in_offsets.ctypes.data, res["out"].ctypes.data, int(out_capacity),
                res["out_offsets"].ctypes.data, res["status"].ctypes.data)
        if rc != 0:
            err = CodecError(self.library.last_error(), "aws_hpack_string_decode_batch")
            err.result = res
            raise err
        return res

    def hpack_device(self, encode, n, in_, in_offsets, in_size, out, out_capacity, out_offsets, status=None, mode=0, stream=None):
        L = self.library.lib
        if encode:
            fn = L.aws_hpack_string_encode_batch_device
            fn.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                           C.c_void_p, C.c_void_p]
            rc = fn(self.handle, n, _ptr(in_), _ptr(in_offsets), int(in_size), mode, _ptr(out), int(out_capacity),
                    _ptr(out_offsets), stream or 0)
        else:
            fn = L.aws_hpack_string_decode_batch_device
            fn.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                           C.c_void_p, C.c_void_p]
            rc = fn(self.handle, n, _ptr(in_), _ptr(in_offsets), int(in_size), _ptr(out), int(out_capacity),
                    _ptr(out_offsets), _ptr(status), stream or 0)
        if rc != 0:
            raise CodecError(self.library.last_error(), "aws_hpack_string_%s_batch_device" % ("encode" if encode else "decode"))

    # ---- HPACK header blocks (hpack_header_block_batch.h) ----
    def _blocks_call(self, fn_name, *args):
        rc = getattr(self.library.lib, fn_name)(self.handle, *args)
        if rc != 0:
            raise CodecError(self.library.last_error(), fn_name)

    def hpack_decode_blocks(self, data, in_offsets, field_capacity=None, strings_capacity=None):
        """Host buffers. Capacities default to the documented bounds (in_size fields, 28 * in_size octets). On
        failure the CodecError carries the arrays as `result` (offsets are complete on AWS_ERROR_SHORT_BUFFER)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        in_size = int(in_offsets[-1])
        field_capacity = in_size if field_capacity is None else int(field_capacity)
        strings_capacity = 28 * in_size if strings_capacity is None else int(strings_capacity)
        res = {"field_offsets": np.zeros(n + 1, dtype=np.uint64), "field_kind": np.zeros(max(field_capacity, 1), np.uint8),
               "field_index": np.zeros(max(field_capacity, 1), np.uint64),
               "strings": np.zeros(max(strings_capacity, 1), np.uint8),
               "string_offsets": np.zeros(2 * field_capacity + 1, np.uint64), "status": np.zeros(n, np.int32)}
        lists = aws_hpack_header_lists(n, _ptr(res["field_offsets"]), field_capacity, _ptr(res["field_kind"]),
                                       _ptr(res["field_index"]), None, _ptr(res["strings"]), strings_capacity,
                                       _ptr(res["string_offsets"]))
        try:
            self._blocks_call("aws_hpack_header_block_decode_batch", n, _ptr(data), _ptr(in_offsets), C.byref(lists),
                              _ptr(res["status"]))
        except CodecError as err:
            err.result = res
            raise
        return res

    def hpack_encode_blocks(self, field_offsets, strings, string_offsets, out_capacity, mode=HPACK_HUFFMAN_SMALLEST,
                            never_indexed=None):
        """Host buffers: header lists in, header blocks out ({"out", "out_offsets"})."""
        field_offsets = np.ascontiguousarray(field_offsets, dtype=np.uint64)
        strings = np.ascontiguousarray(strings, dtype=np.uint8)
        string_offsets = np.ascontiguousarray(string_offsets, dtype=np.uint64)
        if never_indexed is not None:
            never_indexed = np.ascontiguousarray(never_indexed, dtype=np.uint8)
        n = len(field_offsets) - 1
        res = {"out": np.zeros(max(int(out_capacity), 1), dtype=np.uint8), "out_offsets": np.zeros(n + 1, dtype=np.uint64)}
        lists = aws_hpack_header_lists(n, _ptr(field_offsets), 0, None, None, _ptr(never_indexed), _ptr(strings), 0,
                                       _ptr(string_offsets))
        try:
            self._blocks_call("aws_hpack_header_block_encode_batch", C.byref(lists), mode, _ptr(res["out"]),
                              int(out_capacity), _ptr(res["out_offsets"]))
        except CodecError as err:
            err.result = res
            raise
        return res

    def hpack_encode_records(self, field_offsets, field_kind, field_index, strings, string_offsets, out_capacity,
                             mode=HPACK_HUFFMAN_SMALLEST, never_indexed=None):
        """Host buffers: field records (the decoder's, or the caller's own) in, header blocks out ({"out",
        "out_offsets", "status"}). On failure the CodecError carries them as `result`."""
        field_offsets = np.ascontiguousarray(field_offsets, dtype=np.uint64)
        field_kind = np.ascontiguousarray(field_kind, dtype=np.uint8)
        field_index = np.ascontiguousarray(field_index, dtype=np.uint64)
        strings = np.ascontiguousarray(strings, dtype=np.uint8)
        string_offsets = np.ascontiguousarray(string_offsets, dtype=np.uint64)
        if never_indexed is not None:
            never_indexed = np.ascontiguousarray(never_indexed, dtype=np.uint8)
        n = len(field_offsets) - 1
        res = {"out": np.zeros(max(int(out_capacity), 1), dtype=np.uint8), "out_offsets": np.zeros(n + 1, dtype=np.uint64),
               "status": np.full(n, -1, dtype=np.int32)}
        lists = aws_hpack_header_lists(n, _ptr(field_offsets), 0, _ptr(field_kind), _ptr(field_index), _ptr(never_indexed),
                                       _ptr(strings), 0, _ptr(string_offsets))
        try:
            self._blocks_call("aws_hpack_header_block_encode_records_batch", C.byref(lists), mode, _ptr(res["out"]),
                              int(out_capacity), _ptr(res["out_offsets"]), _ptr(res["status"]))
        except CodecError as err:
            err.result = res
            raise
        return res

    def hpack_decode_blocks_device(self, n, in_, in_offsets, in_size, field_offsets, field_kind, field_index, strings,
                                   string_offsets, status=None, stream=None):
        """Torch CUDA tensors; capacities are the tensors' sizes (string_offsets: 2 * field_capacity + 1)."""
        field_capacity = (string_offsets.numel() - 1) // 2
        lists = aws_hpack_header_lists(n, _ptr(field_offsets), field_capacity, _ptr(field_kind), _ptr(field_index), None,
                                       _ptr(strings), strings.numel(), _ptr(string_offsets))
        self._blocks_call("aws_hpack_header_block_decode_batch_device", n, _ptr(in_), _ptr(in_offsets), int(in_size),
                          C.byref(lists), _ptr(status), stream or 0)

    def hpack_encode_blocks_device(self, n, field_offsets, num_fields, strings, string_offsets, strings_size, out,
                                   out_offsets, mode=HPACK_HUFFMAN_SMALLEST, never_indexed=None, stream=None):
        lists = aws_hpack_header_lists(n, _ptr(field_offsets), 0, None, None, _ptr(never_indexed), _ptr(strings), 0,
                                       _ptr(string_offsets))
        self._blocks_call("aws_hpack_header_block_encode_batch_device", C.byref(lists), int(num_fields),
                          int(strings_size), mode, _ptr(out), out.numel(), _ptr(out_offsets), stream or 0)

    def hpack_encode_records_device(self, n, field_offsets, num_fields, field_kind, field_index, strings, string_offsets,
                                    strings_size, out, out_offsets, status=None, mode=HPACK_HUFFMAN_SMALLEST,
                                    never_indexed=None, out_capacity=None, stream=None):
        """Torch CUDA tensors; out_capacity defaults to out.numel()."""
        lists = aws_hpack_header_lists(n, _ptr(field_offsets), 0, _ptr(field_kind), _ptr(field_index), _ptr(never_indexed),
                                       _ptr(strings), 0, _ptr(string_offsets))
        self._blocks_call("aws_hpack_header_block_encode_records_batch_device", C.byref(lists), int(num_fields),
                          int(strings_size), mode, _ptr(out), out.numel() if out_capacity is None else int(out_capacity),
                          _ptr(out_offsets), _ptr(status), stream or 0)

    # ---- QPACK field sections (qpack_field_section_batch.h) ----
    def qpack_decode_sections(self, data, in_offsets, field_capacity=None, strings_capacity=None):
        """Host buffers. Capacities default to the documented bounds (in_size fields, 69 * in_size octets). On
        failure the CodecError carries the arrays as `result` (offsets are complete on AWS_ERROR_SHORT_BUFFER)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        in_size = int(in_offsets[-1])
        field_capacity = in_size if field_capacity is None else int(field_capacity)
        strings_capacity = 69 * in_size if strings_capacity is None else int(strings_capacity)
        res = {"encoded_insert_count": np.zeros(n, np.uint64), "base_sign": np.zeros(n, np.uint8),
               "delta_base": np.zeros(n, np.uint64), "field_offsets": np.zeros(n + 1, dtype=np.uint64),
               "field_kind": np.zeros(max(field_capacity, 1), np.uint8),
               "field_index": np.zeros(max(field_capacity, 1), np.uint64),
               "never_indexed": np.zeros(max(field_capacity, 1), np.uint8),
               "strings": np.zeros(max(strings_capacity, 1), np.uint8),
               "string_offsets": np.zeros(2 * field_capacity + 1, np.uint64), "status": np.zeros(n, np.int32)}
        sections = aws_qpack_field_sections(
            n, _ptr(res["encoded_insert_count"]), _ptr(res["base_sign"]), _ptr(res["delta_base"]),
            _ptr(res["field_offsets"]), field_capacity, _ptr(res["field_kind"]), _ptr(res["field_index"]),
            _ptr(res["never_indexed"]), _ptr(res["strings"]), strings_capacity, _ptr(res["string_offsets"]))
        try:
            self._blocks_call("aws_qpack_field_section_decode_batch", n, _ptr(data), _ptr(in_offsets), C.byref(sections),
                              _ptr(res["status"]))
        except CodecError as err:
            err.result = res
            raise
        return res

    def qpack_encode_sections(self, field_offsets, strings, string_offsets, out_capacity, mode=HPACK_HUFFMAN_SMALLEST,
                              never_indexed=None, records=None):
        """Host buffers: header lists in, field sections out ({"out", "out_offsets"}, and "status" for records).
        records = (encoded_insert_count, base_sign, delta_base, field_kind, field_index): the records encoder
        (aws_qpack_field_section_encode_records_batch); None: the stateless one. On failure the CodecError carries
        the arrays as `result`."""
        field_offsets = np.ascontiguousarray(field_offsets, dtype=np.uint64)
        strings = np.ascontiguousarray(strings, dtype=np.uint8)
        string_offsets = np.ascontiguousarray(string_offsets, dtype=np.uint64)
        if never_indexed is not None:
            never_indexed = np.ascontiguousarray(never_indexed, dtype=np.uint8)
        n = len(field_offsets) - 1
        res = {"out": np.zeros(max(int(out_capacity), 1), dtype=np.uint8), "out_offsets": np.zeros(n + 1, dtype=np.uint64)}
        prefix, kind, index = (None, None, None), None, None
        if records is not None:
            eic, sign, delta, kind, index = records
            prefix = (np.ascontiguousarray(eic, dtype=np.uint64), np.ascontiguousarray(sign, dtype=np.uint8),
                      np.ascontiguousarray(delta, dtype=np.uint64))
            kind = np.ascontiguousarray(kind, dtype=np.uint8)
            index = np.ascontiguousarray(index, dtype=np.uint64)
            res["status"] = np.full(n, -1, dtype=np.int32)
        sections = aws_qpack_field_sections(n, *[_ptr(a) for a in prefix], _ptr(field_offsets), 0, _ptr(kind), _ptr(index),
                                            _ptr(never_indexed), _ptr(strings), 0, _ptr(string_offsets))
        try:
            if records is None:
                self._blocks_call("aws_qpack_field_section_encode_batch", C.byref(sections), mode, _ptr(res["out"]),
                                  int(out_capacity), _ptr(res["out_offsets"]))
            else:
                self._blocks_call("aws_qpack_field_section_encode_records_batch", C.byref(sections), mode,
                                  _ptr(res["out"]), int(out_capacity), _ptr(res["out_offsets"]), _ptr(res["status"]))
        except CodecError as err:
            err.result = res
            raise
        return res

    def qpack_decode_sections_device(self, n, in_, in_offsets, in_size, encoded_insert_count, base_sign, delta_base,
                                     field_offsets, field_kind, field_index, never_indexed, strings, string_offsets,
                                     status=None, stream=None, field_capacity=None, strings_capacity=None):
        """Device pointers (torch CUDA tensors, or objects with data_ptr()); capacities default to the tensors' sizes
        (field_capacity: (string_offsets.numel() - 1) // 2)."""
        field_capacity = (string_offsets.numel() - 1) // 2 if field_capacity is None else int(field_capacity)
        strings_capacity = strings.numel() if strings_capacity is None else int(strings_capacity)
        sections = aws_qpack_field_sections(n, _ptr(encoded_insert_count), _ptr(base_sign), _ptr(delta_base),
                                            _ptr(field_offsets), field_capacity, _ptr(field_kind), _ptr(field_index),
                                            _ptr(never_indexed), _ptr(strings), strings_capacity, _ptr(string_offsets))
        self._blocks_call("aws_qpack_field_section_decode_batch_device", n, _ptr(in_), _ptr(in_offsets), int(in_size),
                          C.byref(sections), _ptr(status), stream or 0)

    def qpack_encode_sections_device(self, n, field_offsets, num_fields, strings, string_offsets, strings_size, out,
                                     out_offsets, mode=HPACK_HUFFMAN_SMALLEST, never_indexed=None, records=None,
                                     status=None, out_capacity=None, stream=None):
        """Device pointers; records = (encoded_insert_count, base_sign, delta_base, field_kind, field_index) selects
        the records encoder. out_capacity defaults to out.numel()."""
        prefix, kind, index = (None, None, None), None, None
        if records is not None:
            prefix, (kind, index) = records[:3], records[3:]
        sections = aws_qpack_field_sections(n, *[_ptr(a) for a in prefix], _ptr(field_offsets), 0, _ptr(kind), _ptr(index),
                                            _ptr(never_indexed), _ptr(strings), 0, _ptr(string_offsets))
        cap = out.numel() if out_capacity is None else int(out_capacity)
        if records is None:
            self._blocks_call("aws_qpack_field_section_encode_batch_device", C.byref(sections), int(num_fields),
                              int(strings_size), mode, _ptr(out), cap, _ptr(out_offsets), stream or 0)
        else:
            self._blocks_call("aws_qpack_field_section_encode_records_batch_device", C.byref(sections), int(num_fields),
                              int(strings_size), mode, _ptr(out), cap, _ptr(out_offsets), _ptr(status), stream or 0)

    # ---- QPACK encoder- and decoder-stream instructions (qpack_instruction_batch.h) ----
    def qpack_decode_instructions(self, which, data, in_offsets, instruction_capacity=None, strings_capacity=None):
        """Host buffers. Capacities default to the documented bounds (in_size instructions, 14 * in_size octets). On
        failure the CodecError carries the arrays as `result` (offsets, consumed and status are complete on
        AWS_ERROR_SHORT_BUFFER)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        in_size = int(in_offsets[-1])
        cap = in_size if instruction_capacity is None else int(instruction_capacity)
        strings_capacity = 14 * in_size if strings_capacity is None else int(strings_capacity)
        res = {"instruction_offsets": np.zeros(n + 1, dtype=np.uint64), "kind": np.zeros(max(cap, 1), np.uint8),
               "index": np.zeros(max(cap, 1), np.uint64), "strings": np.zeros(max(strings_capacity, 1), np.uint8),
               "string_offsets": np.zeros(2 * cap + 1, np.uint64), "consumed": np.zeros(n, np.uint64),
               "status": np.zeros(n, np.int32)}
        instr = aws_qpack_instructions(n, _ptr(res["instruction_offsets"]), cap, _ptr(res["kind"]), _ptr(res["index"]),
                                       _ptr(res["strings"]), strings_capacity, _ptr(res["string_offsets"]))
        try:
            self._blocks_call("aws_qpack_instruction_decode_batch", which, n, _ptr(data), _ptr(in_offsets),
                              C.byref(instr), _ptr(res["consumed"]), _ptr(res["status"]))
        except CodecError as err:
            err.result = res
            raise
        return res

    def qpack_encode_instructions(self, which, instruction_offsets, kind, index, strings, string_offsets, out_capacity,
                                  mode=HPACK_HUFFMAN_SMALLEST):
        """Host buffers: instruction records in, chunks of the stream `which` out ({"out", "out_offsets", "status"}).
        On failure the CodecError carries them as `result`."""
        instruction_offsets = np.ascontiguousarray(instruction_offsets, dtype=np.uint64)
        kind = np.ascontiguousarray(kind, dtype=np.uint8)
        index = np.ascontiguousarray(index, dtype=np.uint64)
        strings = np.ascontiguousarray(strings, dtype=np.uint8)
        string_offsets = np.ascontiguousarray(string_offsets, dtype=np.uint64)
        n = len(instruction_offsets) - 1
        res = {"out": np.zeros(max(int(out_capacity), 1), dtype=np.uint8), "out_offsets": np.zeros(n + 1, dtype=np.uint64),
               "status": np.full(n, -1, dtype=np.int32)}
        instr = aws_qpack_instructions(n, _ptr(instruction_offsets), 0, _ptr(kind), _ptr(index), _ptr(strings), 0,
                                       _ptr(string_offsets))
        try:
            self._blocks_call("aws_qpack_instruction_encode_batch", which, C.byref(instr), mode, _ptr(res["out"]),
                              int(out_capacity), _ptr(res["out_offsets"]), _ptr(res["status"]))
        except CodecError as err:
            err.result = res
            raise
        return res

    def qpack_decode_instructions_device(self, which, n, in_, in_offsets, in_size, instruction_offsets, kind, index,
                                         strings, string_offsets, consumed, status=None, stream=None,
                                         instruction_capacity=None, strings_capacity=None):
        """Device pointers (torch CUDA tensors, or objects with data_ptr()); capacities default to the tensors' sizes
        (instruction_capacity: (string_offsets.numel() - 1) // 2; strings None: capacity 0)."""
        cap = (string_offsets.numel() - 1) // 2 if instruction_capacity is None else int(instruction_capacity)
        if strings_capacity is None:
            strings_capacity = strings.numel() if strings is not None else 0
        instr = aws_qpack_instructions(n, _ptr(instruction_offsets), cap, _ptr(kind), _ptr(index), _ptr(strings),
                                       int(strings_capacity), _ptr(string_offsets))
        self._blocks_call("aws_qpack_instruction_decode_batch_device", which, n, _ptr(in_), _ptr(in_offsets),
                          int(in_size), C.byref(instr), _ptr(consumed), _ptr(status), stream or 0)

    def qpack_encode_instructions_device(self, which, n, instruction_offsets, num_instructions, kind, index, strings,
                                         string_offsets, strings_size, out, out_offsets, status=None,
                                         mode=HPACK_HUFFMAN_SMALLEST, out_capacity=None, stream=None):
        """Device pointers; out_capacity defaults to out.numel()."""
        instr = aws_qpack_instructions(n, _ptr(instruction_offsets), 0, _ptr(kind), _ptr(index), _ptr(strings), 0,
                                       _ptr(string_offsets))
        cap = out.numel() if out_capacity is None else int(out_capacity)
        self._blocks_call("aws_qpack_instruction_encode_batch_device", which, C.byref(instr), int(num_instructions),
                          int(strings_size), mode, _ptr(out), cap, _ptr(out_offsets), _ptr(status), stream or 0)

    def encode(self, data, in_offsets, out_capacity, **kw):
        return self._host(True, data, in_offsets, out_capacity, **kw)

    def decode(self, data, in_offsets, out_capacity, **kw):
        return self._host(False, data, in_offsets, out_capacity, **kw)

    def encoded_lengths(self, data, in_offsets):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
        n = len(in_offsets) - 1
        lens = np.zeros(n, dtype=np.uint64)
        rc = self.library.lib.aws_huffman_get_encoded_length_batch(
            self.handle, data.ctypes.data, in_offsets.ctypes.data, n, lens.ctypes.data)
        if rc != 0:
            raise CodecError(self.library.last_error(), "aws_huffman_get_encoded_length_batch")
        return lens

    def encoded_lengths_device(self, n, in_, in_offsets, lens, stream=None):
        rc = self.library.lib.aws_huffman_get_encoded_length_batch_device(
            self.handle, _ptr(in_), _ptr(in_offsets), n, _ptr(lens), stream or 0)
        if rc != 0:
            raise CodecError(self.library.last_error(), "aws_huffman_get_encoded_length_batch_device")

    # ---- device-buffer entry points (torch CUDA tensors; enqueued on `stream`) ----
    def encode_device(self, n, arrays, in_size, out_capacity, stream=None):
        self._call("aws_huffman_encode_batch_device", n, arrays, int(out_capacity), stream=stream or 0,
                   in_size=int(in_size))

    def decode_device(self, n, arrays, in_size, out_capacity, stream=None):
        self._call("aws_huffman_decode_batch_device", n, arrays, int(out_capacity), stream=stream or 0,
                   in_size=int(in_size))


def run_multi(contexts, encode, data, in_offsets, out_capacity):
    """aws_huffman_encode_batch_multi / aws_huffman_decode_batch_multi: one packed batch over several contexts
    (host buffers, numpy in / numpy out)."""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    in_offsets = np.ascontiguousarray(in_offsets, dtype=np.uint64)
    n = len(in_offsets) - 1
    res = {"out": np.zeros(max(int(out_capacity), 1), dtype=np.uint8), "out_offsets": np.zeros(n + 1, dtype=np.uint64),
           "out_lens": np.zeros(n, dtype=np.uint64), "status": np.zeros(n, dtype=np.int32),
           "consumed": np.zeros(n, dtype=np.uint64)}
    b = aws_huffman_batch()
    b.n = n
    b.in_size = int(in_offsets[n]) if n else 0
    b.out_capacity = int(out_capacity)
    b.in_ = _ptr(data)
    b.in_offsets = _ptr(in_offsets)
    for key, value in res.items():
        setattr(b, key, _ptr(value))
    lib = contexts[0].library
    handles = (C.c_void_p * len(contexts))(*[c.handle for c in contexts])
    fn = lib.lib.aws_huffman_encode_batch_multi if encode else lib.lib.aws_huffman_decode_batch_multi
    rc = fn(handles, len(contexts), C.byref(b))
    if rc != 0:
        raise CodecError(lib.last_error(), "aws_huffman_%s_batch_multi" % ("encode" if encode else "decode"))
    return res


def hpack_host_call(target, name, *args, n_ctx=None, library=None):
    """One HPACK host-pointer entry point, `name` as the single-context call is named (e.g.
    "aws_hpack_header_block_decode_batch"), with the raw arguments that follow the context: on one BatchContext, or its
    _multi form when `target` is a list of BatchContexts (None entries are NULL contexts; target None is a NULL array,
    of n_ctx entries). Returns 0, or the error code the call raised."""
    lib = library or (target.library if isinstance(target, BatchContext) else product_library())
    if isinstance(target, BatchContext):
        rc = getattr(lib.lib, name)(target.handle, *args)
    else:
        handles = None if target is None else (C.c_void_p * max(len(target), 1))(
            *[c.handle if c is not None else None for c in target])
        rc = getattr(lib.lib, name + "_multi")(handles, len(target) if n_ctx is None else n_ctx, *args)
    return 0 if rc == 0 else lib.last_error()
