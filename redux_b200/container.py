"""Blocked container (SURVEY.md 8(f) rank 2).  The reference's stream is headerless (src/lib.rs:102-120:
no magic, no parameters, no length), so a batch of independently coded blocks needs an index to be decodable.
This container is NEW (no reference counterpart) and lives strictly OUTSIDE the per-block bytes: every block's
stream inside it is byte-for-byte what redux::compress() writes for that block alone.

    file    := header segment*
    header  := "RDXB" u8 version(1) u8 model_kind u8 symbol_bits u8 freq_bits u8 code_bits u8[3] zero
               u32 block_len
    segment := u32 n_blocks  u32 last_block_raw_len  u32 comp_size[n_blocks]  stream[n_blocks]
               (blocks 0..n-2 hold block_len raw bytes; a segment with n_blocks == 0 ends the file)
All integers little-endian.  Segments let a file be written and read as a stream of batches.

Version 2 stores trained start models (redux_encode_batch_models): a table of frequency rows after the header, and
the row each block starts from in its segment's index.

    header  := "RDXB" u8 version(2) u8 model_kind u8 symbol_bits u8 freq_bits u8 code_bits u8[3] zero u32 block_len
               u32 n_models  u32 freq[n_models][symbol_count]
    segment := u32 n_blocks  u32 last_block_raw_len  u32 model_index[n_blocks]  u32 comp_size[n_blocks]
               stream[n_blocks]
A row is a model's frequency vector, fresh (all ones) or trained: every entry >= 1, total <= freq_max.  Block i's
stream is compress() of the block with a model in that state.  pack / pack_stream still write version 1.
pack_models / pack_stream_models take the index from the caller, pack_auto / pack_stream_auto let the device choose it
(redux_encode_batch_select), and pack_learned / pack_stream_learned also learn the table from the first batch of
blocks (redux_build_models) before the device chooses.

Version 3 is version 2 plus the CRC-32 of every block's raw bytes (zlib's crc32, computed on the device while the
block is coded), so a reader can tell a damaged file from a good one:

    header  := "RDXB" u8 version(3) ... exactly as version 2, model table included
    segment := u32 n_blocks  u32 last_block_raw_len  u32 model_index[n_blocks]  u32 comp_size[n_blocks]
               u32 crc32[n_blocks]  stream[n_blocks]
Every writer takes checksum=False; with checksum=True it writes version 3 (pack / pack_stream with a one-row table
holding the fresh model).  unpack_stream decodes a version 3 segment only when another segment header or the end
marker follows it, and writes it only after every block of it decoded with status OK, to its expected length,
consuming exactly its stored size, to bytes whose CRC is the stored one; otherwise it raises ContainerError naming the
segment (and the block and the check)."""
import io
import struct

import numpy as np

import redux_b200 as rb

MAGIC = b"RDXB"
HEADER = struct.Struct("<4sBBBBB3xI")
MAX_MODEL_TABLE_BYTES = 256 << 20          # REDUX_MAX_MODEL_TABLE_BYTES (include/redux_b200.h)


class ContainerError(rb.InvalidInput):
    pass


def write_header(f, model, block_len):
    p = model.params
    f.write(HEADER.pack(MAGIC, 1, model.kind, p.symbol_bits, p.freq_bits, p.code_bits, block_len))


def read_header(f):
    raw = f.read(HEADER.size)
    if len(raw) != HEADER.size:
        raise ContainerError("container header truncated")
    magic, ver, kind, s, fb, c, block_len = HEADER.unpack(raw)
    if magic != MAGIC or ver != 1 or kind not in (rb.MODEL_LINEAR, rb.MODEL_TREE) or block_len == 0:
        raise ContainerError("not an RDXB v1 container")
    cls = rb.AdaptiveTreeModel if kind == rb.MODEL_TREE else rb.AdaptiveLinearModel
    return cls(rb.Parameters(s, fb, c)), block_len        # Parameters() re-validates (src/model/mod.rs:64)


def read_header_any(f):
    """Reads a version 1, 2 or 3 header.  Returns (version, models, block_len): version 1 gives one fresh model.  A
    version 2 or 3 table is checked here: ContainerError for no rows, a table over the library's cap or a row that is
    not a model's state; Eof when the file ends inside it."""
    raw = f.read(HEADER.size)
    if len(raw) != HEADER.size:
        raise ContainerError("container header truncated")      # as read_header
    magic, ver, kind, s, fb, c, block_len = HEADER.unpack(raw)
    if magic != MAGIC or ver not in (1, 2, 3) or kind not in (rb.MODEL_LINEAR, rb.MODEL_TREE) or block_len == 0:
        raise ContainerError("not an RDXB v1, v2 or v3 container")
    cls = rb.AdaptiveTreeModel if kind == rb.MODEL_TREE else rb.AdaptiveLinearModel
    params = rb.Parameters(s, fb, c)
    if ver == 1:
        return 1, [cls(params)], block_len
    head = f.read(4)
    if len(head) != 4:
        raise rb.Eof("container ended inside the model table")
    (n_models,) = struct.unpack("<I", head)
    nsym = params.symbol_count
    if n_models == 0:
        raise ContainerError("model table has no rows")
    if n_models * (nsym + 1) * 4 > MAX_MODEL_TABLE_BYTES:
        raise ContainerError("model table larger than the library takes in one call")
    body = f.read(4 * n_models * nsym)
    if len(body) != 4 * n_models * nsym:
        raise rb.Eof("container ended inside the model table")
    table = np.frombuffer(body, dtype="<u4").astype(np.uint32).reshape(n_models, nsym)
    bad = np.flatnonzero((table.min(axis=1) < 1) | (table.sum(axis=1, dtype=np.uint64) > params.freq_max))
    if bad.size:
        raise ContainerError("model row %d is not a model's frequency vector" % bad[0])
    models = []
    for row in table:
        m = cls(params)
        m.freq = row.copy()
        models.append(m)
    return ver, models, block_len


def pack_stream(fin, fout, model, block_len=65536, batch_blocks=16384, context=None, checksum=False):
    """Reads fin to the end, codes it in batches of `batch_blocks` blocks, writes the container to fout: version 1,
    or with checksum=True version 3 with a one-row table holding the fresh model.  Returns (raw_bytes,
    container_bytes)."""
    # The header records the model KIND and Parameters only, and unpack_stream() rebuilds a fresh model from it: a
    # model trained before the call would produce streams nothing in the file says how to decode.  Likewise the
    # segment index stores whole bytes per block: with symbol_bits != 8 the reference drops a trailing partial
    # symbol (src/bitio/mod.rs:94-108), so decoded lengths would not match.  Refuse both at pack time.
    if model.freq is not None:
        raise ContainerError("the container stores fresh models only (a trained model is not recorded in the header)")
    if model.params.symbol_bits != 8:
        raise ContainerError("the container stores byte-symbol streams only (symbol_bits must be 8)")
    if checksum:
        def encode(data, off, first):
            comp, coff, _, crc = (context or rb._ctx()).encode_batch_models_crc(data, off, [model], None)
            return comp, coff, np.zeros(off.size - 1, dtype=np.uint32), crc
        return _pack_stream_v2(fin, fout, [model], block_len, batch_blocks, encode, True)
    ctx = context or rb._ctx()
    write_header(fout, model, block_len)
    raw_total, out_total = 0, HEADER.size
    while True:
        chunk = fin.read(block_len * batch_blocks)
        if not chunk:
            break
        data = np.frombuffer(chunk, dtype=np.uint8)
        n = (data.size + block_len - 1) // block_len
        off = np.minimum(np.arange(n + 1, dtype=np.uint64) * np.uint64(block_len), np.uint64(data.size))
        comp, coff, _ = ctx.encode_batch(data, off, model)
        sizes = (coff[1:] - coff[:-1]).astype("<u4")
        fout.write(struct.pack("<II", n, data.size - (n - 1) * block_len))
        fout.write(sizes.tobytes())
        fout.write(comp.tobytes())
        raw_total += data.size
        out_total += 8 + sizes.nbytes + comp.size
    fout.write(struct.pack("<II", 0, 0))
    return raw_total, out_total + 8


def _pack_stream_v2(fin, fout, models, block_len, batch_blocks, encode, checksum, chunk=None):
    """Writes a version 2 (checksum: version 3) container of fin's bytes: the header and model table of `models`, then
    one segment per batch of `batch_blocks` blocks.  encode(data, offsets, first) codes a batch whose first block is
    block `first` of the input and returns (streams, stream offsets, model index, CRCs; None without checksum).
    chunk: the first batch's bytes when the caller has read them from fin already.  Returns (raw_bytes,
    container_bytes)."""
    kind, pc, table = rb._model_table(models)
    if pc.symbol_bits != 8:
        raise ContainerError("the container stores byte-symbol streams only (symbol_bits must be 8)")
    if table.shape[0] * (table.shape[1] + 1) * 4 > MAX_MODEL_TABLE_BYTES:
        raise ContainerError("model table larger than the library takes in one call")
    fout.write(HEADER.pack(MAGIC, 3 if checksum else 2, kind, pc.symbol_bits, pc.freq_bits, pc.code_bits, block_len))
    fout.write(struct.pack("<I", table.shape[0]))
    fout.write(table.astype("<u4").tobytes())
    raw_total, out_total, first = 0, HEADER.size + 4 + table.nbytes, 0
    while True:
        chunk = chunk if chunk is not None else fin.read(block_len * batch_blocks)
        if not chunk:
            break
        data = np.frombuffer(chunk, dtype=np.uint8)
        chunk = None
        n = (data.size + block_len - 1) // block_len
        off = np.minimum(np.arange(n + 1, dtype=np.uint64) * np.uint64(block_len), np.uint64(data.size))
        comp, coff, idx, crc = encode(data, off, first)
        sizes = (coff[1:] - coff[:-1]).astype("<u4")
        fout.write(struct.pack("<II", n, data.size - (n - 1) * block_len))
        fout.write(idx.astype("<u4").tobytes())
        fout.write(sizes.tobytes())
        if checksum:
            fout.write(crc.astype("<u4").tobytes())
        fout.write(comp.tobytes())
        raw_total += data.size
        out_total += 8 + 4 * n + sizes.nbytes + (4 * n if checksum else 0) + comp.size
        first += n
    fout.write(struct.pack("<II", 0, 0))
    return raw_total, out_total + 8


def pack_stream_models(fin, fout, models, block_model, block_len=65536, batch_blocks=16384, context=None,
                       checksum=False):
    """pack_stream with a start model per block, as version 2 (checksum=True: version 3): block i (counted over the
    whole input) is coded from models[block_model[i]], each model fresh or trained (one kind and one Parameters, byte
    symbols).  Raises ContainerError for an index out of range, and for a block_model shorter than the blocks of a
    batch before that batch is coded.  Returns (raw_bytes, container_bytes)."""
    models = list(models)
    rb._model_table(models)
    bm = np.ascontiguousarray(block_model, dtype=np.int64).ravel()
    if bm.size and (bm.min() < 0 or bm.max() >= len(models)):
        raise ContainerError("block_model holds an index outside the %d models" % len(models))
    bm = bm.astype(np.uint32)

    def encode(data, off, first):
        n = off.size - 1
        if first + n > bm.size:
            raise ContainerError("block_model has %d entries for at least %d blocks" % (bm.size, first + n))
        idx = bm[first:first + n]
        if checksum:
            comp, coff, _, crc = (context or rb._ctx()).encode_batch_models_crc(data, off, models, idx)
            return comp, coff, idx, crc
        comp, coff, _ = (context or rb._ctx()).encode_batch_models(data, off, models, idx)
        return comp, coff, idx, None

    return _pack_stream_v2(fin, fout, models, block_len, batch_blocks, encode, checksum)


def _select_encoder(models, context, checksum):
    """_pack_stream_v2's encode with each block's model chosen on the device (Context.encode_batch_select)."""

    def encode(data, off, first):
        if checksum:
            comp, coff, _, idx, crc = (context or rb._ctx()).encode_batch_select_crc(data, off, models)
            return comp, coff, idx, crc
        comp, coff, _, idx = (context or rb._ctx()).encode_batch_select(data, off, models)
        return comp, coff, idx, None

    return encode


def pack_stream_auto(fin, fout, models, block_len=65536, batch_blocks=16384, context=None, checksum=False):
    """pack_stream_models with each block's start model chosen on the device (Context.encode_batch_select): the model
    with the smallest estimated compressed size of the block.  Writes version 2 (checksum=True: version 3).  Returns
    (raw_bytes, container_bytes)."""
    models = list(models)
    return _pack_stream_v2(fin, fout, models, block_len, batch_blocks, _select_encoder(models, context, checksum),
                           checksum)


def pack_stream_learned(fin, fout, model, k=16, iterations=8, block_len=65536, batch_blocks=16384, context=None,
                        checksum=False):
    """pack_stream_auto with a model table learned from the data itself: the first batch of `batch_blocks` blocks is
    clustered into k groups (Context.build_models, `iterations` rounds), and every batch is then coded with each
    block's start model chosen on the device from the k + 1 models (fresh first).  model gives the kind and Parameters
    only (fresh, byte symbols).  Writes version 2 (checksum=True: version 3); unpack_stream reads it.  Returns
    (raw_bytes, container_bytes)."""
    if model.freq is not None and (np.asarray(model.freq) != 1).any():
        raise ContainerError("pack_learned learns its models: pass a fresh model for the kind and Parameters")
    if model.params.symbol_bits != 8:
        raise ContainerError("the container stores byte-symbol streams only (symbol_bits must be 8)")
    chunk = fin.read(block_len * batch_blocks)
    models = [model]
    if chunk:
        data = np.frombuffer(chunk, dtype=np.uint8)
        n = (data.size + block_len - 1) // block_len
        off = np.minimum(np.arange(n + 1, dtype=np.uint64) * np.uint64(block_len), np.uint64(data.size))
        models, _, _ = (context or rb._ctx()).build_models(data, off, model, k, iterations)

    return _pack_stream_v2(fin, fout, models, block_len, batch_blocks, _select_encoder(models, context, checksum),
                           checksum, chunk)


def check_segment(segment, status, raw_lens, lens, used, sizes, crc, stored_crc):
    """The version 3 reader's checks on one decoded segment, block by block: status OK, the expected length, bytes
    consumed equal to the stored size, the stored CRC.  Raises ContainerError naming the segment, the block and the
    first check it fails."""
    checks = (("status %s", status != rb.OK, status), ("decoded length %s", raw_lens != lens, raw_lens),
              ("consumed %s bytes of its stream", used != sizes, used), ("CRC-32 %08x", crc != stored_crc, crc))
    for i in range(len(status)):
        for what, bad, got in checks:
            if bad[i]:
                raise ContainerError("segment %d, block %d: %s, not what the container records"
                                     % (segment, i, what % (int(got[i]),)))


def unpack_stream(fin, fout, context=None):
    """Inverse of pack_stream, pack_stream_models and pack_stream_auto (versions 1, 2 and 3). Returns
    (container_bytes, raw_bytes). Raises Eof on a truncated file, with one exception: a version 3 file that ends right
    after a segment (neither the next segment's header nor the end marker follows) raises ContainerError, before that
    segment is decoded.  Each segment is checked before it is decoded, and a version 3 segment again before its bytes
    are written (check_segment)."""
    ctx = context
    ver, models, block_len = read_header_any(fin)
    consumed, raw_total, segment = HEADER.size, 0, 0
    if ver >= 2:
        consumed += 4 + 4 * len(models) * models[0].params.symbol_count
    head = None
    while True:
        head = head if head is not None else fin.read(8)
        if len(head) != 8:
            raise rb.Eof("container ended inside a segment header")
        n, last = struct.unpack("<II", head)
        head = None
        consumed += 8
        if n == 0:
            return consumed, raw_total
        if last == 0 or last > block_len:
            raise ContainerError("bad segment")
        idx = None
        if ver >= 2:
            raw_idx = fin.read(4 * n)
            if len(raw_idx) != 4 * n:
                raise rb.Eof("container ended inside a segment's model index")
            idx = np.frombuffer(raw_idx, dtype="<u4").astype(np.uint32)
            if int(idx.max()) >= len(models):
                raise ContainerError("a block names model %d of %d" % (int(idx.max()), len(models)))
            consumed += 4 * n
        raw_sizes = fin.read(4 * n)
        if len(raw_sizes) != 4 * n:
            raise rb.Eof("container ended inside a segment index")
        sizes = np.frombuffer(raw_sizes, dtype="<u4").astype(np.uint64)
        stored_crc = None
        if ver == 3:
            raw_crc = fin.read(4 * n)
            if len(raw_crc) != 4 * n:
                raise rb.Eof("container ended inside a segment's CRCs")
            stored_crc = np.frombuffer(raw_crc, dtype="<u4").astype(np.uint32)
            consumed += 4 * n
        coff = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(sizes, out=coff[1:])
        blob = fin.read(int(coff[-1]))
        if len(blob) != int(coff[-1]):
            raise rb.Eof("container ended inside a segment's streams")
        lens = np.full(n, block_len, dtype=np.uint64)
        lens[-1] = last
        roff = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(lens, out=roff[1:])
        comp = np.frombuffer(blob, dtype=np.uint8)
        if ver == 3:
            # a checksummed file is whole: the segment is followed by another one or the end marker, checked before
            # any of it is decoded or written
            head = fin.read(8)
            if len(head) != 8:
                raise ContainerError("segment %d is followed by neither a segment nor the end marker" % segment)
        ctx = ctx or rb._ctx()
        if ver == 1:
            raw, raw_lens, used, status = ctx.decode_batch(comp, coff, roff, models[0])
        elif ver == 2:
            raw, raw_lens, used, status = ctx.decode_batch_models(comp, coff, roff, models, idx)
        else:
            raw, raw_lens, used, status, crc = ctx.decode_batch_models_crc(comp, coff, roff, models, idx, check=False)
            check_segment(segment, status, raw_lens, lens, used, sizes, crc, stored_crc)
        if not (raw_lens == lens).all() or not (used == sizes).all():
            raise ContainerError("a block decoded to an unexpected length")
        fout.write(raw[: int(roff[-1])].tobytes())
        consumed += 4 * n + len(blob)
        raw_total += int(roff[-1])
        segment += 1


def pack(data, model, block_len=65536, context=None, checksum=False):
    out = io.BytesIO()
    pack_stream(io.BytesIO(bytes(data)), out, model, block_len, context=context, checksum=checksum)
    return out.getvalue()


def pack_models(data, models, block_model, block_len=65536, context=None, checksum=False):
    """pack with a start model per block (version 2, checksum=True: version 3); see pack_stream_models.  The whole
    block_model is checked against the data's block count before anything is coded."""
    data = bytes(data)
    n = (len(data) + block_len - 1) // block_len
    if len(block_model) < n:
        raise ContainerError("block_model has %d entries for %d blocks" % (len(block_model), n))
    out = io.BytesIO()
    pack_stream_models(io.BytesIO(data), out, models, block_model, block_len, context=context, checksum=checksum)
    return out.getvalue()


def pack_auto(data, models, block_len=65536, context=None, checksum=False):
    """pack with each block's start model chosen on the device (version 2, checksum=True: version 3); see
    pack_stream_auto."""
    out = io.BytesIO()
    pack_stream_auto(io.BytesIO(bytes(data)), out, models, block_len, context=context, checksum=checksum)
    return out.getvalue()


def pack_learned(data, model, k=16, iterations=8, block_len=65536, context=None, checksum=False):
    """pack with a model table learned from the data (version 2, checksum=True: version 3); see
    pack_stream_learned."""
    out = io.BytesIO()
    pack_stream_learned(io.BytesIO(bytes(data)), out, model, k, iterations, block_len, context=context,
                        checksum=checksum)
    return out.getvalue()


def unpack(blob, context=None):
    out = io.BytesIO()
    unpack_stream(io.BytesIO(bytes(blob)), out, context=context)
    return out.getvalue()
