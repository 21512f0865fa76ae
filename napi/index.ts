// index.ts -- the reference's public object (src/index.ts:8-12) over the B200 addon.
// NOT COMPILED IN THIS IMAGE (no Node / tsc). Signatures equal the reference's; bodies only marshal.
// The tested equivalent is zlib.ts_b200/api.py (same C ABI, same glue).
/* eslint-disable @typescript-eslint/no-var-requires */
const native = require('./build/Release/zlibts_b200.node');

export enum CompressionType { NONE = 0, FIXED = 1, DYNAMIC = 2, RESERVED = 3 }      // src/RawDeflate.ts:12-17
export enum BufferType { BLOCK = 0, ADAPTIVE = 1 }                                   // src/RawInflate.ts:5-8
export interface RawDeflateOptions { lazy?: number; compressionType?: CompressionType;
    outputBuffer?: number[] | Uint8Array; outputIndex?: number;
    b200?: { chunkBytes?: number; mode?: 'compat' | 'fast' | 'primed' | 'fast-primed'; depth?: number; smallest?: boolean; lazy?: boolean;
             dictionary?: Uint8Array } }   // dictionary: a preset dictionary (zlib's deflateSetDictionary)
// engine-only knob -> ZLB_MODE_* (include/zlibts_b200.h); the default is the reference-compatible mode
const modeOf = (o: RawDeflateOptions = {}) => { const b = o.b200 ?? {}; const m = b.mode ?? 'compat';
    return (m.startsWith('fast') ? 1 | ((b.depth ?? 0) << 8) : 0) | (m.endsWith('primed') ? 2 : 0) | (b.smallest ? 4 : 0) |
        (b.lazy && m.startsWith('fast') ? 8 : 0); };   // lazy: ZLB_MODE_LAZY, a fast-mode option
export interface RawInflateOptions { index?: number; bufferSize?: number; bufferType?: BufferType; resize?: boolean;
    b200?: { dictionary?: Uint8Array } }   // a preset dictionary (zlib's inflateSetDictionary)

const STATUS_TEXT: { [k: number]: string } = {                                       // include/zlibts_b200.h
    1: 'input buffer is broken', 2: 'unknown BTYPE: 3', 3: 'invalid code length',
    5: 'invalid uncompressed block header: LEN', 6: 'invalid deflate stream: undefined code or distance',
    7: 'invalid deflate stream: over-subscribed code lengths' };
// the reference's message for a zlb_result.status: N of 'invalid code length: N' and LEN / NLEN ride above bit 7
const statusText = (st: number) => (st & 0xFF) === 3 ? 'invalid code length: ' + (st >>> 8) :
    (st & 0xFF) === 5 && (st >>> 8) ? 'invalid uncompressed block header: NLEN' : (STATUS_TEXT[st & 0xFF] ?? 'inflate failed');
const u8 = (x: number[] | Uint8Array) => x instanceof Uint8Array ? x : new Uint8Array(x);

export class RawDeflate {                                                            // src/RawDeflate.ts:50-114
    input: Uint8Array; output: Uint8Array; op: number; compressionType: CompressionType; lazy: number; chunk: number;
    mode: number; dictionary?: Uint8Array;
    constructor(input: number[] | Uint8Array, opts: RawDeflateOptions = {}) {
        this.input = u8(input);
        this.lazy = opts.lazy ?? 0;
        if (this.lazy) throw new Error('lazy matching is not supported: the reference corrupts data with lazy > 0');
        this.compressionType = opts.compressionType ?? CompressionType.DYNAMIC;
        this.output = opts.outputBuffer ? u8(opts.outputBuffer) : new Uint8Array(0);
        this.op = opts.outputIndex ?? 0;
        this.chunk = opts.b200?.chunkBytes ?? 0;
        this.mode = modeOf(opts);
        this.dictionary = opts.b200?.dictionary;
    }
    compress(flags = 0): Uint8Array {
        const r = native.deflateBatch([this.input], this.compressionType, this.chunk, flags, this.mode, this.dictionary);
        (this as any).adler32 = r.adler32[0];
        const body: Uint8Array = r.outputs[0];
        const out = new Uint8Array(this.op + body.length);
        out.set(this.output.subarray(0, Math.min(this.op, this.output.length)));     // caller's prefix survives
        out.set(body, this.op);
        this.output = out; this.op = out.length;
        return out;
    }
}

export class RawInflate {                                                            // src/RawInflate.ts:70-140
    input: Uint8Array; ip: number; bufferSize?: number; buffer: Uint8Array | null = null; op = 0; dictionary?: Uint8Array;
    constructor(input: Uint8Array, opts: RawInflateOptions = {}) {
        this.input = u8(input); this.ip = opts.index ?? 0; this.bufferSize = opts.bufferSize;
        this.dictionary = opts.b200?.dictionary;
    }
    decompress(flags = 0): Uint8Array {
        let cap = this.bufferSize ?? Math.max(0x8000, 4 * (this.input.length - this.ip));
        for (;;) {                                                                   // the reference grows its buffer
            const r = native.inflateBatch(this.input, [this.ip], [this.input.length - this.ip], [cap], flags, this.dictionary);
            if (r.status[0] === 4) { cap *= 4; continue; }
            if (r.status[0] !== 0) throw new Error(statusText(r.status[0]));
            this.ip += r.inUsed[0]; this.buffer = r.outputs[0]; this.op = r.outputs[0].length;
            (this as any).crc32 = r.crc32[0]; (this as any).adler32 = r.adler32[0];
            return r.outputs[0];
        }
    }
}

export const CRC32 = {                                                               // src/CRC32.ts
    create(data: number[] | Uint8Array, pos?: number, length?: number): number { return CRC32.update(data, 0, pos, length); },
    update(data: number[] | Uint8Array, crc: number, pos = 0, length?: number): number {
        const piece = u8(data).subarray(pos, pos + (length ?? data.length));
        const c = native.checksumBatch([piece], 1).crc32[0];
        return crc ? native.crc32Combine(crc >>> 0, c, piece.length) : c;
    } };
export const Adler32 = {                                                             // src/Adler32.ts
    create(array: string | number[] | Uint8Array): number {
        if (typeof array === 'string') array = Array.from(array, ch => ch.charCodeAt(0) & 0xFF);
        return Adler32.update(1, u8(array)); },
    update(adler: number, array: Uint8Array, len?: number, pos = 0): number {
        const piece = array.subarray(pos, pos + (len ?? array.length));
        const c = native.checksumBatch([piece], 2).adler32[0];
        return adler === 1 ? c : native.adler32Combine(adler >>> 0, c, piece.length);
    } };

export class Deflate {                                                               // src/Deflate.ts
    adler32: number | null = null; output: Uint8Array | null = null;
    constructor(public input: Uint8Array | number[], public opts: RawDeflateOptions = {}) {}
    static compress(input: number[] | Uint8Array, opts: RawDeflateOptions) { return new Deflate(input, opts).compress(); }
    compress(): Uint8Array {
        const type = this.opts.compressionType ?? CompressionType.DYNAMIC;
        const dict = this.opts.b200?.dictionary;
        if (dict && dict.length) {
            // preset dictionary: FDICT, DICTID (the dictionary's Adler-32), the dictionary deflate, Adler-32 of the input
            const cmf = 120; let flg = type << 6 | 0x20; flg |= 31 - ((cmf << 8) + flg) % 31;
            const raw = new RawDeflate(this.input, this.opts), body = raw.compress(2), id = Adler32.create(dict);
            this.adler32 = (raw as any).adler32 as number;
            const out = new Uint8Array(6 + body.length + 4), v = new DataView(out.buffer);
            out[0] = cmf; out[1] = flg; v.setUint32(2, id); out.set(body, 6); v.setUint32(6 + body.length, this.adler32);
            return this.output = out;
        }
        const cmf = 120; let flg = type << 6; flg |= 31 - ((cmf << 8) + flg) % 31;     // :67-78
        // header, raw stream and big-endian Adler-32 (:95) are put together on the device (zlb_archive_host, kind 1)
        const r = native.archive(1, [u8(this.input)], [new Uint8Array([cmf, flg])], null, null, new Uint8Array(0),
                                 type, this.opts.b200?.chunkBytes ?? 0, modeOf(this.opts));
        this.adler32 = r.adler32[0];
        return this.output = r.output;
    }
}

export class Inflate {                                                               // src/Inflate.ts
    ip: number; verify: boolean; adler32: number | null = null; rawinflate: RawInflate;
    constructor(public input: Uint8Array, opts: RawInflateOptions & { verify?: boolean } = {}) {
        this.ip = opts.index ?? 0; this.verify = opts.verify ?? false;
        const cmf = input[this.ip++], flg = input[this.ip++];
        if ((cmf & 0x0f) !== 8) throw new Error('unsupported compression method');
        if (((cmf << 8) + flg) % 31 !== 0) throw new Error('invalid fcheck flag:' + ((cmf << 8) + flg) % 31);
        // a preset dictionary is used for FDICT streams only; other streams ignore it, like zlib
        const dict = flg & 0x20 ? opts.b200?.dictionary : undefined;
        if (flg & 0x20) {
            if (!dict) throw new Error('fdict flag is not supported');
            const p = this.ip, id = (input[p] << 24 | input[p + 1] << 16 | input[p + 2] << 8 | input[p + 3]) >>> 0;
            const have = Adler32.create(dict) >>> 0;
            if (have !== id) throw new Error('invalid dictionary: adler-32 0x' + have.toString(16).padStart(8, '0') +
                                             ', DICTID 0x' + id.toString(16).padStart(8, '0'));
            this.ip += 4;
        }
        this.rawinflate = new RawInflate(input, { index: this.ip, bufferSize: opts.bufferSize, b200: { dictionary: dict } });
    }
    decompress(): Uint8Array {
        const buffer = this.rawinflate.decompress(this.verify ? 2 : 0);
        this.ip = this.rawinflate.ip;
        if (this.verify) {
            const i = this.input, p = this.ip;
            this.adler32 = (this.rawinflate as any).adler32;
            if (this.adler32 !== ((i[p] << 24 | i[p + 1] << 16 | i[p + 2] << 8 | i[p + 3]) >>> 0)) throw new Error('invalid adler-32 checksum');
        }
        return buffer;
    }
}
// Whole containers in one call (what GZip.compress / Zip.compress do entry by entry, src/GZip.ts:96-194,
// src/Zip.ts:117-372): every entry checksummed + deflated in one batch, headers / trailers / central directory / end
// record written and packed on the device. heads / cdirs / tail are the byte templates described in the header.
export const archive = (kind: 1 | 2 | 3, inputs: Uint8Array[], heads: Uint8Array[], cdirs: Uint8Array[] | null,
                        methods: number[] | null, tail: Uint8Array, opts: RawDeflateOptions = {}) =>
    native.archive(kind, inputs, heads, cdirs, methods, tail, opts.compressionType ?? CompressionType.DYNAMIC,
                   opts.b200?.chunkBytes ?? 0, modeOf(opts)) as
    { output: Uint8Array; crc32: number[]; adler32: number[]; offsets: number[]; lengths: number[] };

// GZip / GUnzip / Zip / Unzip keep the reference's own source (src/GZip.ts, src/GUnzip.ts, src/Zip.ts, src/Unzip.ts)
// unchanged: they only call RawDeflate, RawInflate and CRC32, which resolve to the classes above once the
// reference's imports of "./RawDeflate", "./RawInflate", "./CRC32", "./Adler32" point at this file (INTEGRATION.md).
