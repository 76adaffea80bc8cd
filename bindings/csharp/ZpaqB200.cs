// ZpaqB200.cs -- P/Invoke binding of libzpaqb200.so for ZPAQSharp (source only: this image has no
// .NET toolchain, so the file is not compiled or tested here; the same entry points are exercised
// through ctypes in zpaqsharp_b200/libzpaq.py and tests/).
//
// Drop-in: LibZPAQ.Compress / compressBlock / decompress (LibZPAQ.cs:84,117,65) keep their
// signatures; their bodies gather blocks from the Reader, call the batch ABI once, and write the
// result to the Writer.  LibZPAQ.error (LibZPAQ.cs:22-24) keeps its role: a negative return code
// becomes error(zpq_last_error()).
using System;
using System.Runtime.InteropServices;
using System.Text;

namespace ZPAQSharp
{
    internal static unsafe class ZpaqB200Native
    {
        const string Lib = "zpaqb200";   // libzpaqb200.so / zpaqb200.dll

        [DllImport(Lib)] public static extern int zpq_create(int* deviceIds, int ndev, out IntPtr ctx);
        [DllImport(Lib)] public static extern void zpq_destroy(IntPtr ctx);
        [DllImport(Lib)] public static extern IntPtr zpq_last_error(IntPtr ctx);
        [DllImport(Lib)] public static extern int zpq_compress_blocks(IntPtr ctx, byte* input, ulong* inOff, uint nb,
            [MarshalAs(UnmanagedType.LPStr)] string method, [MarshalAs(UnmanagedType.LPStr)] string filename0,
            [MarshalAs(UnmanagedType.LPStr)] string comment0, int dosha1, byte* output, ulong outCap, ulong* outOff);
        [DllImport(Lib)] public static extern int zpq_compress_blocks_level(IntPtr ctx, int level, byte* input, ulong* inOff, uint nb,
            [MarshalAs(UnmanagedType.LPStr)] string filename0, [MarshalAs(UnmanagedType.LPStr)] string comment0,
            int dosha1, int withTag, byte* output, ulong outCap, ulong* outOff);
        [DllImport(Lib)] public static extern int zpq_compress_blocks_model(IntPtr ctx, byte* hdr, ulong hdrLen, byte* pcomp, ulong pcompLen,
            int* args9, byte* input, ulong* inOff, uint nb, [MarshalAs(UnmanagedType.LPStr)] string filename0,
            [MarshalAs(UnmanagedType.LPStr)] string comment0, int dosha1, int withTag, byte* output, ulong outCap, ulong* outOff);
        [DllImport(Lib)] public static extern long zpq_find_blocks(byte* archive, ulong n, ulong* offsets, ulong maxBlocks);
        [DllImport(Lib)] public static extern long zpq_decompressed_bound(byte* input, ulong* inOff, uint nb);
        [DllImport(Lib)] public static extern int zpq_decompress_blocks(IntPtr ctx, byte* input, ulong* inOff, uint nb, byte* output,
            ulong outCap, ulong* outOff, byte* sha1Status, byte* blockStatus);
        [DllImport(Lib)] public static extern long zpq_make_config([MarshalAs(UnmanagedType.LPStr)] string method, int* args9,
            byte* text, ulong textCap);
        [DllImport(Lib)] public static extern int zpq_compile_config([MarshalAs(UnmanagedType.LPStr)] string config, int* args9,
            byte* hdr, ulong hdrCap, out ulong hdrLen, byte* pcomp, ulong pcompCap, out ulong pcompLen);
        [DllImport(Lib)] public static extern long zpq_builtin_model(int level, byte* hdr, ulong hdrCap);
        [DllImport(Lib)] public static extern double zpq_block_memory(byte* hdr, ulong hdrLen);
        [DllImport(Lib)] public static extern long zpq_device_state_bytes(byte* hdr, ulong hdrLen, int forDecode);
        [DllImport(Lib)] public static extern long zpq_device_state_bytes_for(byte* hdr, ulong hdrLen, int forDecode, ulong maxBlockBytes);
        [DllImport(Lib)] public static extern long zpq_post_kind(int ph, int pm, byte* pcomp, ulong len);
        [DllImport(Lib)] public static extern long zpq_specialize_pcomp(int ph, int pm, byte* pcomp, ulong len, byte* source, ulong sourceCap, byte* log, ulong logCap);
        [DllImport(Lib)] public static extern int zpq_encoder_plan(byte* hdr, ulong hdrLen, uint smemBytes, uint blocksPerSm, int* out8);
        [DllImport(Lib)] public static extern int zpq_scrypt(byte* pw, ulong pwLen, byte* salt, ulong saltLen, ulong n, uint r, uint p,
            byte* output, ulong outLen);
        [DllImport(Lib)] public static extern int zpq_stretch_key(byte* in32, byte* salt32, byte* out32);
        [DllImport(Lib)] public static extern int zpq_aes_ctr(IntPtr ctx, byte* key, int keyLen, byte* iv8, byte* buf, ulong n, ulong offset);
        [DllImport(Lib)] public static extern int zpq_aes_ctr_dev(IntPtr ctx, byte* key, int keyLen, byte* iv8, byte* dBuf, ulong n, ulong offset);
    }

    /// <summary>GPU-backed bodies for the LibZPAQ entry points of the compress/decompress path.</summary>
    public static unsafe class LibZPAQB200
    {
        static IntPtr ctx;

        static IntPtr Ctx()
        {
            if (ctx == IntPtr.Zero && ZpaqB200Native.zpq_create(null, 0, out ctx) != 0)
                LibZPAQ.error(Marshal.PtrToStringAnsi(ZpaqB200Native.zpq_last_error(IntPtr.Zero)));
            return ctx;
        }

        static void Check(int rc)
        {
            if (rc != 0) LibZPAQ.error(Marshal.PtrToStringAnsi(ZpaqB200Native.zpq_last_error(ctx)));
        }

        /// <summary>LibZPAQ.Compress (LibZPAQ.cs:84-108): split by the method's block size, code all blocks at once.</summary>
        public static void Compress(Reader input, Writer output, string method, string filename = null, string comment = null, bool dosha1 = true)
        {
            int bs = 4;
            if (method.Length > 1 && char.IsDigit(method[1]))
            {
                bs = method[1] - '0';
                if (method.Length > 2 && char.IsDigit(method[2])) bs = bs * 10 + method[2] - '0';
                if (bs > 11) bs = 11;
            }
            long blockSize = (0x100000L << bs) - 4096;
            var data = new System.IO.MemoryStream();
            var buf = new char[1 << 16];
            int n;
            while ((n = input.read(buf, buf.Length)) > 0)
                for (int i = 0; i < n; ++i) data.WriteByte((byte)buf[i]);
            byte[] all = data.ToArray();
            uint nb = (uint)((all.Length + blockSize - 1) / blockSize);
            if (nb == 0) return;
            var off = new ulong[nb + 1];
            for (uint i = 0; i <= nb; ++i) off[i] = (ulong)Math.Min(all.Length, i * blockSize);
            var outBuf = new byte[all.Length + all.Length / 4 + 8192 * (nb + 1) + 65536];
            var outOff = new ulong[nb + 1];
            fixed (byte* pin = all, pout = outBuf)
            fixed (ulong* poff = off, pooff = outOff)
                Check(ZpaqB200Native.zpq_compress_blocks(Ctx(), pin, poff, nb, method, filename, comment, dosha1 ? 1 : 0,
                                                          pout, (ulong)outBuf.Length, pooff));
            for (ulong i = 0; i < outOff[nb]; ++i) output.put(outBuf[i]);
        }

        /// <summary>LibZPAQ.decompress (LibZPAQ.cs:65-79): every block and segment of the archive, in order.</summary>
        public static void Decompress(Reader input, Writer output)
        {
            var data = new System.IO.MemoryStream();
            int c;
            while ((c = input.get()) >= 0) data.WriteByte((byte)c);
            byte[] arc = data.ToArray();
            fixed (byte* p = arc)
            {
                long nb = ZpaqB200Native.zpq_find_blocks(p, (ulong)arc.Length, null, 0);
                if (nb < 0) LibZPAQ.error(Marshal.PtrToStringAnsi(ZpaqB200Native.zpq_last_error(IntPtr.Zero)));
                if (nb == 0) return;
                var pairs = new ulong[2 * nb];
                fixed (ulong* pp = pairs) ZpaqB200Native.zpq_find_blocks(p, (ulong)arc.Length, pp, (ulong)nb);
                // blocks are decoded from their "zPQ"; pack them back to back for the batch call
                var packed = new System.IO.MemoryStream();
                var off = new ulong[nb + 1];
                for (long i = 0; i < nb; ++i)
                {
                    off[i] = (ulong)packed.Length;
                    packed.Write(arc, (int)pairs[2 * i], (int)(pairs[2 * i + 1] - pairs[2 * i]));
                }
                off[nb] = (ulong)packed.Length;
                byte[] blocks = packed.ToArray();
                fixed (byte* pb = blocks)
                fixed (ulong* poff = off)
                {
                    long bound = ZpaqB200Native.zpq_decompressed_bound(pb, poff, (uint)nb);
                    var outBuf = new byte[Math.Max(bound, 16)];
                    var outOff = new ulong[nb + 1];
                    fixed (byte* po = outBuf)
                    fixed (ulong* pooff = outOff)
                        Check(ZpaqB200Native.zpq_decompress_blocks(Ctx(), pb, poff, (uint)nb, po, (ulong)outBuf.Length, pooff, null, null));
                    for (ulong i = 0; i < outOff[nb]; ++i) output.put(outBuf[i]);
                }
            }
        }

        /// <summary>libzpaq stretchKey(out, in, salt), the body StretchKey.cs:13-163 restates: scrypt(in, 32, salt, 32,
        /// 16384, 8, 1, out, 32), computed on the host by the library.  in32 is SHA-256 of the password.</summary>
        public static void StretchKey(byte[] out32, byte[] in32, byte[] salt32)
        {
            if (out32 == null || in32 == null || salt32 == null || out32.Length < 32 || in32.Length < 32 || salt32.Length < 32)
                LibZPAQ.error("stretchKey takes 32-byte buffers");
            fixed (byte* po = out32, pi = in32, ps = salt32)
                CheckHost(ZpaqB200Native.zpq_stretch_key(pi, ps, po));
        }

        /// <summary>libzpaq scrypt(pw, pwlen, salt, saltlen, n, r, p, buf, buflen) (RFC 7914), StretchKey.cs:13-163.</summary>
        public static void Scrypt(byte[] pw, int pwlen, byte[] salt, int saltlen, int n, int r, int p, byte[] buf, int buflen)
        {
            if (pwlen < 0 || saltlen < 0 || buflen < 0 || r < 0 || p < 0 || n < 0) LibZPAQ.error("scrypt: negative argument");
            fixed (byte* ppw = pw, ps = salt, pb = buf)
                CheckHost(ZpaqB200Native.zpq_scrypt(ppw, (ulong)pwlen, ps, (ulong)saltlen, (ulong)n, (uint)r, (uint)p, pb, (ulong)buflen));
        }

        static void CheckHost(int rc)
        {
            if (rc != 0) LibZPAQ.error(Marshal.PtrToStringAnsi(ZpaqB200Native.zpq_last_error(IntPtr.Zero)));
        }

        internal static IntPtr Context() { return Ctx(); }
        internal static void CheckCtx(int rc) { Check(rc); }
    }

    /// <summary>libzpaq 7.12's AES_CTR (the reference has it as prose only, LICENSE:635-665): AES in counter mode with
    /// keystream block j = AES_key(iv[0..7] || big-endian j).  encrypt(buf, n, offset) XORs buf[0..n) with the keystream
    /// from stream byte offset on the GPU; decrypting is the same call.  The key bytes are kept only to pass them to each
    /// call; the library expands and wipes the key schedule inside the call.</summary>
    public unsafe class AesCtrB200
    {
        readonly byte[] key;
        readonly byte[] iv;

        public AesCtrB200(byte[] key, int keylen, byte[] iv = null)
        {
            if (keylen != 16 && keylen != 24 && keylen != 32) LibZPAQ.error("AES_CTR: key length must be 16, 24 or 32");
            this.key = new byte[keylen];
            Array.Copy(key, this.key, keylen);
            if (iv != null) { this.iv = new byte[8]; Array.Copy(iv, this.iv, 8); }
        }

        public void encrypt(byte[] buf, int n, ulong offset)
        {
            if (n < 0 || n > buf.Length) LibZPAQ.error("AES_CTR: n is outside the buffer");
            fixed (byte* pk = key, pi = iv, pb = buf)
                LibZPAQB200.CheckCtx(ZpaqB200Native.zpq_aes_ctr(LibZPAQB200.Context(), pk, key.Length, pi, pb, (ulong)n, offset));
        }
    }
    /// <summary>Replacement body of Compressor (Compressor.cs:12-304) over the batch ABI: same methods, same call order,
    /// same bytes.  A segment is buffered; finished blocks are QUEUED and coded by the GPU a wave at a time through one
    /// zpq_compress_blocks_model call per model (when BatchBlocks of them are pending, on flush() and on Dispose()): a block
    /// coded alone waits for its own serial bit chain, a wave of 1600 takes the same time.  Everything written after a
    /// pending block is held back with it, so the Writer receives the reference's bytes in the reference's order.
    /// One segment per block.  The Python model of this class, zpaqsharp_b200/facade.py, is what the tests run
    /// (tests/test_facade_host.py, tests/test_gpu_facade.py).</summary>
    public unsafe class CompressorB200 : IDisposable
    {
        enum State { INIT, BLOCK1, SEG1, BLOCK2, SEG2 }
        sealed class Pending { public byte[] hdr, pcomp, data, sha1; public byte[] body; }
        State state = State.INIT;
        Writer output; Reader input;
        byte[] hdr = new byte[0], pz = new byte[0], pcomp = new byte[0];
        readonly System.IO.MemoryStream seg = new System.IO.MemoryStream();
        readonly System.Collections.Generic.List<object> queue = new System.Collections.Generic.List<object>();   // byte[] | Pending, in output order
        int npending;
        /// <summary>Blocks that wait for one GPU call (1 = code every block when it ends).</summary>
        public int BatchBlocks = 1600;
        static IntPtr ctx;
        static IntPtr Ctx()
        {
            if (ctx == IntPtr.Zero && ZpaqB200Native.zpq_create(null, 0, out ctx) != 0)
                LibZPAQ.error(Marshal.PtrToStringAnsi(ZpaqB200Native.zpq_last_error(IntPtr.Zero)));
            return ctx;
        }

        void emit(params byte[] b)
        {
            if (queue.Count > 0) queue.Add(b);
            else foreach (byte x in b) output.put(x);
        }
        static bool same(byte[] a, byte[] b) { return a.Length == b.Length && System.Linq.Enumerable.SequenceEqual(a, b); }

        /// <summary>Code every queued block (one batch call per model) and hand the held-back bytes to the Writer in order.</summary>
        public void flush()
        {
            var todo = new System.Collections.Generic.List<Pending>();
            foreach (object it in queue) if (it is Pending p) todo.Add(p);
            while (todo.Count > 0)
            {
                Pending first = todo[0];
                var group = todo.FindAll(q => same(q.hdr, first.hdr) && same(q.pcomp, first.pcomp));
                todo.RemoveAll(q => group.Contains(q));
                ulong total = 0;
                var off = new ulong[group.Count + 1];
                for (int i = 0; i < group.Count; ++i) { off[i] = total; total += (ulong)group[i].data.Length; }
                off[group.Count] = total;
                var data = new byte[total + 1];
                for (int i = 0; i < group.Count; ++i) Array.Copy(group[i].data, 0, data, (long)off[i], group[i].data.Length);
                var outBuf = new byte[(long)total + (long)total / 4 + (first.hdr.Length + first.pcomp.Length * 4 + 65536L) * group.Count];
                var outOff = new ulong[group.Count + 1];
                var args = new int[9];
                fixed (byte* ph = first.hdr, pp = first.pcomp, pi = data, po = outBuf)
                fixed (ulong* poff = off, pooff = outOff)
                fixed (int* pa = args)
                {
                    int rc = ZpaqB200Native.zpq_compress_blocks_model(Ctx(), ph, (ulong)first.hdr.Length, first.pcomp.Length > 0 ? pp : null,
                                                                      (ulong)first.pcomp.Length, pa, pi, poff, (uint)group.Count, null, null, 0, 0,
                                                                      po, (ulong)outBuf.Length, pooff);
                    if (rc != 0) LibZPAQ.error(Marshal.PtrToStringAnsi(ZpaqB200Native.zpq_last_error(ctx)));
                }
                for (int i = 0; i < group.Count; ++i)
                {
                    // the library wrote "zPQ" level 1, the header and a segment header with its default comment (the decimal size)
                    // in front of the coded bytes, and 254 255 behind them; this class has written its own headers already
                    int n = group[i].data.Length;
                    long skip = (long)outOff[i] + 5 + first.hdr.Length + 1 + 1 + n.ToString().Length + 1 + 1;
                    long end = (long)outOff[i + 1] - 2;          // up to and including the four zero bytes
                    var body = new System.IO.MemoryStream();
                    body.Write(outBuf, (int)skip, (int)(end - skip));
                    if (group[i].sha1 != null) { body.WriteByte(253); body.Write(group[i].sha1, 0, 20); }
                    else body.WriteByte(254);
                    group[i].body = body.ToArray();
                }
            }
            var q2 = queue.ToArray();
            queue.Clear(); npending = 0;
            foreach (object it in q2)
                foreach (byte x in (it is Pending p2 ? p2.body : (byte[])it)) output.put(x);
        }
        public void Dispose() { flush(); }

        public void setOutput(Writer o) { if (output != null) flush(); output = o; }
        public void setInput(Reader i) { input = i; }

        public void writeTag()                                   // Compressor.cs:27-43
        {
            emit(0x37, 0x6b, 0x53, 0x74, 0xa0, 0x31, 0x83, 0xd3, 0x8c, 0xb2, 0x28, 0xb0, 0xd3);
        }

        public void startBlock(int level)                        // Compressor.cs:45-83
        {
            if (level < 1) LibZPAQ.error("compression level must be at least 1");
            var buf = new byte[1024];
            long n;
            fixed (byte* p = buf) n = ZpaqB200Native.zpq_builtin_model(level, p, (ulong)buf.Length);
            if (n < 0) LibZPAQ.error("compression level too high");
            Array.Resize(ref buf, (int)n);
            startBlock(buf);
        }

        public void startBlock(byte[] hcomp)                     // Compressor.cs:85-99
        {
            hdr = hcomp; pz = new byte[0];
            emit((byte)'z', (byte)'P', (byte)'Q', (byte)(1 + (hdr[6] == 0 ? 1 : 0)), 1);
            emit(hdr);
            state = State.BLOCK1;
        }

        public void startSegment(string filename = null, string comment = null)   // Compressor.cs:133-146
        {
            if (state == State.BLOCK2) LibZPAQ.error("the device path codes one segment per block");
            emit(1);
            if (filename != null) emit(System.Text.Encoding.Latin1.GetBytes(filename));
            emit(0);
            if (comment != null) emit(System.Text.Encoding.Latin1.GetBytes(comment));
            emit(0, 0);
            seg.SetLength(0);
            pcomp = new byte[0];
            state = State.SEG1;
        }

        public void postProcess(byte[] program = null, int len = 0)               // Compressor.cs:156-190
        {
            if (state == State.SEG2) return;
            if (program == null) pcomp = pz;
            else if (len == 0) { len = program[0] + 256 * program[1]; pcomp = new byte[len]; Array.Copy(program, 2, pcomp, 0, len); }
            else { pcomp = new byte[len]; Array.Copy(program, 0, pcomp, 0, len); }
            state = State.SEG2;
        }

        public bool compress(int n = -1)                         // Compressor.cs:193-221
        {
            if (state == State.SEG1) postProcess();
            const int BUFSIZE = 1 << 14;
            var buf = new char[BUFSIZE];
            while (n != 0)
            {
                int nbuf = BUFSIZE;
                if (n >= 0 && n < nbuf) nbuf = n;
                int nr = input.read(buf, nbuf);
                if (nr < 0 || nr > BUFSIZE || nr > nbuf) LibZPAQ.error("invalid read size");
                if (nr <= 0) return false;
                if (n >= 0) n -= nr;
                for (int i = 0; i < nr; ++i) seg.WriteByte((byte)buf[i]);
            }
            return true;
        }

        public void endSegment(byte[] sha1string = null)         // Compressor.cs:224-249
        {
            if (state == State.SEG1) postProcess();
            queue.Add(new Pending { hdr = hdr, pcomp = pcomp, data = seg.ToArray(), sha1 = sha1string });
            ++npending;
            state = State.BLOCK2;
        }

        public void endBlock()                                   // Compressor.cs:294-299
        {
            emit(255);
            state = State.INIT;
            if (npending >= BatchBlocks) flush();
        }
    }
}
