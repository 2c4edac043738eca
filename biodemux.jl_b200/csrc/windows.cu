// windows.cu -- search-window read input (include/bdx.h, bdx_submit_windows): the device side.
//
// A classification depends on a read's length and on its bytes inside the columns of read_windows (literal.cuh)
// only.  The host sends just those bytes -- the "window bytes" of every read, spans in column order, as bytes or as
// the 4-bit codes of packed.cu -- plus the full reads' offsets and the offsets of the window stream.  This kernel
// rebuilds the slot's ordinary full-length sequence buffer: window columns from the stream, every other column a
// fixed filler byte (the one code 0 expands to, a byte in no barcode, when the config has codes; else 0).  The
// filler only makes the buffer deterministic; no result depends on it.  The classification kernels run unchanged.
// HBM-bound: the window bytes in, every byte of the batch out.
#include "literal.cuh"

namespace bdx {

struct WinRep {
    uint64_t rep[2];        // code k -> representative byte k of these 16 (packed windows); byte 0 is the filler
};

// A group of G lanes (4..32, a power of two) per read, grid-stride over the reads: short reads keep many reads in
// flight per warp, long ones spread their chunks over a whole warp.  The read's own 16-byte aligned chunks take
// vector stores; the bytes of the chunks it shares with its neighbours are stored one by one.
template <bool PACKED>
__global__ void __launch_bounds__(256)
k_expand_windows(const uint8_t *__restrict__ win, const int *__restrict__ win_off, const int *__restrict__ off,
                 uint8_t *__restrict__ seq, const int n_reads, const int G, const __grid_constant__ DevParams P,
                 const WinRep T)
{
    const int lane = threadIdx.x & (G - 1);
    const int warps = (gridDim.x * blockDim.x) / G;
    const uint8_t fill = (uint8_t)T.rep[0];
    const uint32_t fill4 = fill * 0x01010101u;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) / G; i < n_reads; i += warps) {
        const int base = off[i], n = off[i + 1] - base, w0 = win_off[i];
        int sp[4];
        read_windows(P, n, sp);
        const int len1 = max(0, sp[1] - sp[0] + 1);
        // byte of column c (1-based)
        auto byte_at = [&](int c) -> uint8_t {
            int k;
            if (c >= sp[0] && c <= sp[1]) k = w0 + c - sp[0];
            else if (c >= sp[2] && c <= sp[3]) k = w0 + len1 + c - sp[2];
            else return fill;
            if (!PACKED) return __ldg(win + k);
            const int code = (__ldg(win + (k >> 1)) >> ((k & 1) * 4)) & 15;
            return (uint8_t)(((code & 8) ? T.rep[1] : T.rep[0]) >> (8 * (code & 7)));
        };
        const int a = (base + 15) & ~15, b = max(a, (base + n) & ~15);   // aligned interior [a, b)
        for (int p = base + lane; p < min(a, base + n); p += G) seq[p] = byte_at(p - base + 1);
        for (int p = max(b, base) + lane; p < base + n; p += G) seq[p] = byte_at(p - base + 1);
        for (int v = a + lane * 16; v < b; v += G * 16) {
            const int c0 = v - base + 1, c1 = c0 + 15;                   // columns of this chunk
            uint4 o;
            const bool in_gap = (c1 < sp[0] || c0 > sp[1]) && (c1 < sp[2] || c0 > sp[3]);
            if (in_gap) {
                o = make_uint4(fill4, fill4, fill4, fill4);
            } else {
                uint32_t w[4];
#pragma unroll
                for (int q = 0; q < 4; q++)
                    w[q] = byte_at(c0 + 4 * q) | (byte_at(c0 + 4 * q + 1) << 8) | (byte_at(c0 + 4 * q + 2) << 16) |
                           ((uint32_t)byte_at(c0 + 4 * q + 3) << 24);
                o = make_uint4(w[0], w[1], w[2], w[3]);
            }
            *reinterpret_cast<uint4 *>(seq + v) = o;
        }
    }
}

cudaError_t launch_expand_windows(const uint8_t *d_win, bool packed, const int *d_win_off, const int *d_off,
                                  uint8_t *d_seq, int n_reads, long long bytes, const DevParams &P, const uint8_t rep[16],
                                  int sm_count, cudaStream_t st)
{
    if (n_reads <= 0) return cudaSuccess;
    WinRep T{};
    for (int k = 0; k < 16; k++) T.rep[k >> 3] |= (uint64_t)rep[k] << (8 * (k & 7));
    int G = 4;                                        // lanes per read: about four 16-byte chunks of a mean read each
    while (G < 32 && (long long)G * 64 < bytes / n_reads) G *= 2;
    const long long groups = 256 / G;
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n_reads + groups - 1) / groups, (long long)sm_count * 8));
    if (packed) k_expand_windows<true><<<blocks, 256, 0, st>>>(d_win, d_win_off, d_off, d_seq, n_reads, G, P, T);
    else k_expand_windows<false><<<blocks, 256, 0, st>>>(d_win, d_win_off, d_off, d_seq, n_reads, G, P, T);
    return cudaGetLastError();
}

}  // namespace bdx
