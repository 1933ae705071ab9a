/*
 * grok_b200/csrc/ht_dec.cu -- HTJ2K (ITU-T T.814) cleanup-pass block DECODER for sm_100a, fused with
 * the T1 post-processing (dequantisation into the Mallat buffer).
 *
 * Replaces (reference, CPU): T1OJPH::decompress            t1/part15/CoderOJPH.cpp L212-262
 *                            ojph_decode_codeblock32        t1/part15/coding/ojph_block_decoder32.cpp L742-1317
 *                            ShiftOJPHFilter/ScaleOJPHFilter t1/part15/PostDecodeFiltersOJPH.h L48-66, L100-119
 * The cleanup pass is all Grok's own encoder ever emits (CoderOJPH.cpp L200-205).  It is decoded in two
 * launches:
 *  (a) k_ht_decode_vlc, one THREAD per code block: the MEL + CxtVLC + U-VLC symbols, which have no
 *      parallel parse, are decoded serially into one record per quad in global scratch;
 *  (b) k_ht_decode_magsgn, one WARP per code block: per quad row the per-sample bit counts follow from
 *      the records, a warp prefix sum gives every lane its bit offset into an un-stuffed shared-memory
 *      bit ring that is refilled 256 bytes at a time (8 bytes per lane, stuffing resolved with one
 *      ballot since on the decode side a byte's width only depends on its predecessor's VALUE), and the
 *      lanes dequantise their quads straight into the Mallat buffer.
 * Blocks of foreign streams that carry SigProp / MagRef refinement (ojph_block_decoder32.cpp
 * L1318-1616) leave (b) as raw sign-magnitude words and are finished by k_ht_decode_refine, which also
 * dequantises them.
 */
#include "b2k_internal.h"
#define HT_TABLE_QUAL static __device__ const
#include "ht_tables.h"

namespace {

constexpr int MS_RING_WORDS = 256;

__device__ __forceinline__ int mel_exp_d(int k) { return (int)((0x58da489200ull >> (3 * k)) & 7ull); }

__device__ __forceinline__ int uvlc_prefix(uint32_t bits, int& len)
{
  if(bits & 1) { len = 1; return 1; }
  if(bits & 2) { len = 2; return 2; }
  if(bits & 4) { len = 3; return 3; }
  len = 3;
  return 5;
}
__device__ __forceinline__ int uvlc_suflen(int pfx) { return pfx == 3 ? 1 : (pfx == 5 ? 5 : 0); }

template <typename T>
__device__ __forceinline__ T warp_excl_scan_d(T v, int lane, T& total)
{
  T x = v;
#pragma unroll
  for(int o = 1; o < 32; o <<= 1)
  {
    const T y = __shfl_up_sync(0xffffffffu, x, o);
    if(lane >= o)
      x += y;
  }
  total = __shfl_sync(0xffffffffu, x, 31);
  return x - v;
}

/* =============================================================================================
 * Phase A -- MEL + CxtVLC + UVLC parse, ONE THREAD PER CODE BLOCK.
 * Context-adaptive variable-length codes cannot be parsed in parallel inside a block, but blocks
 * are independent: 32 blocks per warp keep every lane busy (a warp-per-block version of this
 * loop runs the same instruction stream with 1/32 of the lanes doing useful work).
 * Output: one record per quad in global scratch, rho[3:0] | e_k[7:4] | e_1[11:8] | u[17:12],
 * consumed by phase B (k_ht_decode_magsgn, warp per block).  The records of 32 consecutive blocks are
 * interleaved word by word (entry k of a block sits at rec_off + 32 k): the 32 lanes of this kernel
 * -- 32 different blocks at the same quad -- store 128 contiguous bytes instead of 32 scattered words.
 * =========================================================================================== */

/* ---- phase A readers: the serial parse is latency-bound, so its byte streams must not put a global load into the
 * dependency chain for every byte.  Both streams are read through an aligned 8-byte register window with the NEXT
 * window already in flight (issued when the current one is entered, ~4 quad pairs of parsing ahead of its first use). */
struct VlcFast
{ /* backward reader of the VLC segment (rev_read / rev_init, ojph_block_decoder32.cpp L296-395) */
  const uint8_t* d;
  const uint64_t* ap; /* aligned window holding the byte at `pos` */
  uint64_t cur, nxt, nx2, tmp; /* the window in use and the two below it, already in flight */
  int pos, lo, bits, unstuff;
};
__device__ __forceinline__ uint64_t vlcf_load(const VlcFast& v, const uint64_t* a)
{ /* a window that lies wholly below the segment is never looked at */
  return reinterpret_cast<const uint8_t*>(a) + 7 >= v.d + v.lo ? __ldg(a) : 0ull;
}
__device__ __forceinline__ void vlcf_init(VlcFast& v)
{
  const uint8_t* a = v.d + (v.pos > 0 ? v.pos : 0);
  v.ap = reinterpret_cast<const uint64_t*>(reinterpret_cast<uintptr_t>(a) & ~(uintptr_t)7);
  v.cur = vlcf_load(v, v.ap);
  v.nxt = vlcf_load(v, v.ap - 1);
  v.nx2 = vlcf_load(v, v.ap - 2);
}
__device__ __forceinline__ void vlcf_rotate(VlcFast& v)
{
  --v.ap;
  v.cur = v.nxt;
  v.nxt = v.nx2;
  v.nx2 = vlcf_load(v, v.ap - 2); /* 16 bytes (six or seven quad pairs of parsing) ahead of its first use */
}
/* at least 32 un-stuffed bits buffered (a quad pair takes at most 31).  Four bytes per refill: only a byte whose low
   seven bits are all ones can be a stuffed (7-bit) byte, so when none of the four is (97 % of the time) they go into
   the bit buffer with one shift; otherwise, and at the segment's start, byte by byte as rev_read does */
__device__ __forceinline__ void vlcf_fill32(VlcFast& v)
{
  if(v.bits >= 32)
    return;
  if(v.pos - 3 >= v.lo)
  {
    if(v.d + v.pos < reinterpret_cast<const uint8_t*>(v.ap))
      vlcf_rotate(v); /* the byte-wise path below moves pos without moving the window */
    const int o = (int)((v.d + v.pos) - reinterpret_cast<const uint8_t*>(v.ap)); /* byte `pos` inside cur: 0 .. 7 */
    /* bytes pos-3 .. pos as a little-endian word, from cur (and the window below it when o < 3) */
    const uint32_t le = o >= 3 ? (uint32_t)(v.cur >> (8 * (o - 3))) : (uint32_t)((v.nxt >> (8 * (o + 5))) | (v.cur << (8 * (3 - o))));
    const uint32_t w = __byte_perm(le, 0, 0x0123); /* byte `pos` lowest: the order the stream is read in */
    if((((w & 0x7F7F7F7Fu) + 0x01010101u) & 0x80808080u) == 0)
    {
      v.tmp |= (uint64_t)w << v.bits;
      v.bits += 32;
      v.unstuff = (w >> 24) > 0x8Fu;
      v.pos -= 4;
      if(v.d + v.pos < reinterpret_cast<const uint8_t*>(v.ap))
        vlcf_rotate(v);
      return;
    }
  }
  while(v.bits < 32)
  {
    uint32_t b = 0;
    if(v.pos >= v.lo)
    {
      const uint8_t* a = v.d + v.pos;
      if(a < reinterpret_cast<const uint8_t*>(v.ap))
        vlcf_rotate(v);
      b = (uint32_t)(v.cur >> (8 * (int)(a - reinterpret_cast<const uint8_t*>(v.ap)))) & 0xFFu;
    }
    v.pos--;
    const int nb = 8 - ((v.unstuff && ((b & 0x7F) == 0x7F)) ? 1 : 0);
    v.tmp |= (uint64_t)b << v.bits;
    v.bits += nb;
    v.unstuff = b > 0x8F;
  }
}
struct MelFast
{ /* forward reader of the MEL segment (mel_read / mel_decode, L92-206) */
  const uint8_t* d;
  const uint64_t* ap;
  uint64_t cur, nxt;
  int size, pos, bits, unstuff, k, run, have;
  uint32_t tmp;
};
__device__ __forceinline__ void melf_init(MelFast& m)
{
  m.ap = reinterpret_cast<const uint64_t*>(reinterpret_cast<uintptr_t>(m.d) & ~(uintptr_t)7);
  m.cur = __ldg(m.ap);
  m.nxt = reinterpret_cast<const uint8_t*>(m.ap + 1) < m.d + m.size ? __ldg(m.ap + 1) : 0ull;
}
__device__ __forceinline__ int melf_bit(MelFast& m)
{
  if(m.bits == 0)
  {
    uint32_t v = 0xFF;
    if(m.pos < m.size)
    {
      const uint8_t* a = m.d + m.pos;
      if(a >= reinterpret_cast<const uint8_t*>(m.ap + 1))
      {
        ++m.ap;
        m.cur = m.nxt;
        m.nxt = reinterpret_cast<const uint8_t*>(m.ap + 1) < m.d + m.size ? __ldg(m.ap + 1) : 0ull;
      }
      v = (uint32_t)(m.cur >> (8 * (int)(a - reinterpret_cast<const uint8_t*>(m.ap)))) & 0xFFu;
      if(m.pos == m.size - 1)
        v |= 0xF;
      m.pos++;
    }
    m.bits = 8 - m.unstuff;
    m.tmp = v;
    m.unstuff = (v == 0xFF);
  }
  m.bits--;
  return (int)((m.tmp >> m.bits) & 1u);
}
__device__ __forceinline__ int melf_symbol(MelFast& m)
{
  if(!m.have)
  {
    const int ev = mel_exp_d(m.k);
    if(melf_bit(m))
    {
      m.run = 1 << ev;
      m.have = 1;
      m.k = min(12, m.k + 1);
    }
    else
    {
      int r = 0;
      for(int i = 0; i < ev; ++i)
        r = (r << 1) | melf_bit(m);
      m.run = r;
      m.have = 2;
      m.k = max(0, m.k - 1);
    }
  }
  if(m.run > 0)
  {
    m.run--;
    if(m.run == 0 && m.have == 1)
      m.have = 0;
    return 0;
  }
  m.have = 0;
  return 1;
}

/* ---------------------------------------------------------------------------------------------
 * The parse is arranged so that a quad pair costs one refill check, two CxtVLC look-ups and ONE
 * U-VLC look-up instead of a tree of branches:
 *  - uvlc[mode * 64 + next 6 bits] holds, for the pair's two u-offset flags (mode 0..3) and for the
 *    first row's "both flags set, MEL said 0" rule (mode 4, T.814 7.3.6 / ojph_block_decoder32.cpp
 *    L966-1010), the bits the two prefixes take, the two suffix lengths and the two base values;
 *    the table is built in shared memory at kernel start from the prefix code itself;
 *  - the neighbourhood bit of a quad's context is one shift of a 64-bit mask of the row above
 *    (A = bl | br << 1).  Blocks at most 64 samples wide (32 quads, WIDE = false) keep the row's
 *    significance in one register word per side and build A once per row; wider ones (up to 1024
 *    samples, 512 quads) keep 16 words per side and rebuild A every 32 quads.
 * The serial chain per quad is what bounds this phase; this halves it against a branchy parse.
 * ------------------------------------------------------------------------------------------- */
__device__ __forceinline__ uint32_t uvlc_entry(int mode, uint32_t bits)
{ /* plen[2:0] | l0[5:3] | l1[8:6] | p0[11:9] | p1[14:12] */
  int plen = 0, l0 = 0, l1 = 0, p0 = 0, p1 = 0, len;
  if(mode < 4)
  {
    if(mode & 1)
    {
      p0 = uvlc_prefix(bits, len);
      bits >>= len;
      plen += len;
      l0 = uvlc_suflen(p0);
    }
    if(mode & 2)
    {
      p1 = uvlc_prefix(bits, len);
      plen += len;
      l1 = uvlc_suflen(p1);
    }
  }
  else
  { /* first quad row, both u-offsets set, MEL symbol 0 */
    p0 = uvlc_prefix(bits, len);
    bits >>= len;
    plen += len;
    if(p0 > 2)
    {
      p1 = 1 + (int)(bits & 1u); /* u1 is 1 or 2: one bit, sitting where the second prefix would */
      plen += 1;
      l0 = uvlc_suflen(p0);
    }
    else
    {
      p1 = uvlc_prefix(bits, len);
      plen += len;
      l1 = uvlc_suflen(p1);
    }
  }
  return (uint32_t)plen | ((uint32_t)l0 << 3) | ((uint32_t)l1 << 6) | ((uint32_t)p0 << 9) | ((uint32_t)p1 << 12);
}

template <bool WIDE>
__global__ void __launch_bounds__(32)
    k_ht_decode_vlc(const HtBlockDesc* __restrict__ blocks, const uint8_t* __restrict__ bytes, uint32_t* __restrict__ recs,
                    HtBlockOut* __restrict__ status, uint32_t nblocks)
{
  __shared__ uint16_t tbl0[1024], tbl1[1024], uvlc[5 * 64];
  for(int i = threadIdx.x; i < 1024; i += blockDim.x)
  {
    tbl0[i] = HT_DEC_VLC0[i];
    tbl1[i] = HT_DEC_VLC1[i];
  }
  for(int i = threadIdx.x; i < 5 * 64; i += blockDim.x)
    uvlc[i] = (uint16_t)uvlc_entry(i >> 6, (uint32_t)(i & 63));
  __syncthreads();
  const uint32_t bidx = blockIdx.x * blockDim.x + threadIdx.x;
  if(bidx >= nblocks)
    return;
  const HtBlockDesc B = blocks[bidx];
  const int w = B.w, h = B.h, nq = (w + 1) >> 1;
  const uint32_t lcup = B.length;
  const uint8_t* data = bytes + B.slot_off;
  HtBlockOut st;
  st.ms_len = 0; st.mel_len = 0; st.vlc_len = 0; st.total = 0;
  int scup = 0;
  if(lcup >= 2)
  {
    scup = ((int)__ldg(data + lcup - 1) << 4) + (int)(__ldg(data + lcup - 2) & 0xF);
    if(scup < 2 || scup > (int)lcup || scup > 4079 || B.mmsbs > 29)
      st.total = 2; /* malformed */
  }
  else
    st.total = lcup == 0 ? 1 : 2; /* 1: empty block (all zero), 2: malformed */
  if(st.total)
  {
    status[bidx] = st;
    return;
  }
  st.ms_len = lcup - (uint32_t)scup;

  MelFast mel;
  mel.d = data + lcup - scup;
  mel.size = scup - 1;
  mel.pos = mel.bits = mel.unstuff = mel.k = mel.run = mel.have = 0;
  mel.tmp = 0;
  melf_init(mel);
  VlcFast vlc;
  vlc.d = data;
  vlc.pos = (int)lcup - 3;
  vlc.lo = (int)lcup - scup;
  {
    const uint32_t d = __ldg(data + lcup - 2);
    vlc.tmp = d >> 4;
    vlc.bits = 4 - (((vlc.tmp & 7) == 7) ? 1 : 0);
    vlc.unstuff = (d | 0xF) > 0x8F;
  }
  vlcf_init(vlc);
  uint32_t* rec = recs + B.rec_off;
  /* significance of the bottom-left / bottom-right samples of the row above (p) and of this row (c), one bit per quad,
     32 quads per word */
  constexpr int NW = WIDE ? 16 : 1;
  const int nw = WIDE ? (nq + 31) >> 5 : 1;
  uint32_t pbl[NW] = {}, pbr[NW] = {};
  auto above = [&](int k) { /* bit j: something significant above-left or above quad 32 k + j (j up to 32) */
    uint64_t a = (uint64_t)pbl[k] | ((uint64_t)pbr[k] << 1);
    if constexpr(WIDE)
      a |= (k > 0 ? pbr[k - 1] >> 31 : 0u) | (k + 1 < NW ? (uint64_t)pbl[k + 1] << 32 : 0ull);
    return a;
  };

  for(int y = 0; y < h; y += 2)
  {
    const uint16_t* tbl = y ? tbl1 : tbl0;
    uint64_t A = above(0);
    uint32_t cbl[NW] = {}, cbr[NW] = {};
    int rho_left = 0;
    for(int q0 = 0; q0 < nq; q0 += 2)
    {
      const int k = WIDE ? q0 >> 5 : 0, qa = WIDE ? q0 & 31 : q0; /* the word holding quads q0, q0 + 1 and q0's bit in A */
      if(WIDE && qa == 0 && q0 > 0)
        A = above(k);
      vlcf_fill32(vlc);
      const bool has1 = q0 + 1 < nq;
      uint64_t tmp = vlc.tmp;
      /* ---- CxtVLC of the two quads ---- */
      const int cq0 = y == 0 ? ((rho_left >> 1) | (rho_left & 1))
                             : (int)(((A >> qa) & 1u) | ((rho_left & 0xC) ? 2u : 0u) | (((A >> (qa + 1)) & 1u) << 2));
      uint32_t t0 = tbl[(cq0 << 7) | ((uint32_t)tmp & 0x7F)];
      if(cq0 == 0 && !melf_symbol(mel))
        t0 = 0;
      tmp >>= (t0 >> 13);
      int used = (int)(t0 >> 13);
      const int rho0 = t0 & 0xF;
      uint32_t t1 = 0;
      int rho1 = 0;
      if(has1)
      {
        const int cq1 = y == 0 ? ((rho0 >> 1) | (rho0 & 1))
                               : (int)(((A >> (qa + 1)) & 1u) | ((rho0 & 0xC) ? 2u : 0u) | (((A >> (qa + 2)) & 1u) << 2));
        t1 = tbl[(cq1 << 7) | ((uint32_t)tmp & 0x7F)];
        if(cq1 == 0 && !melf_symbol(mel))
          t1 = 0;
        tmp >>= (t1 >> 13);
        used += (int)(t1 >> 13);
        rho1 = t1 & 0xF;
      }
      rho_left = has1 ? rho1 : rho0;
      cbl[k] |= ((uint32_t)((rho0 >> 1) & 1) << qa) | ((uint32_t)((rho1 >> 1) & 1) << (qa + 1));
      cbr[k] |= ((uint32_t)((rho0 >> 3) & 1) << qa) | ((uint32_t)((rho1 >> 3) & 1) << (qa + 1));
      /* ---- U-VLC of the pair: one look-up ---- */
      int u0 = 0, u1 = 0;
      const int uo = (int)((t0 >> 12) & 1u) | (int)(((t1 >> 12) & 1u) << 1);
      if(uo)
      {
        int mode = uo, add = 0;
        if(y == 0 && uo == 3)
        {
          if(melf_symbol(mel))
            add = 2; /* both > 2: the plain codes, offset by 2 */
          else
            mode = 4;
        }
        const uint32_t e = uvlc[mode * 64 + ((uint32_t)tmp & 63u)];
        const int plen = e & 7, l0 = (e >> 3) & 7, l1 = (e >> 6) & 7;
        tmp >>= plen;
        u0 = (int)((e >> 9) & 7u) + (int)((uint32_t)tmp & ((1u << l0) - 1u));
        tmp >>= l0;
        u1 = (int)((e >> 12) & 7u) + (int)((uint32_t)tmp & ((1u << l1) - 1u));
        tmp >>= l1;
        used += plen + l0 + l1;
        if(uo & 1)
          u0 += add;
        if(uo & 2)
          u1 += add;
      }
      vlc.tmp = tmp;
      vlc.bits -= used;
      rec[(size_t)q0 * 32] = (t0 & 0xFFFu) | ((uint32_t)u0 << 12); /* rho | e_k<<4 | e_1<<8 | u<<12 */
      if(has1)
        rec[(size_t)(q0 + 1) * 32] = (t1 & 0xFFFu) | ((uint32_t)u1 << 12);
    }
    rec += (size_t)nq * 32; /* records of 32 consecutive blocks are interleaved word by word */
    for(int i = 0; i < nw; ++i)
    {
      pbl[i] = cbl[i];
      pbr[i] = cbr[i];
    }
  }
  status[bidx] = st;
}

/* record per quad: rho[3:0] | e_k[7:4] | e_1[11:8] | u[17:12] */
/* IRREV: the launch's blocks are dequantised to float (one coding per launch); REFINE: some block of the launch carries
   SigProp / MagRef passes (foreign streams), so B.passes is looked at -- the common launch has neither branch compiled in */
template <bool IRREV, bool REFINE>
__global__ void __launch_bounds__(B2K_WARPS_PER_CTA * 32)
    k_ht_decode_magsgn(const HtBlockDesc* __restrict__ blocks, const uint8_t* __restrict__ bytes,
                       const uint32_t* __restrict__ recs, const HtBlockOut* __restrict__ status, uint32_t nblocks,
                       uint32_t line_entries, int* __restrict__ err)
{
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint32_t* rings = reinterpret_cast<uint32_t*>(smem_raw);
  uint16_t* lines_all = reinterpret_cast<uint16_t*>(rings + B2K_WARPS_PER_CTA * MS_RING_WORDS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bidx = blockIdx.x * B2K_WARPS_PER_CTA + warp;
  if(bidx >= nblocks)
    return;
  const HtBlockDesc B = blocks[bidx];
  const HtBlockOut st = status[bidx];
  uint32_t* ring = rings + warp * MS_RING_WORDS;
  uint16_t* const lines = lines_all + (size_t)warp * 2 * line_entries; /* two rows of bottom-sample exponents, used alternately */

  const int w = B.w, h = B.h, nq = (w + 1) >> 1;
  const int kmax = B.kmax;
  int32_t* coef = reinterpret_cast<int32_t*>(B.coef);
  bool bad = st.total == 2;
  if(st.total)
  { /* empty (not in any packet) or malformed: all coefficients zero */
    for(int y = 0; y < h; ++y)
      for(int x = lane; x < w; x += 32)
        coef[(size_t)y * B.pitch + x] = 0;
    if(lane == 0 && bad)
      atomicAdd(err, 1);
    return;
  }
  const uint8_t* data = bytes + B.slot_off;
  const int mmsbs = (int)B.mmsbs;
  const int p = 30 - mmsbs;
  const uint32_t mmsbp2 = (uint32_t)mmsbs + 2u;
  const int post_shift = 31 - kmax;

  for(int i = lane; i < MS_RING_WORDS; i += 32)
    ring[i] = 0;
  for(uint32_t i = lane; i < 2 * line_entries; i += 32)
    lines[i] = 0;
  __syncwarp();

  const int ms_size = (int)st.ms_len;
  int ms_pos = 0;
  uint32_t ms_head = 0, ms_tail = 0;
  bool ms_prevff = false;
  const uint32_t* rec = recs + B.rec_off;
  uint32_t r_next = lane < nq ? __ldg(rec + (size_t)lane * 32) : 0u;
  uint32_t pw0 = 0, pw1 = 0, pw2 = 0; /* this lane's three aligned words of the next 256-byte refill */
  auto load_chunk = [&](int pos) {
    if(pos + 8 * lane < ms_size)
    {
      const uint32_t* a = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(data + pos + 8 * lane) & ~(uintptr_t)3);
      pw0 = __ldg(a);
      pw1 = __ldg(a + 1);
      pw2 = __ldg(a + 2); /* at most 11 bytes past the lane's first: inside the arena's slack */
    }
  };
  load_chunk(0);

  const bool vec_ok = ((reinterpret_cast<uintptr_t>(coef) | ((uintptr_t)B.pitch << 2)) & 7u) == 0;
  for(int y = 0; y < h && !bad; y += 2)
  {
    const int cur = (y >> 1) & 1;
    const uint16_t* labove = lines + (cur ^ 1) * line_entries;
    uint16_t* lcur = lines + cur * line_entries;
    int32_t* const crow = coef + (size_t)y * B.pitch;
    for(int qb = 0; qb < nq; qb += 32)
    {
      /* keep at least 4096 un-stuffed bits (or the rest of the segment + 1-fill) in the ring: 256 segment bytes per
         round, 8 per lane, read as three aligned words (frwd_read L628-669: a byte after 0xFF carries 7 bits, 0xFF is fed
         once the segment is exhausted).  The un-stuffing is done on whole words: ff = the bytes equal to 0xFF (bit 7 of
         each), d = the bytes that follow one (their top bit is dropped), then two 16-bit halves are closed up. */
      while(ms_tail - ms_head < 4096u)
      {
        const int at = ms_pos + 8 * lane;
        uint32_t v0 = 0xFFFFFFFFu, v1 = 0xFFFFFFFFu;
        if(at < ms_size)
        {
          const int bsh = 8 * (int)(reinterpret_cast<uintptr_t>(data + at) & 3); /* loaded one refill ago */
          v0 = __funnelshift_r(pw0, pw1, bsh);
          v1 = __funnelshift_r(pw1, pw2, bsh);
          const int left = ms_size - at;
          if(left < 8)
          {
            if(left < 4)
              v0 |= 0xFFFFFFFFu << (8 * left);
            v1 = left > 4 ? (v1 | (0xFFFFFFFFu << (8 * (left - 4)))) : 0xFFFFFFFFu;
          }
        }
        load_chunk(ms_pos + 256); /* the next 256 bytes are in flight while these are parsed */
        const uint32_t ff0 = ((v0 & 0x7F7F7F7Fu) + 0x01010101u) & v0 & 0x80808080u;
        const uint32_t ff1 = ((v1 & 0x7F7F7F7Fu) + 0x01010101u) & v1 & 0x80808080u;
        const unsigned lastff = __ballot_sync(0xffffffffu, (ff1 >> 31) != 0);
        const uint32_t fin = lane == 0 ? (ms_prevff ? 1u : 0u) : ((lastff >> (lane - 1)) & 1u);
        const uint32_t d0 = (ff0 << 8) | (fin << 7), d1 = (ff1 << 8) | (ff0 >> 24);
        auto squeeze = [](uint32_t v, uint32_t d, int& nb) -> uint32_t {
          v &= ~d;
          uint32_t h0 = v & 0xFFFFu, h1 = v >> 16;
          if(d & 0x80u)
            h0 = (h0 & 0xFFu) | ((h0 & 0xFF00u) >> 1);
          if(d & 0x800000u)
            h1 = (h1 & 0xFFu) | ((h1 & 0xFF00u) >> 1);
          nb = 32 - __popc(d);
          return h0 | (h1 << (16 - __popc(d & 0x8080u))); /* a dropped top bit was masked to 0: the next piece lands on it */
        };
        int nb0, nb1;
        const uint32_t a0 = squeeze(v0, d0, nb0), a1 = squeeze(v1, d1, nb1);
        const uint64_t acc = (uint64_t)a0 | ((uint64_t)a1 << nb0);
        uint32_t tot;
        const uint32_t off = warp_excl_scan_d<uint32_t>((uint32_t)(nb0 + nb1), lane, tot);
        const uint32_t pos = ms_tail + off;
        { /* the words this refill lands in are cleared here (65 whole words after the one the tail sits in; the unread
             bits span fewer than 128 of the ring's 256 words): the consumer does not clean up behind itself */
          const uint32_t wt = ms_tail >> 5;
          ring[(wt + 1 + lane) & (MS_RING_WORDS - 1)] = 0;
          ring[(wt + 33 + lane) & (MS_RING_WORDS - 1)] = 0;
          if(lane == 0)
            ring[(wt + 65) & (MS_RING_WORDS - 1)] = 0;
          __syncwarp();
        }
        {
          const int sh = pos & 31;
          const uint32_t wi = pos >> 5;
          const uint64_t sft = acc << sh;
          const uint32_t lo = (uint32_t)sft, mid = (uint32_t)(sft >> 32), hi = sh ? (uint32_t)(acc >> (64 - sh)) : 0u;
          if(lo)
            atomicOr(&ring[wi & (MS_RING_WORDS - 1)], lo);
          if(mid)
            atomicOr(&ring[(wi + 1) & (MS_RING_WORDS - 1)], mid);
          if(hi)
            atomicOr(&ring[(wi + 2) & (MS_RING_WORDS - 1)], hi);
        }
        ms_tail += tot;
        ms_prevff = (lastff >> 31) & 1u;
        ms_pos += 256;
        __syncwarp();
      }

      const int q = qb + lane, x = 2 * q;
      const bool qv = q < nq;
      const uint32_t r = r_next; /* loaded one step ago (the interleaved records are a 32-sector gather: latency, not bandwidth) */
      {
        int qn = qb + 32 + lane, yn = y;
        const uint32_t* recn = rec;
        if(qb + 32 >= nq)
        {
          qn = lane;
          yn = y + 2;
          recn = rec + (size_t)nq * 32;
        }
        r_next = (yn < h && qn < nq) ? __ldg(recn + (size_t)qn * 32) : 0u;
      }
      const int rho = r & 0xF, ekq = (r >> 4) & 0xF, e1q = (r >> 8) & 0xF, uq = (int)(r >> 12);
      int kappa = 1;
      if(y > 0 && qv)
      {
        const uint32_t a = labove[q], b = labove[q + 1], c = labove[q + 2];
        const int emx = max(max((int)(a >> 8), (int)(b & 0xFF)), max((int)(b >> 8), (int)(c & 0xFF)));
        kappa = (rho & (rho - 1)) ? max(1, emx) : 1;
      }
      const uint32_t U = (uint32_t)(uq + kappa);
      if(qv && U > mmsbp2)
        bad = true;
      /* the samples this lane reads MagSgn bits for: none past the block's right edge (the reference never reads bits for
         the missing right column, L1138-1139), none once the block is known to be damaged */
      const int rho_eff = (qv && !bad) ? ((x + 1 < w) ? rho : (rho & 3)) : 0;
      int m[4], mlen = 0;
#pragma unroll
      for(int i = 0; i < 4; ++i)
      {
        m[i] = ((rho_eff >> i) & 1) ? (int)U - ((ekq >> i) & 1) : 0;
        mlen += m[i];
      }
      uint32_t total;
      const uint32_t off = warp_excl_scan_d<uint32_t>((uint32_t)mlen, lane, total);
      const uint32_t pos = ms_head + off;
      const uint32_t wi = pos >> 5;
      const int sh = pos & 31;
      uint32_t wv[5];
#pragma unroll
      for(int i = 0; i < 5; ++i)
        wv[i] = ring[(wi + i) & (MS_RING_WORDS - 1)];
      uint32_t bits[4];
#pragma unroll
      for(int i = 0; i < 4; ++i)
        bits[i] = __funnelshift_r(wv[i], wv[i + 1], sh);
      /* branch-free over the quad's four samples (an insignificant one has m = 0 and its value is dropped at the end):
         the window moves on by m bits after each sample; a later sample can only need what is left of 93, 62 and 31 bits,
         so the shifts shrink from three words to one */
      uint32_t w0 = bits[0], w1 = bits[1], w2 = bits[2];
      const uint32_t w3 = bits[3];
      int ebot[2] = {0, 0};
      uint32_t outv[4];
      const bool refine = REFINE && B.passes > 1;
#pragma unroll
      for(int i = 0; i < 4; ++i)
      {
        const bool on = ((rho_eff >> i) & 1) != 0;
        const int mi = m[i]; /* <= 31 (U <= mmsbs + 2 <= 31) */
        const uint32_t msv = w0;
        if(i == 0)
        {
          w0 = __funnelshift_r(w0, w1, mi);
          w1 = __funnelshift_r(w1, w2, mi);
          w2 = __funnelshift_r(w2, w3, mi);
        }
        else if(i == 1)
        {
          w0 = __funnelshift_r(w0, w1, mi);
          w1 = __funnelshift_r(w1, w2, mi);
        }
        else if(i == 2)
          w0 = __funnelshift_r(w0, w1, mi);
        uint32_t v_n = msv & ((1u << mi) - 1u);
        v_n |= (uint32_t)((e1q >> i) & 1) << mi;
        v_n |= 1u;
        const uint32_t mag = ((v_n + 2u) << (p - 1)) & 0x7FFFFFFFu;
        const uint32_t sgn = msv & 1u;
        if(i & 1)
          ebot[i >> 1] = on ? 31 - __clz(v_n | 2u) : 0;
        uint32_t val;
        if(refine)
          val = (sgn << 31) | mag; /* k_ht_decode_refine finishes and dequantises the block */
        else if(!IRREV)
        {
          const int32_t mv = (int32_t)(mag >> post_shift);
          val = (uint32_t)(sgn ? -mv : mv);
        }
        else
          val = __float_as_uint(__fmul_rn((float)(int32_t)mag, B.quant)) | (sgn << 31); /* quant > 0: the sign bit is free */
        outv[i] = on ? val : 0u;
      }
      if(qv)
      {
        int32_t* c0 = crow + x; /* (x, y); the row below at + pitch */
        if(vec_ok && x + 1 < w)
        { /* the lane's two columns of a row are one aligned 8-byte store: a row of the warp is 256 contiguous bytes */
          *reinterpret_cast<uint2*>(c0) = make_uint2(outv[0], outv[2]);
          if(y + 1 < h)
            *reinterpret_cast<uint2*>(c0 + B.pitch) = make_uint2(outv[1], outv[3]);
        }
        else
        {
          c0[0] = (int32_t)outv[0];
          if(x + 1 < w)
            c0[1] = (int32_t)outv[2];
          if(y + 1 < h)
          {
            c0[B.pitch] = (int32_t)outv[1];
            if(x + 1 < w)
              c0[B.pitch + 1] = (int32_t)outv[3];
          }
        }
      }
      if(qv)
        lcur[q + 1] = (uint16_t)(ebot[0] | (ebot[1] << 8));
      ms_head += total;
      bad = __any_sync(0xffffffffu, bad);
      __syncwarp();
    }
    rec += (size_t)nq * 32; /* records of 32 consecutive blocks are interleaved word by word */
  }
  if(bad)
  {
    __syncwarp();
    for(int y = 0; y < h; ++y)
      for(int x = lane; x < w; x += 32)
        coef[(size_t)y * B.pitch + x] = 0;
    if(lane == 0)
      atomicAdd(err, 1);
  }
}

/* ---- SigProp + MagRef ------------------------------------------------------------------------------
 * One warp per block that carries refinement passes.  Both passes are bit-serial by construction (a
 * sample's membership depends on what the previous samples of the scan decoded), so lane 0 walks the
 * scan while the warp does the memory work around it: per stripe of 4 rows the lanes turn the block's
 * words into significance bitmaps with ballots (coalesced loads), lane 0 decodes the stripe against
 * those bitmaps, and the lanes write the new / refined samples back (coalesced stores).
 * Scan, membership and the two bit streams: see oracle/j2k_oracle.c "HT refinement passes", which is
 * the restatement this kernel is tested against.  Any block width (<= 1024) and height. */
constexpr int RF_WORDS = 32; /* bitmap words per row: 1024 columns */
struct RefineRows
{
  uint32_t sig[6][RF_WORDS]; /* [0] row above the stripe, [1..4] the stripe, [5] row below (cleanup only) */
  uint32_t nw[4][RF_WORDS];  /* SigProp: newly significant / MagRef: samples to refine */
  uint32_t sg[4][RF_WORDS];  /* SigProp: signs of the new samples / MagRef: decoded bit */
};
__device__ __forceinline__ uint32_t rf_bit(const uint32_t* row, int x, int w)
{
  return (x < 0 || x >= w) ? 0u : ((row[x >> 5] >> (x & 31)) & 1u);
}
__device__ __forceinline__ uint32_t rf_window6(const uint32_t* row, int x0, int w)
{ /* bits of columns x0 .. x0+5 */
  uint32_t v = 0;
#pragma unroll
  for(int i = 0; i < 6; ++i)
    v |= rf_bit(row, x0 + i, w) << i;
  return v;
}
struct SppR
{ /* forward reader, zeros after the end (frwd_read<0>, L609-654) */
  const uint8_t* d;
  int size, pos, bits, unstuff;
  uint32_t tmp;
};
__device__ __forceinline__ uint32_t spp_get(SppR& s)
{
  if(s.bits == 0)
  {
    const uint32_t b = s.pos < s.size ? (uint32_t)__ldg(s.d + s.pos) : 0u;
    s.pos++;
    s.tmp = b;
    s.bits = 8 - s.unstuff;
    s.unstuff = (b == 0xFFu);
  }
  const uint32_t v = s.tmp & 1u;
  s.tmp >>= 1;
  s.bits--;
  return v;
}
struct MrpR
{ /* backward reader (rev_read_mrp / rev_init_mrp, L453-541) */
  const uint8_t* last;
  int size, pos, bits, unstuff;
  uint32_t tmp;
};
__device__ __forceinline__ uint32_t mrp_get(MrpR& m)
{
  if(m.bits == 0)
  {
    const uint32_t b = m.pos < m.size ? (uint32_t)__ldg(m.last - m.pos) : 0u;
    m.pos++;
    m.tmp = b;
    m.bits = 8 - ((m.unstuff && (b & 0x7Fu) == 0x7Fu) ? 1 : 0);
    m.unstuff = b > 0x8Fu;
  }
  const uint32_t v = m.tmp & 1u;
  m.tmp >>= 1;
  m.bits--;
  return v;
}

__global__ void __launch_bounds__(B2K_WARPS_PER_CTA * 32)
    k_ht_decode_refine(const HtBlockDesc* __restrict__ blocks, const uint8_t* __restrict__ bytes,
                       const HtBlockOut* __restrict__ status, uint32_t nblocks, int stripe_causal)
{
  __shared__ RefineRows rows_all[B2K_WARPS_PER_CTA];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bidx = blockIdx.x * B2K_WARPS_PER_CTA + warp;
  if(bidx >= nblocks)
    return;
  const HtBlockDesc B = blocks[bidx];
  if(B.passes <= 1 || status[bidx].total != 0) /* cleanup-only blocks are finished; empty / rejected ones are zero */
    return;
  RefineRows& R = rows_all[warp];
  const int w = B.w, h = B.h, nwords = (w + 31) >> 5;
  const int p = 30 - (int)B.mmsbs;
  uint32_t* coef = reinterpret_cast<uint32_t*>(B.coef);
  const uint8_t* seg = bytes + B.slot_off + B.length;
  const uint32_t newval = 3u << (p - 2);

  /* row y of the block as a "non-zero" bitmap (cleanup significance while SigProp has not reached it) */
  auto load_row = [&](uint32_t* dst, int y) {
    for(int xb = 0; xb < nwords * 32; xb += 32)
    {
      const int x = xb + lane;
      const uint32_t v = (y >= 0 && y < h && x < w) ? coef[(size_t)y * B.pitch + x] : 0u;
      const unsigned m = __ballot_sync(0xffffffffu, (v & 0x7FFFFFFFu) != 0u);
      if(lane == 0)
        dst[xb >> 5] = m;
    }
  };

  /* ---------------- SigProp ---------------- */
  SppR sp{seg, (int)B.length2, 0, 0, 0, 0u};
  for(int i = lane; i < RF_WORDS; i += 32)
    R.sig[0][i] = 0;
  for(int y0 = 0; y0 < h; y0 += 4)
  {
    for(int k = 1; k <= 5; ++k)
      load_row(R.sig[k], (k == 5 && stripe_causal) ? -1 : y0 + k - 1);
    for(int k = 0; k < 4; ++k)
      for(int i = lane; i < nwords; i += 32)
      {
        R.nw[k][i] = 0;
        R.sg[k][i] = 0;
      }
    __syncwarp();
    if(lane == 0)
    {
      const int rows = min(4, h - y0);
      for(int gx = 0; gx < w; gx += 4)
      {
        uint32_t S[6], C[4];
#pragma unroll
        for(int k = 0; k < 6; ++k)
          S[k] = rf_window6(R.sig[k], gx - 1, w);
#pragma unroll
        for(int k = 0; k < 4; ++k)
          C[k] = S[k + 1];
        uint32_t found = 0; /* bit 4c+r: sample (r, c) of the group became significant */
        for(int c = 0; c < 4 && gx + c < w; ++c)
          for(int r = 0; r < rows; ++r)
          {
            if((C[r] >> (c + 1)) & 1u)
              continue;
            const uint32_t nb = ((S[r] | S[r + 1] | S[r + 2]) >> c) & 7u;
            if(!nb)
              continue;
            if(spp_get(sp))
            {
              S[r + 1] |= 1u << (c + 1);
              found |= 1u << (4 * c + r);
            }
          }
        while(found)
        {
          const int i = __ffs(found) - 1;
          found &= found - 1;
          const int c = i >> 2, r = i & 3, x = gx + c;
          const uint32_t bit = 1u << (x & 31);
          R.sig[r + 1][x >> 5] |= bit;
          R.nw[r][x >> 5] |= bit;
          if(spp_get(sp))
            R.sg[r][x >> 5] |= bit;
        }
      }
    }
    __syncwarp();
    for(int r = 0; r < 4 && y0 + r < h; ++r)
      for(int x = lane; x < w; x += 32)
        if((R.nw[r][x >> 5] >> (x & 31)) & 1u)
          coef[(size_t)(y0 + r) * B.pitch + x] = (((R.sg[r][x >> 5] >> (x & 31)) & 1u) << 31) | newval;
    for(int i = lane; i < nwords; i += 32)
      R.sig[0][i] = R.sig[4][i]; /* the stripe's last row, new samples included, is the next stripe's row above */
    __syncwarp();
  }

  /* ---------------- MagRef ---------------- */
  if(B.passes > 2)
  {
    MrpR mr{seg + B.length2 - 1, (int)B.length2, 0, 0, 1, 0u};
    for(int y0 = 0; y0 < h; y0 += 4)
    {
      for(int k = 0; k < 4; ++k)
      { /* members: significant after the cleanup pass, i.e. non-zero and not one of SigProp's samples */
        const int y = y0 + k;
        for(int xb = 0; xb < nwords * 32; xb += 32)
        {
          const int x = xb + lane;
          const uint32_t v = (y < h && x < w) ? (coef[(size_t)y * B.pitch + x] & 0x7FFFFFFFu) : 0u;
          const unsigned m = __ballot_sync(0xffffffffu, v != 0u && v != newval);
          if(lane == 0)
          {
            R.nw[k][xb >> 5] = m;
            R.sg[k][xb >> 5] = 0;
          }
        }
      }
      __syncwarp();
      if(lane == 0)
        for(int x = 0; x < w; ++x)
#pragma unroll
          for(int r = 0; r < 4; ++r)
            if((R.nw[r][x >> 5] >> (x & 31)) & 1u)
              if(mrp_get(mr))
                R.sg[r][x >> 5] |= 1u << (x & 31);
      __syncwarp();
      for(int r = 0; r < 4 && y0 + r < h; ++r)
        for(int x = lane; x < w; x += 32)
          if((R.nw[r][x >> 5] >> (x & 31)) & 1u)
          {
            const uint32_t bit = (R.sg[r][x >> 5] >> (x & 31)) & 1u;
            coef[(size_t)(y0 + r) * B.pitch + x] ^= ((1u - bit) << (p - 1)) | (1u << (p - 2));
          }
      __syncwarp();
    }
  }

  /* ---------------- dequantise in place (PostDecodeFiltersOJPH.h L48-66 / L100-119) ---------------- */
  const int post_shift = 31 - (int)B.kmax;
  for(int y = 0; y < h; ++y)
    for(int x = lane; x < w; x += 32)
    {
      const uint32_t v = coef[(size_t)y * B.pitch + x];
      const uint32_t mag = v & 0x7FFFFFFFu;
      uint32_t outv;
      if(!B.irreversible)
      {
        const int32_t mv = (int32_t)(mag >> post_shift);
        outv = (uint32_t)((v >> 31) ? -mv : mv);
      }
      else
      {
        float f = __fmul_rn((float)(int32_t)mag, B.quant);
        if(v >> 31)
          f = -f;
        outv = __float_as_uint(f);
      }
      coef[(size_t)y * B.pitch + x] = outv;
    }
}

} /* namespace */

/* decode descriptors of the engine's OWN last encode, built on the device (device-resident round trip):
   length/offset from the encoder's outputs, numbps = 1 as the encoder signals (CoderOJPH.cpp L203-206) */
namespace {
__global__ void k_build_dec_desc(const HtBlockDesc* __restrict__ enc, const HtBlockOut* __restrict__ outs,
                                 const uint64_t* __restrict__ offsets, const float* __restrict__ dec_quant,
                                 HtBlockDesc* __restrict__ dec, uint32_t n)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n)
    return;
  HtBlockDesc d = enc[i];
  const uint32_t t = outs[i].total;
  d.length = t == 0xFFFFFFFFu ? 0 : t;
  d.slot_off = offsets[i];
  d.mmsbs = (uint8_t)(d.kmax - 1);
  d.passes = 1;
  d.length2 = 0;
  d.quant = dec_quant[i];
  dec[i] = d;
}
} // namespace
void b2k_launch_build_dec_desc(const HtBlockDesc* d_enc, const HtBlockOut* d_out, const uint64_t* d_offsets,
                               const float* d_dec_quant, HtBlockDesc* d_dec, uint32_t n, cudaStream_t st)
{
  if(!n)
    return;
  k_build_dec_desc<<<(n + 255) / 256, 256, 0, st>>>(d_enc, d_out, d_offsets, d_dec_quant, d_dec, n);
  b2k_count_launch();
}

void b2k_launch_ht_decode_vlc(const HtBlockDesc* d_blocks, const uint8_t* d_bytes, uint32_t* d_recs, HtBlockOut* d_status,
                              uint32_t nblocks, uint32_t max_w, cudaStream_t st)
{
  if(!nblocks)
    return;
  /* 32 threads per CTA: the kernel is a serial chain per thread, so spread the blocks over as many
     SMs as possible instead of packing 4 warps onto one */
  if(max_w > 64)
    k_ht_decode_vlc<true><<<(nblocks + 31) / 32, 32, 0, st>>>(d_blocks, d_bytes, d_recs, d_status, nblocks);
  else
    k_ht_decode_vlc<false><<<(nblocks + 31) / 32, 32, 0, st>>>(d_blocks, d_bytes, d_recs, d_status, nblocks);
  b2k_count_launch();
}

void b2k_launch_ht_decode_magsgn(const HtBlockDesc* d_blocks, const uint8_t* d_bytes, const uint32_t* d_recs,
                                 const HtBlockOut* d_status, uint32_t nblocks, uint32_t max_w, int* d_err, int irreversible,
                                 int any_refinement, cudaStream_t st)
{
  if(!nblocks)
    return;
  const uint32_t line_entries = ((max_w + 1) / 2 + 4 + 1) & ~1u;
  const size_t smem = (size_t)B2K_WARPS_PER_CTA * MS_RING_WORDS * sizeof(uint32_t) +
                      (size_t)B2K_WARPS_PER_CTA * 2 * line_entries * sizeof(uint16_t);
  const uint32_t grid = (nblocks + B2K_WARPS_PER_CTA - 1) / B2K_WARPS_PER_CTA;
  using Kernel = void (*)(const HtBlockDesc*, const uint8_t*, const uint32_t*, const HtBlockOut*, uint32_t, uint32_t, int*);
  static const Kernel variants[4] = {k_ht_decode_magsgn<false, false>, k_ht_decode_magsgn<false, true>,
                                     k_ht_decode_magsgn<true, false>, k_ht_decode_magsgn<true, true>};
  variants[(irreversible ? 2 : 0) + (any_refinement ? 1 : 0)]<<<grid, B2K_WARPS_PER_CTA * 32, smem, st>>>(
      d_blocks, d_bytes, d_recs, d_status, nblocks, line_entries, d_err);
  b2k_count_launch();
}

void b2k_launch_ht_decode_refine(const HtBlockDesc* d_blocks, const uint8_t* d_bytes, const HtBlockOut* d_status,
                                 uint32_t nblocks, int stripe_causal, cudaStream_t st)
{
  if(!nblocks)
    return;
  const uint32_t grid = (nblocks + B2K_WARPS_PER_CTA - 1) / B2K_WARPS_PER_CTA;
  k_ht_decode_refine<<<grid, B2K_WARPS_PER_CTA * 32, 0, st>>>(d_blocks, d_bytes, d_status, nblocks, stripe_causal);
  b2k_count_launch();
}

void b2k_launch_ht_decode(const HtBlockDesc* d_blocks, const uint8_t* d_bytes, uint32_t* d_recs, HtBlockOut* d_status,
                          uint32_t nblocks, uint32_t max_w, int* d_err, int irreversible, int any_refinement, cudaStream_t st)
{
  b2k_launch_ht_decode_vlc(d_blocks, d_bytes, d_recs, d_status, nblocks, max_w, st);
  b2k_launch_ht_decode_magsgn(d_blocks, d_bytes, d_recs, d_status, nblocks, max_w, d_err, irreversible, any_refinement, st);
}
