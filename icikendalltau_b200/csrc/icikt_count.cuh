// icikt_count.cuh -- the memory-space accessors and pass A, the bucket-free inversion-counting
// pass on 16-bit keys (see icikt_pairs.cu for the counting scheme).  Shared by the pair kernel
// (icikt_pairs.cu) and the fused column kernel (icikt_columns.cu), which runs the pass on the
// column's own sorted ranks to get the per-column constant `cconst`.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace icikt {
namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}
__device__ __forceinline__ uint32_t lanemask_le() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_le;" : "=r"(m));
  return m;
}
// lanes strictly below the highest set bit of `bits` (bits != 0)
__device__ __forceinline__ uint32_t below_top(uint32_t bits) {
  return (1u << (31 - __clz((int)bits))) - 1u;
}

// ---- memory-space accessors ----------------------------------------------------------------
// The counting passes run either on shared memory (32-bit shared-window addresses, explicit
// ld/st.shared) or, for vectors too long for one CTA's shared memory, on a per-CTA scratch in
// global memory that stays L2-resident.  Offsets are in bytes.
__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
// Constants handed over as kernel parameters so that the assembler keeps multiplications by
// them as IMAD / IMAD.HI (FMA pipe) instead of strength-reducing them to integer-ALU shifts/adds.
struct PipeConst {
  uint32_t one, two, c64k;
  uint32_t c4410, c4432;  // PRMT selectors: low / high 16-bit half of a register, zero-extended
};
__host__ __device__ inline PipeConst make_pipe_const() {
  PipeConst pc;
  pc.one = 1u;
  pc.two = 2u;
  pc.c64k = 65536u;
  pc.c4410 = 0x4410u;
  pc.c4432 = 0x4432u;
  return pc;
}

// Pass A's low-nibble level (count_pass, after the two-bit levels down to bit 4).  For a key with low
// nibble b3 b2 b1 b0, the four one-bit levels below bit 4 add, at every bit whose value is 0, the keys
// before it that agree with it on the nibble's higher bits and have that bit set: a binary tree of 15
// nodes.  Earlier buckets and the other subtrees only add terms that depend on column y alone (cconst
// takes them), so ONE sweep over the order the last two-bit level left counts all four bits, and
// nothing has to be stored.  A thread keeps the counts of its range's keys seen so far in byte fields
// (a range holds R = 8 kk <= 255 keys):
//   C    keys per class (b3 b2)            root: c2 + c3 ones, node b3: c(2 b3 + 1) ones
//   D2   ones of b1 per (b3 b2)
//   D3a  ones of b0 per (b2 b1), b3 = 0;  D3b the same for b3 = 1
// Every key adds, unpredicated, the ones counters of the four nodes on its path (one dp4a per register,
// C with byte weights 0,1,1,1 or 0,0,1,2); the keys with bit 1 at a node add C(n1, 2) there in all,
// which nibble_level takes back out in closed form.
struct NibbleCounts {
  uint32_t C, D2, D3a, D3b, acc;
};

// ---- TMA bulk copy global -> shared, completion on an mbarrier (sm_90+) ---------------------
// Used for the one contiguous bulk transfer of the pair kernel: y's dense-rank table into the
// second sequence buffer.  One thread issues it; the copy engine moves the bytes while the CTA
// does the bit-mask counting, then everybody waits on the barrier's phase.
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
  // earlier generic-proxy accesses to the destination are ordered before the async-proxy writes
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(mbar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(mbar), "r"(parity)
        : "memory");
  } while (!done);
}

template <bool G>
struct Mem;
template <>
struct Mem<false> {
  typedef uint32_t ptr;
  static __device__ __forceinline__ ptr add(ptr p, int32_t bytes) { return p + (uint32_t)bytes; }
  static __device__ __forceinline__ uint32_t ld16(ptr p) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(p) : "memory");
    return v;
  }
  // 16-bit load zero-extended straight into a 32-bit register (no conversion afterwards)
  static __device__ __forceinline__ uint32_t ld16w(ptr p) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(p) : "memory");
    return v;
  }
  static __device__ __forceinline__ uint32_t ld32(ptr p) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(p) : "memory");
    return v;
  }
  static __device__ __forceinline__ void ld128(ptr p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(p) : "memory");
  }
  // position of p for the inversion accumulator: any value that differs from the byte offset
  // inside the buffer by a per-level constant (here the shared-window address itself)
  static __device__ __forceinline__ uint32_t off(ptr p, ptr) { return p; }
  // a + b on the FMA pipe (IMAD with a multiplier the assembler cannot fold): the integer ALU
  // pipe is the binding one in pass A, both pipes issue one warp instruction per two cycles
  static __device__ __forceinline__ uint32_t fadd(uint32_t a, uint32_t b, uint32_t one) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(one), "r"(b));
    return d;
  }
  // high 16-bit key of a word on the FMA pipe (IMAD.HI by 65536)
  static __device__ __forceinline__ uint32_t hi16(uint32_t w, uint32_t c64k) {
    uint32_t d;
    asm("mul.hi.u32 %0, %1, %2;" : "=r"(d) : "r"(w), "r"(c64k));
    return d;
  }
  // one key of pass A's scatter sweep (two bits per level, see count_pass): Q01/Q23 hold the
  // next free slot (element index, 16 bits each) of digit classes 0|1 and 2|3.  acc2 sums, over
  // ALL keys, the running slot of the key's lo = 1 sibling class (one IMAD.HI on the FMA pipe, no
  // predicate); count_pass takes the lo = 1 keys' own share back out in closed form.  `two` and the
  // other constants are registers the assembler cannot fold, so the slot address is an IMAD and
  // not an LEA.  11 instructions per key.
  static __device__ __forceinline__ void step4(uint32_t& Q01, uint32_t& Q23, uint32_t& acc2, uint32_t w,
                                               uint32_t bit_lo, uint32_t bit_hi, uint32_t key, ptr base,
                                               const PipeConst& pc) {
    asm volatile(
        "{\n\t"
        ".reg .pred ph, pl;\n\t"
        ".reg .b32 t, qs, sel, idx, ad, inc;\n\t"
        "and.b32 t, %3, %5;\n\t"
        "setp.ne.u32 ph, t, 0;\n\t"
        "and.b32 t, %3, %4;\n\t"
        "setp.ne.u32 pl, t, 0;\n\t"
        "selp.b32 qs, %1, %0, ph;\n\t"
        "mad.hi.u32 %2, qs, %9, %2;\n\t"
        "selp.b32 sel, %11, %10, pl;\n\t"
        "prmt.b32 idx, qs, 0, sel;\n\t"
        "mad.lo.u32 ad, idx, %8, %7;\n\t"
        "st.shared.u16 [ad], %6;\n\t"
        "selp.b32 inc, %9, %12, pl;\n\t"
        "@ph add.u32 %1, %1, inc;\n\t"
        "@!ph add.u32 %0, %0, inc;\n\t"
        "}"
        : "+r"(Q01), "+r"(Q23), "+r"(acc2)
        : "r"(w), "r"(bit_lo), "r"(bit_hi), "h"((unsigned short)key), "r"(base), "r"(pc.two), "r"(pc.c64k),
          "r"(pc.c4410), "r"(pc.c4432), "r"(pc.one)
        : "memory");
  }
  // one key of the low-nibble level (see NibbleCounts): the key's nibble sits at bit SH of w, a2 / a3 hold
  // 8*(b3 b2) / 8*(b2 b1) in their low five bits (a shift by a register uses those only).  ~16 instructions.
  template <int SH>
  static __device__ __forceinline__ void step16(NibbleCounts& s, uint32_t w, uint32_t a2, uint32_t a3) {
    asm volatile(
        "{\n\t"
        ".reg .pred p3, p1, p0;\n\t"
        ".reg .b32 t, W1, W2, W3, Ds;\n\t"
        "and.b32 t, %5, %8;\n\t"
        "setp.ne.u32 p3, t, 0;\n\t"
        "and.b32 t, %5, %9;\n\t"
        "setp.ne.u32 p1, t, 0;\n\t"
        "and.b32 t, %5, %10;\n\t"
        "setp.ne.u32 p0, t, 0;\n\t"
        "selp.b32 W1, 0x02010000, 0x01010100, p3;\n\t"
        "dp4a.u32.u32 %4, %0, W1, %4;\n\t"
        "shf.l.wrap.b32 W2, 0, 1, %6;\n\t"
        "add.u32 %0, %0, W2;\n\t"
        "dp4a.u32.u32 %4, %1, W2, %4;\n\t"
        "@p1 add.u32 %1, %1, W2;\n\t"
        "shf.l.wrap.b32 W3, 0, 1, %7;\n\t"
        "selp.b32 Ds, %3, %2, p3;\n\t"
        "dp4a.u32.u32 %4, Ds, W3, %4;\n\t"
        "selp.b32 W3, W3, 0, p0;\n\t"
        "@p3 add.u32 %3, %3, W3;\n\t"
        "@!p3 add.u32 %2, %2, W3;\n\t"
        "}"
        : "+r"(s.C), "+r"(s.D2), "+r"(s.D3a), "+r"(s.D3b), "+r"(s.acc)
        : "r"(w), "r"(a2), "r"(a3), "n"(8u << SH), "n"(2u << SH), "n"(1u << SH));
  }
  // step16 at a bit position known at run time only (a radix-16 level, see radix_level): m8 / m2 / m1 are the
  // masks of the key's digit bits 3 / 1 / 0 in w
  static __device__ __forceinline__ void step16_at(NibbleCounts& s, uint32_t w, uint32_t a2, uint32_t a3, uint32_t m8,
                                                   uint32_t m2, uint32_t m1) {
    asm volatile(
        "{\n\t"
        ".reg .pred p3, p1, p0;\n\t"
        ".reg .b32 t, W1, W2, W3, Ds;\n\t"
        "and.b32 t, %5, %8;\n\t"
        "setp.ne.u32 p3, t, 0;\n\t"
        "and.b32 t, %5, %9;\n\t"
        "setp.ne.u32 p1, t, 0;\n\t"
        "and.b32 t, %5, %10;\n\t"
        "setp.ne.u32 p0, t, 0;\n\t"
        "selp.b32 W1, 0x02010000, 0x01010100, p3;\n\t"
        "dp4a.u32.u32 %4, %0, W1, %4;\n\t"
        "shf.l.wrap.b32 W2, 0, 1, %6;\n\t"
        "add.u32 %0, %0, W2;\n\t"
        "dp4a.u32.u32 %4, %1, W2, %4;\n\t"
        "@p1 add.u32 %1, %1, W2;\n\t"
        "shf.l.wrap.b32 W3, 0, 1, %7;\n\t"
        "selp.b32 Ds, %3, %2, p3;\n\t"
        "dp4a.u32.u32 %4, Ds, W3, %4;\n\t"
        "selp.b32 W3, W3, 0, p0;\n\t"
        "@p3 add.u32 %3, %3, W3;\n\t"
        "@!p3 add.u32 %2, %2, W3;\n\t"
        "}"
        : "+r"(s.C), "+r"(s.D2), "+r"(s.D3a), "+r"(s.D3b), "+r"(s.acc)
        : "r"(w), "r"(a2), "r"(a3), "r"(m8), "r"(m2), "r"(m1));
  }
  // one key of a radix-16 level's scatter: its digit d = (key >> s) & 15 selects this thread's slot counter
  // cnt[d] (u16, at me + d * row), the key goes to that slot of buffer `base` and the counter moves on.  The
  // key's high 16 bits are ignored.  8 instructions, three of them on the FMA pipe.
  static __device__ __forceinline__ void scatter16(uint32_t key, uint32_t s, uint32_t me, uint32_t row, ptr base,
                                                   const PipeConst& pc) {
    asm volatile(
        "{\n\t"
        ".reg .b32 d, ca, sl, ad;\n\t"
        "shr.b32 d, %0, %1;\n\t"
        "and.b32 d, d, 15;\n\t"
        "mad.lo.u32 ca, d, %3, %2;\n\t"
        "ld.shared.u16 sl, [ca];\n\t"
        "mad.lo.u32 ad, sl, %5, %4;\n\t"
        "st.shared.u16 [ad], %0;\n\t"
        "mad.lo.u32 sl, %6, %6, sl;\n\t"
        "st.shared.u16 [ca], sl;\n\t"
        "}" ::"r"(key),
        "r"(s), "r"(me), "r"(row), "r"(base), "r"(pc.two), "r"(pc.one)
        : "memory");
  }
  static __device__ __forceinline__ void red_add32(ptr p, uint32_t v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(p), "r"(v) : "memory");
  }
  static __device__ __forceinline__ uint32_t atom_or32(ptr p, uint32_t v) {  // returns the old word
    uint32_t old;
    asm volatile("atom.shared.or.b32 %0, [%1], %2;" : "=r"(old) : "r"(p), "r"(v) : "memory");
    return old;
  }
  static __device__ __forceinline__ ptr from_shared(const void* q) { return smem_addr(q); }
  static __device__ __forceinline__ void st16(ptr p, uint32_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(p), "h"((unsigned short)v) : "memory");
  }
  static __device__ __forceinline__ void st32(ptr p, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(p), "r"(v) : "memory");
  }
  static __device__ __forceinline__ void st128(ptr p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
  }
};
template <>
struct Mem<true> {
  typedef unsigned char* ptr;
  static __device__ __forceinline__ ptr add(ptr p, int32_t bytes) { return p + bytes; }
  static __device__ __forceinline__ uint32_t ld16(ptr p) { return *reinterpret_cast<const unsigned short*>(p); }
  static __device__ __forceinline__ uint32_t ld16w(ptr p) { return *reinterpret_cast<const unsigned short*>(p); }
  static __device__ __forceinline__ uint32_t ld32(ptr p) { return *reinterpret_cast<const uint32_t*>(p); }
  static __device__ __forceinline__ void ld128(ptr p, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    a = v.x; b = v.y; c = v.z; d = v.w;
  }
  static __device__ __forceinline__ uint32_t off(ptr p, ptr base) { return (uint32_t)(p - base); }
  static __device__ __forceinline__ uint32_t fadd(uint32_t a, uint32_t b, uint32_t) { return a + b; }
  static __device__ __forceinline__ uint32_t hi16(uint32_t w, uint32_t) { return w >> 16; }
  static __device__ __forceinline__ void step4(uint32_t& Q01, uint32_t& Q23, uint32_t& acc2, uint32_t w,
                                               uint32_t bit_lo, uint32_t bit_hi, uint32_t key, ptr base,
                                               const PipeConst&) {
    const bool ph = (w & bit_hi) != 0u, pl = (w & bit_lo) != 0u;
    const uint32_t qs = ph ? Q23 : Q01;
    const uint32_t idx = pl ? (qs >> 16) : (qs & 0xffffu);
    *reinterpret_cast<unsigned short*>(base + 2 * (size_t)idx) = (unsigned short)key;
    const uint32_t inc = pl ? 0x10000u : 1u;
    if (ph) Q23 += inc; else Q01 += inc;
    acc2 += qs >> 16;
  }
  template <int SH>
  static __device__ __forceinline__ void step16(NibbleCounts& s, uint32_t w, uint32_t a2, uint32_t a3) {
    const bool p3 = (w >> SH) & 8u, p1 = (w >> SH) & 2u, p0 = (w >> SH) & 1u;
    s.acc = __dp4a(s.C, p3 ? 0x02010000u : 0x01010100u, s.acc);
    const uint32_t W2 = 1u << (a2 & 31u), W3 = 1u << (a3 & 31u);
    s.C += W2;
    s.acc = __dp4a(s.D2, W2, s.acc);
    if (p1) s.D2 += W2;
    s.acc = __dp4a(p3 ? s.D3b : s.D3a, W3, s.acc);
    if (p0) {
      if (p3) s.D3b += W3; else s.D3a += W3;
    }
  }
  static __device__ __forceinline__ void red_add32(ptr p, uint32_t v) { atomicAdd(reinterpret_cast<uint32_t*>(p), v); }
  static __device__ __forceinline__ uint32_t atom_or32(ptr p, uint32_t v) { return atomicOr(reinterpret_cast<uint32_t*>(p), v); }
  // generic addressing reaches shared memory too
  static __device__ __forceinline__ ptr from_shared(const void* q) { return (ptr) const_cast<void*>(q); }
  static __device__ __forceinline__ void st16(ptr p, uint32_t v) {
    *reinterpret_cast<unsigned short*>(p) = (unsigned short)v;
  }
  static __device__ __forceinline__ void st32(ptr p, uint32_t v) { *reinterpret_cast<uint32_t*>(p) = v; }
  static __device__ __forceinline__ void st128(ptr p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    *reinterpret_cast<uint4*>(p) = make_uint4(a, b, c, d);
  }
};

// Pass A: the bucket-free counting pass on 16-bit keys (see the file header), lane-sequential,
// TWO bits per level.  Thread t of the CTA owns the contiguous range [t*R, (t+1)*R) of the
// sequence, R = 8*kk keys, and walks it with 128-bit loads (kk must be ODD: the 16-byte accesses
// of a quarter warp then fall into distinct bank groups).  A level on bits (s+1, s) is the fusion
// of the two one-bit levels s+1 and s: a stable partition of the whole sequence into the digit
// classes 0,1,2,3 (digit = 2*hi + lo), and the count
//     sum over keys with hi = 0 of #(hi = 1 keys before it)                        [bit s+1]
//   + sum over keys with lo = 0 of #(lo = 1 keys before it after the hi partition)  [bit s]
// where the second term is, for a key of class 0, the class-1 keys before it, and for a key of
// class 2 all N1 class-1 keys plus the class-3 keys before it.  Per level:
//   sweep 1  counts the range's keys per class, two keys per 32-bit word at once
//            ((w >> s) & 0x00010001 summed in two 16-bit fields), and -- same fields, one more
//            IMAD per word -- the sum J1 of the local indices of the hi = 1 keys: the whole hi-bit
//            term of the thread follows from it in closed form (a hi = 0 key at local index j has
//            j - (hi = 0 keys before it) hi = 1 keys before it inside the range);
//   two packed warp scans + warp-total reductions give the class counts before the range;
//   sweep 2  walks the range with four running slot indices (packed 2 x 16 bit in Q01, Q23),
//            stores every key to its slot of the other buffer and sums the running slot of the
//            key's lo = 1 sibling class over all keys (step4); the lo = 1 keys' own share of that
//            sum -- their destination slots, two arithmetic series -- is taken out in closed form.
// No ballots, no per-key population counts: about 16 instructions per key and level of two bits.
// With an odd number of bits the first level treats the missing top bit as zero.  The two-bit levels
// stop at bit 4; the low four bits take one count-only sweep (NibbleCounts, nibble_level).
//   acc64 += the count over all levels (this thread's share)
struct LevelCounts {
  uint32_t n1, n2, n3, J1;
};
// class counts and the hi-index sum of one thread's range from the packed sums of sweep 1:
// cl/ch/cb = per-half sums of the lo / hi / lo&hi bits, wm = per-half sums of (word index) * hi bit
__device__ __forceinline__ LevelCounts fold_counts(uint32_t cl, uint32_t ch, uint32_t cb, uint32_t wm) {
  LevelCounts c;
  c.n3 = (cb & 0xffffu) + (cb >> 16);
  c.n2 = (ch & 0xffffu) + (ch >> 16) - c.n3;
  c.n1 = (cl & 0xffffu) + (cl >> 16) - c.n3;
  // key 2m sits in the low half of word m, key 2m+1 in the high half
  c.J1 = 2u * ((wm & 0xffffu) + (wm >> 16)) + (ch >> 16);
  return c;
}
// the thread's share of a level's count (all arithmetic modulo 2^32; the true value is small):
//   hi term   n_hi0 * (hi keys before the range) + sum_{hi=0 keys} j - C(n_hi0, 2)
//   lo term   acc2 (all keys) - slots of the class-1 keys - slots of the class-3 keys
//             - n0 * N0 - n2 * (N0 + N2)     (class bases; N1 class-1 keys precede every class-2 key)
__device__ __forceinline__ uint32_t level_share(const LevelCounts& c, uint32_t R, uint32_t acc2, uint32_t e23,
                                                uint32_t start1, uint32_t start3, uint32_t N0, uint32_t N2) {
  const uint32_t nh0 = R - c.n2 - c.n3, n0 = nh0 - c.n1;
  const uint32_t hi_term = nh0 * e23 + ((R * (R - 1u)) >> 1) - c.J1 - ((nh0 * (nh0 - 1u)) >> 1);
  const uint32_t lo_term = acc2 - c.n1 * start1 - ((c.n1 * (c.n1 - 1u)) >> 1) - c.n3 * start3 -
                           ((c.n3 * (c.n3 - 1u)) >> 1) - n0 * N0 - c.n2 * (N0 + N2);
  return hi_term + lo_term;
}

// the low-nibble sweep over one 32-bit word (two keys, the low one first)
template <bool G>
__device__ __forceinline__ void nibble_word(NibbleCounts& s, uint32_t w) {
  const uint32_t a2 = (w << 1) & 0x00180018u, a3 = (w << 2) & 0x00180018u;
  Mem<G>::template step16<0>(s, w, a2, a3);
  Mem<G>::template step16<16>(s, w, a2 >> 16, a3 >> 16);
}

// this thread's share of a nibble-tree count (see nibble_level) from its sweep's counts s, the ones r at the
// root and the ones E[] before its range, packed as nibble_level's q[]
__device__ __forceinline__ uint32_t nibble_share(const NibbleCounts& s, const uint32_t R, const uint32_t r,
                                                 const uint32_t E[8]) {
  // zeros per node: b1 = 0 per (b3 b2), then b0 = 0 per (b3 b2 b1) (bytewise, no borrows)
  const uint32_t N2 = s.C - s.D2;
  const uint32_t N3a = __byte_perm(N2, s.D2, 0x5140) - s.D3a, N3b = __byte_perm(N2, s.D2, 0x7362) - s.D3b;
  uint32_t x = (R - r) * E[1];
  x = __dp2a_lo(E[0], __byte_perm(s.C, 0u, 0x4420), x);  // c0 * E(c1) + c2 * E(c3)
  x = __dp2a_hi(E[3], N2, __dp2a_lo(E[2], N2, x));
  x = __dp2a_hi(E[5], N3a, __dp2a_lo(E[4], N3a, x));
  x = __dp2a_hi(E[7], N3b, __dp2a_lo(E[6], N3b, x));
  // sum of C(n1, 2) = (sum n1^2 - sum n1) / 2 over the 15 nodes
  const uint32_t sq = __dp4a(s.D2, s.D2, __dp4a(s.D3a, s.D3a, __dp4a(s.D3b, s.D3b, __dp4a(s.C & 0xff00ff00u, s.C, r * r))));
  const uint32_t li = __dp4a(s.D2, 0x01010101u, __dp4a(s.D3a, 0x01010101u, __dp4a(s.D3b, 0x01010101u, __dp4a(s.C, 0x01000100u, r))));
  return s.acc + x - ((sq - li) >> 1);
}

// The low-nibble level after its sweep: this thread's share is
//   acc - sum over nodes of C(n1, 2)                    (within the range)
//   + sum over nodes of n0 * (ones at the node in earlier ranges)
// The 15 ones counts go through one warp scan as 16-bit pairs; lane 31 leaves the warp's totals in the
// first 32 bytes of the warp's part of `a` (its keys are read and are not needed afterwards), where the
// later warps add them after the barrier.  Two block-wide barriers.
template <bool G>
__device__ __forceinline__ void nibble_level(const NibbleCounts& s, const uint32_t R, const bool idle, const int lane,
                                             const int warp, typename Mem<G>::ptr a, unsigned long long& acc64) {
  typedef Mem<G> M;
  const uint32_t warp_bytes = R << 6;
  const uint32_t r = ((s.C >> 16) & 0xffu) + (s.C >> 24);  // ones at the root
  const uint32_t q[8] = {__byte_perm(s.C, 0u, 0x4341),   r,
                         __byte_perm(s.D2, 0u, 0x4140),  __byte_perm(s.D2, 0u, 0x4342),
                         __byte_perm(s.D3a, 0u, 0x4140), __byte_perm(s.D3a, 0u, 0x4342),
                         __byte_perm(s.D3b, 0u, 0x4140), __byte_perm(s.D3b, 0u, 0x4342)};
  uint32_t incl[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) incl[k] = q[k];
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint32_t t = __shfl_up_sync(FULL, incl[k], d);
      if (lane >= d) incl[k] += t;
    }
  }
  __syncwarp();
  if (lane == 31) {
    const typename M::ptr mine = M::add(a, (int32_t)((uint32_t)warp * warp_bytes));
    M::st128(mine, incl[0], incl[1], incl[2], incl[3]);
    M::st128(M::add(mine, 16), incl[4], incl[5], incl[6], incl[7]);
  }
  __syncthreads();
  uint32_t v[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  if (lane < warp) {
    const typename M::ptr o = M::add(a, (int32_t)((uint32_t)lane * warp_bytes));
    M::ld128(o, v[0], v[1], v[2], v[3]);
    M::ld128(M::add(o, 16), v[4], v[5], v[6], v[7]);
  }
  uint32_t E[8];  // ones before the range (exclusive prefix over the CTA; below 65 536)
#pragma unroll
  for (int k = 0; k < 8; ++k) E[k] = __reduce_add_sync(FULL, v[k]) + incl[k] - q[k];
  if (!idle) acc64 += (unsigned long long)nibble_share(s, R, r, E);
  __syncthreads();  // the warp totals are read before anybody reuses the buffer
}

// The 16 digit counts (b3 b2 b1 b0) of N keys whose node ones counts are e[] (packed as nibble_level's q[]):
// each node splits its keys into the ones and the rest, from the root down.
__device__ __forceinline__ void nibble_digits(uint32_t N, const uint32_t e[8], uint32_t dig[16]) {
  const uint32_t c1 = e[0] & 0xffffu, c3 = e[0] >> 16, r = e[1];
  const uint32_t cls[4] = {N - r - c1, c1, r - c3, c3};
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint32_t d2 = (e[2 + (c >> 1)] >> (16 * (c & 1))) & 0xffffu;
    const uint32_t pre[2] = {cls[c] - d2, d2};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int p = 2 * c + h;
      const uint32_t d3 = (e[4 + (p >> 1)] >> (16 * (p & 1))) & 0xffffu;
      dig[2 * p] = pre[h] - d3;
      dig[2 * p + 1] = d3;
    }
  }
}

// A radix-16 level of pass A on bits s+3 .. s (s >= 4, shared memory only): the count of the nibble level at
// bit s -- the same tree over the same order, so it counts what the two two-bit levels it replaces count on
// those bits, up to terms of column y alone -- and a stable partition of the sequence by the 4-bit digit.
//   sweep 1  the nibble tree over the range (step16_at);
//   one warp scan of the 15 node ones counts, the warps' totals through `tot` (32 bytes per warp), gives the
//            count's cross-range share and, split node by node (nibble_digits), every digit's keys before the
//            range and in the whole buffer; the start slot of each digit goes to this thread's column of the
//            u16 counter table cnt[16][T] at `ctr` (odd threads' counters 64 bytes further on, so that a warp's
//            even lanes hit banks 0-15 and its odd lanes banks 16-31 whatever their digits: conflict-free; the
//            last row's odd counters run 64 bytes past the table);
//   sweep 2  stores every key to slot cnt[d][tid]++ of the other buffer (scatter16).
// Threads outside the sequence (TAIL) enter the scan with the counts of R padding keys, digit 15.  Two
// block-wide barriers.
template <bool TAIL>
__device__ __forceinline__ void radix_level(const uint32_t a, const uint32_t b, const uint32_t ctr, const uint32_t s,
                                            const int kk, const int nwarps, const bool idle, const bool tail,
                                            const int lane, const int warp, const PipeConst& pc,
                                            unsigned long long& acc64) {
  typedef Mem<false> M;
  const uint32_t T = (uint32_t)nwarps << 5, tid = ((uint32_t)warp << 5) + (uint32_t)lane;
  const uint32_t R = (uint32_t)kk << 3, my_pos = tid * R, ra = a + tid * (R << 1);
  const uint32_t tot = ctr + (T << 5) + 64u;
  NibbleCounts nc = {0u, 0u, 0u, 0u, 0u};
  if (TAIL && tail) nc.C = nc.D2 = nc.D3b = R << 24;
  {
    uint32_t m8 = 8u << s, m2 = 2u << s, m1 = 1u << s;
    uint32_t h8 = m8 << 16, h2 = m2 << 16, h1 = m1 << 16;
    const uint32_t s2 = s - 1u, s3 = s - 2u;
#pragma unroll 1
    for (int c = 0; c < (idle ? 0 : kk); ++c) {
      uint32_t w[4];
      M::ld128(ra + (c << 4), w[0], w[1], w[2], w[3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t a2 = (w[j] >> s2) & 0x00180018u, a3 = (w[j] >> s3) & 0x00180018u;
        M::step16_at(nc, w[j], a2, a3, m8, m2, m1);
        M::step16_at(nc, w[j], a2 >> 16, a3 >> 16, h8, h2, h1);
      }
    }
  }
  const uint32_t r = ((nc.C >> 16) & 0xffu) + (nc.C >> 24);
  const uint32_t q[8] = {__byte_perm(nc.C, 0u, 0x4341),   r,
                         __byte_perm(nc.D2, 0u, 0x4140),  __byte_perm(nc.D2, 0u, 0x4342),
                         __byte_perm(nc.D3a, 0u, 0x4140), __byte_perm(nc.D3a, 0u, 0x4342),
                         __byte_perm(nc.D3b, 0u, 0x4140), __byte_perm(nc.D3b, 0u, 0x4342)};
  uint32_t incl[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) incl[k] = q[k];
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint32_t t = __shfl_up_sync(FULL, incl[k], d);
      if (lane >= d) incl[k] += t;
    }
  }
  if (lane == 31) {
    M::st128(tot + ((uint32_t)warp << 5), incl[0], incl[1], incl[2], incl[3]);
    M::st128(tot + ((uint32_t)warp << 5) + 16u, incl[4], incl[5], incl[6], incl[7]);
  }
  __syncthreads();
  uint32_t v[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  if (lane < nwarps) {
    M::ld128(tot + ((uint32_t)lane << 5), v[0], v[1], v[2], v[3]);
    M::ld128(tot + ((uint32_t)lane << 5) + 16u, v[4], v[5], v[6], v[7]);
  }
  uint32_t E[8], N[8];  // ones before the range / in the whole buffer, per node
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    E[k] = __reduce_add_sync(FULL, (lane < warp) ? v[k] : 0u) + incl[k] - q[k];
    N[k] = __reduce_add_sync(FULL, v[k]);
  }
  if (!idle) {
    acc64 += (unsigned long long)nibble_share(nc, R, r, E);
    uint32_t before[16], total[16];
    nibble_digits(my_pos, E, before);
    nibble_digits(T * R, N, total);
    const uint32_t me = ctr + (tid << 1) + ((tid & 1u) << 6), row = T << 1;
    uint32_t run = 0u;
#pragma unroll
    for (int d = 0; d < 16; ++d) {
      M::st16(me + (uint32_t)d * row, run + before[d]);
      run += total[d];
    }
#pragma unroll 1
    for (int c = 0; c < kk; ++c) {
      uint32_t w[4];
      M::ld128(ra + (c << 4), w[0], w[1], w[2], w[3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        M::scatter16(w[j], s, me, row, b, pc);
        M::scatter16(M::hi16(w[j], pc.c64k), s, me, row, b, pc);
      }
    }
  }
  __syncthreads();  // the next level reads the other buffer; also protects `tot`
}

// block-wide barriers count_pass executes for L bits (threads that skip it must keep them)
__host__ __device__ constexpr int count_pass_barriers(int L) { return 2 * (L > 4 ? ((L - 1) >> 1) : 1); }

// `lead`: the sequence is known to START with that many zero keys (x's first tie group is written in
// ascending y order, so its rows of y's lowest rank -- on left-censored data the rows missing in BOTH
// columns, a fifth of all rows -- come first).  Zero keys are class 0 at every level and the stable
// partition keeps a leading block of them exactly where it is; no one-key ever precedes them, so they
// add nothing to any count.  Threads whose whole range lies inside that block skip the sweeps of
// every level (they only take part in the scans, with zero counts, and in the barriers).
// TAIL (besides `lead`): only the first `len` keys are the sequence, the rest is all-ones padding
// (2^L - 1); len = cap for a full sequence.  Padding is the largest key, so it is in the last non-empty class at every level and
// the stable partition keeps it where it is; it never adds to a count.  Threads whose whole range
// lies at or beyond `len` skip the sweeps of every level: they enter the scans with the class
// counts of R padding keys (closed form) and add nothing; nobody reads their ranges.  The thread
// that straddles `len` writes the padding of its own range before its first sweep.
template <bool G, bool TAIL = false>
__device__ __forceinline__ void count_pass(typename Mem<G>::ptr a, typename Mem<G>::ptr b, const int kk,
                                           const int nwarps, const int L, uint32_t* descA, uint32_t* descB,
                                           const int lane, const int warp, const PipeConst pc,
                                           unsigned long long& acc64, const uint32_t lead = 0u,
                                           const uint32_t len = 0u, const uint32_t ctr = 0u) {
  typedef Mem<G> M;
  // ctr != 0 (shared memory only): the bits from 4 up to the highest multiple of 4 below L take radix-16
  // levels (radix_level, counter table at ctr), the two-bit levels only the bits above them
  const int nr = (!G && ctr != 0u && L > 4) ? (L - 4) >> 2 : 0;
  const uint32_t tid = ((uint32_t)warp << 5) + (uint32_t)lane;
  const uint32_t R = (uint32_t)kk << 3;                // keys per thread range
  const uint32_t my_off = tid * (R << 1);              // bytes
  const uint32_t my_pos = tid * R;
  const uint32_t cap = ((uint32_t)nwarps << 5) * R;    // keys per buffer
  const uint32_t padA = (1u << L) - 1u;
  const bool tail = TAIL && my_pos >= len;
  const bool idle = tail || my_pos + R <= lead;
  if constexpr (TAIL) {
    if (!idle)
      for (uint32_t q = len; q < my_pos + R; ++q) M::st16(M::add(a, (int32_t)(q << 1)), padA);
  }
  if (idle && !tail && L > 4) {  // the block must read as zeros in the other buffer too (levels alternate)
    const typename M::ptr rb = M::add(b, (int32_t)my_off);
    for (int c = 0; c < kk; ++c) M::st128(M::add(rb, c << 4), 0u, 0u, 0u, 0u);
  }
  for (int s = (L - 1) & ~1; s >= 4 + 4 * nr; s -= 2) {
    const typename M::ptr ra = M::add(a, (int32_t)my_off);
    uint32_t cl = 0, cb = 0, wm = 0, m4 = 0;
    uint32_t chj[4] = {0u, 0u, 0u, 0u};
#pragma unroll 1
    for (int c = 0; c < (idle ? 0 : kk); ++c) {
      uint32_t w[4];
      M::ld128(M::add(ra, c << 4), w[0], w[1], w[2], w[3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t lo = (w[j] >> s) & 0x00010001u, hi = (w[j] >> (s + 1)) & 0x00010001u;
        cl = M::fadd(cl, lo, pc.one);
        chj[j] = M::fadd(chj[j], hi, pc.one);
        cb = M::fadd(cb, lo & hi, pc.one);
        wm += hi * m4;  // word index 4c + j: the 4c part here, the j part from chj[] below
      }
      m4 += 4u;
    }
    const uint32_t ch = chj[0] + chj[1] + chj[2] + chj[3];
    wm += chj[1] + 2u * chj[2] + 3u * chj[3];
    const LevelCounts lc = fold_counts(cl, ch, cb, wm);
    const uint32_t n1 = lc.n1, n2 = lc.n2, n3 = lc.n3;
    uint32_t A = n1 | (n2 << 16), B = n3;
    if constexpr (TAIL) {
      if (tail) {  // R padding keys: class 3, or class 1 on the first level of an odd L (its top bit is 0)
        const uint32_t pcl = (padA >> s) & 3u;
        A = pcl == 1u ? R : 0u;
        B = pcl == 3u ? R : 0u;
      }
    }
    uint32_t inclA = A, inclB = B;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t tA = __shfl_up_sync(FULL, inclA, d), tB = __shfl_up_sync(FULL, inclB, d);
      if (lane >= d) {
        inclA += tA;
        inclB += tB;
      }
    }
    if (lane == 31) {
      descA[warp] = inclA;
      descB[warp] = inclB;
    }
    __syncthreads();
    const uint32_t vA = (lane < nwarps) ? descA[lane] : 0u, vB = (lane < nwarps) ? descB[lane] : 0u;
    const uint32_t totA = __reduce_add_sync(FULL, vA), totB = __reduce_add_sync(FULL, vB);
    const uint32_t exA = __reduce_add_sync(FULL, (lane < warp) ? vA : 0u) + inclA - A;
    const uint32_t exB = __reduce_add_sync(FULL, (lane < warp) ? vB : 0u) + inclB - B;
    const uint32_t e1 = exA & 0xffffu, e2 = exA >> 16, e3 = exB;           // class counts before my range
    const uint32_t N1 = totA & 0xffffu, N2 = totA >> 16, N3 = totB;
    const uint32_t N0 = cap - N1 - N2 - N3;
    const uint32_t start1 = N0 + e1, start3 = N0 + N1 + N2 + e3;
    uint32_t Q01 = (start1 << 16) | (my_pos - e1 - e2 - e3);
    uint32_t Q23 = (start3 << 16) | (N0 + N1 + e2);
    uint32_t acc2 = 0;
    uint32_t bLl = 1u << s, bHl = 2u << s, bLh = 1u << (s + 16), bHh = 2u << (s + 16);
    asm volatile("" : "+r"(bLl), "+r"(bHl), "+r"(bLh), "+r"(bHh));  // keep the bit tests single LOP3s
    if (idle) {
      // nothing to move, nothing to count
    } else {
#pragma unroll 1
      for (int c = 0; c < kk; ++c) {
        uint32_t w[4];
        M::ld128(M::add(ra, c << 4), w[0], w[1], w[2], w[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          M::step4(Q01, Q23, acc2, w[j], bLl, bHl, w[j], b, pc);
          M::step4(Q01, Q23, acc2, w[j], bLh, bHh, M::hi16(w[j], pc.c64k), b, pc);
        }
      }
    }
    (void)N3;
    if (!idle) acc64 += (unsigned long long)level_share(lc, R, acc2, e2 + e3, start1, start3, N0, N2);
    __syncthreads();  // also protects descA/descB for the next level
    const typename M::ptr t = a;
    a = b;
    b = t;
  }
  if constexpr (!G) {
    for (int s = 4 * nr; s >= 4; s -= 4) {
      radix_level<TAIL>(a, b, ctr, (uint32_t)s, kk, nwarps, idle, tail, lane, warp, pc, acc64);
      const uint32_t t = a;
      a = b;
      b = t;
    }
  }
  NibbleCounts nc = {0u, 0u, 0u, 0u, 0u};
  const typename M::ptr ra = M::add(a, (int32_t)my_off);
#pragma unroll 1
  for (int c = 0; c < (idle ? 0 : kk); ++c) {
    uint32_t w[4];
    M::ld128(M::add(ra, c << 4), w[0], w[1], w[2], w[3]);
#pragma unroll
    for (int j = 0; j < 4; ++j) nibble_word<G>(nc, w[j]);
  }
  nibble_level<G>(nc, R, idle, lane, warp, a, acc64);
}

}  // namespace
}  // namespace icikt
