// sva_vec.cuh — per-lane vector moves of NR packed-u16x2 registers (global -> shared async copies, shared loads, stores, REDs),
// shared by the SGM marches (k_sgm.cu) and the WTA march (k_wta.cu).
#pragma once
#include "sva_common.cuh"

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int NR> struct Vec;
template <> struct Vec<1> {
    static __device__ __forceinline__ void load(const uint16_t* p, uint32_t (&r)[1]) { r[0] = ldg_stream_u32(p); }
    static __device__ __forceinline__ void load_rw(const uint16_t* p, uint32_t (&r)[1]) {
        asm volatile("ld.global.L1::no_allocate.u32 %0, [%1];" : "=r"(r[0]) : "l"(p));
    }
    static __device__ __forceinline__ void cp_async(uint32_t dst, const uint16_t* p) { asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(p) : "memory"); }
    static __device__ __forceinline__ void lds(uint32_t src, uint32_t (&r)[1]) { asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r[0]) : "r"(src)); }
    static __device__ __forceinline__ void store(uint16_t* p, const uint32_t (&r)[1]) { *reinterpret_cast<uint32_t*>(p) = r[0]; }
    static __device__ __forceinline__ void red(uint16_t* p, const uint32_t (&r)[1]) {
        asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(r[0]) : "memory");
    }
};
template <> struct Vec<2> {
    static __device__ __forceinline__ void load(const uint16_t* p, uint32_t (&r)[2]) { uint2 v = ldg_stream_u64(p); r[0] = v.x; r[1] = v.y; }
    static __device__ __forceinline__ void load_rw(const uint16_t* p, uint32_t (&r)[2]) {
        asm volatile("ld.global.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "l"(p));
    }
    static __device__ __forceinline__ void cp_async(uint32_t dst, const uint16_t* p) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(p) : "memory"); }
    static __device__ __forceinline__ void lds(uint32_t src, uint32_t (&r)[2]) { asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(src)); }
    static __device__ __forceinline__ void store(uint16_t* p, const uint32_t (&r)[2]) { *reinterpret_cast<uint2*>(p) = make_uint2(r[0], r[1]); }
    static __device__ __forceinline__ void red(uint16_t* p, const uint32_t (&r)[2]) {
        unsigned long long v = ((unsigned long long)r[1] << 32) | r[0];
        asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
    }
};
template <> struct Vec<4> {
    static __device__ __forceinline__ void load(const uint16_t* p, uint32_t (&r)[4]) { uint4 v = ldg_stream_u128(p); r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w; }
    static __device__ __forceinline__ void load_rw(const uint16_t* p, uint32_t (&r)[4]) {
        asm volatile("ld.global.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(p));
    }
    static __device__ __forceinline__ void cp_async(uint32_t dst, const uint16_t* p) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(p) : "memory"); }
    static __device__ __forceinline__ void lds(uint32_t src, uint32_t (&r)[4]) { asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(src)); }
    static __device__ __forceinline__ void store(uint16_t* p, const uint32_t (&r)[4]) { *reinterpret_cast<uint4*>(p) = make_uint4(r[0], r[1], r[2], r[3]); }
    static __device__ __forceinline__ void red(uint16_t* p, const uint32_t (&r)[4]) {
        unsigned long long v0 = ((unsigned long long)r[1] << 32) | r[0], v1 = ((unsigned long long)r[3] << 32) | r[2];
        asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v0) : "memory");
        asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p + 4), "l"(v1) : "memory");
    }
};

template <> struct Vec<6> {  // 24 bytes per lane: three 8-byte pieces (a lane's slot is only 8-byte aligned)
    static __device__ __forceinline__ void cp_async(uint32_t dst, const uint16_t* p) {
#pragma unroll
        for (int i = 0; i < 3; i++) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 8 * i), "l"(p + 4 * i) : "memory");
    }
    static __device__ __forceinline__ void lds(uint32_t src, uint32_t (&r)[6]) {
#pragma unroll
        for (int i = 0; i < 3; i++) asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r[2 * i]), "=r"(r[2 * i + 1]) : "r"(src + 8 * i));
    }
    static __device__ __forceinline__ void store(uint16_t* p, const uint32_t (&r)[6]) {
#pragma unroll
        for (int i = 0; i < 3; i++) reinterpret_cast<uint2*>(p)[i] = make_uint2(r[2 * i], r[2 * i + 1]);
    }
    static __device__ __forceinline__ void red(uint16_t* p, const uint32_t (&r)[6]) {
#pragma unroll
        for (int i = 0; i < 3; i++) {
            unsigned long long v = ((unsigned long long)r[2 * i + 1] << 32) | r[2 * i];
            asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p + 4 * i), "l"(v) : "memory");
        }
    }
};
template <> struct Vec<8> {
    static __device__ __forceinline__ void cp_async(uint32_t dst, const uint16_t* p) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(p) : "memory");
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16), "l"(p + 8) : "memory");
    }
    static __device__ __forceinline__ void lds(uint32_t src, uint32_t (&r)[8]) {
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(src));
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(src + 16));
    }
    static __device__ __forceinline__ void store(uint16_t* p, const uint32_t (&r)[8]) {
        reinterpret_cast<uint4*>(p)[0] = make_uint4(r[0], r[1], r[2], r[3]);
        reinterpret_cast<uint4*>(p)[1] = make_uint4(r[4], r[5], r[6], r[7]);
    }
    static __device__ __forceinline__ void red(uint16_t* p, const uint32_t (&r)[8]) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            unsigned long long v = ((unsigned long long)r[2 * i + 1] << 32) | r[2 * i];
            asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p + 4 * i), "l"(v) : "memory");
        }
    }
};

// "Block" layout for 8 disparities per lane on BL lanes (D = 8 BL: 256 on a full warp, 192 on 24 lanes): lane l owns the 8-byte pairs
// l and BL + l of the 2 BL pairs of a cell, i.e. disparities 4l..4l+3 and 4BL+4l..4BL+4l+3.  Every copy / load / RED instruction then
// covers 8 BL contiguous bytes (whole sectors); in the plain layout (16 contiguous bytes per lane) each of the two 64-bit REDs of a lane
// touches half of every sector of the cell, which is what bounded the D > 128 marches (B200: 0.71 -> 0.46 ms per row-sweeping launch at
// 1280x960x256).  p points at the lane's first pair; the ring slot is 8 bytes per lane, the second block 8 BL bytes further.
template <int BL> struct VecBlk4 {
    static __device__ __forceinline__ void cp_async(uint32_t dst, const uint16_t* p) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(p) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 8 * BL), "l"(p + 4 * BL) : "memory");
    }
    static __device__ __forceinline__ void lds(uint32_t src, uint32_t (&r)[4]) {
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(src));
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r[2]), "=r"(r[3]) : "r"(src + 8 * BL));
    }
    static __device__ __forceinline__ void store(uint16_t* p, const uint32_t (&r)[4]) {
        *reinterpret_cast<uint2*>(p) = make_uint2(r[0], r[1]);
        *reinterpret_cast<uint2*>(p + 4 * BL) = make_uint2(r[2], r[3]);
    }
    static __device__ __forceinline__ void load(const uint16_t* p, uint32_t (&r)[4]) {
        const uint2 a = *reinterpret_cast<const uint2*>(p), b = *reinterpret_cast<const uint2*>(p + 4 * BL);
        r[0] = a.x; r[1] = a.y; r[2] = b.x; r[3] = b.y;
    }
    static __device__ __forceinline__ void red(uint16_t* p, const uint32_t (&r)[4]) {
        unsigned long long v0 = ((unsigned long long)r[1] << 32) | r[0], v1 = ((unsigned long long)r[3] << 32) | r[2];
        asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v0) : "memory");
        asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p + 4 * BL), "l"(v1) : "memory");
    }
};

template <int NR, int BL> struct VecSel { using type = VecBlk4<BL>; };
template <int NR> struct VecSel<NR, 0> { using type = Vec<NR>; };
