// BCF 2.2 typed values, shared by the decoder (bcf.cu) and the VCF formatter (bcfout.cu).
#pragma once
#include "common.cuh"

namespace {

constexpr int BT_NULL = 0, BT_INT8 = 1, BT_INT16 = 2, BT_INT32 = 3, BT_FLOAT = 5, BT_CHAR = 7;
constexpr uint32_t FLOAT_MISSING = 0x7F800001u, FLOAT_EOV = 0x7F800002u;

__host__ __device__ __forceinline__ uint32_t ld_u32(const uint8_t* p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// bytes per value of a type; -1 for a type BCF 2.2 does not define
__host__ __device__ __forceinline__ int type_width(int t) {
    switch (t) {
        case BT_NULL: return 0;
        case BT_INT8: case BT_CHAR: return 1;
        case BT_INT16: return 2;
        case BT_INT32: case BT_FLOAT: return 4;
        default: return -1;
    }
}

__host__ __device__ __forceinline__ bool is_int_type(int t) { return t == BT_INT8 || t == BT_INT16 || t == BT_INT32; }

// one integer of type t at p.  0: a value (*v), 1: missing, 2: end of vector, 3: a reserved value
__host__ __device__ __forceinline__ int ld_int(const uint8_t* p, int t, int32_t* v) {
    int32_t x, lo;
    if (t == BT_INT8) {
        x = (int8_t)p[0];
        lo = -128;
    } else if (t == BT_INT16) {
        x = (int16_t)(uint16_t)(p[0] | (p[1] << 8));
        lo = -32768;
    } else {
        x = (int32_t)ld_u32(p);
        lo = (int32_t)0x80000000u;
    }
    *v = x;
    if (x > lo + 7) return 0;
    if (x == lo) return 1;
    if (x == lo + 1) return 2;
    return 3;
}

// the type byte of a typed value at p (and the typed integer of an overflowing count); p advanced past them.
// false: it runs past e, or a type (or a count's type) is not one of BCF 2.2's
__host__ __device__ __forceinline__ bool typed_hdr(const uint8_t* b, int64_t& p, int64_t e, int* type, int64_t* count,
                                                   uint8_t* why) {
    if (p >= e) { *why |= UNFZ_BCF_BAD_OVERRUN; return false; }
    const uint8_t t = b[p++];
    *type = t & 15;
    int64_t n = t >> 4;
    if (type_width(*type) < 0) { *why |= UNFZ_BCF_BAD_TYPE; return false; }
    if (n == 15) {                                       // the count follows as a typed integer
        if (p >= e) { *why |= UNFZ_BCF_BAD_OVERRUN; return false; }
        const uint8_t t2 = b[p++];
        const int ct = t2 & 15;
        if ((t2 >> 4) != 1 || !is_int_type(ct)) { *why |= UNFZ_BCF_BAD_TYPE; return false; }
        const int w = type_width(ct);
        if (p + w > e) { *why |= UNFZ_BCF_BAD_OVERRUN; return false; }
        int32_t v;
        if (ld_int(b + p, ct, &v) != 0 || v < 0) { *why |= UNFZ_BCF_BAD_TYPE; return false; }
        p += w;
        n = v;
    }
    *count = n;
    return true;
}

}  // namespace
