/*
 * group.c -- ristretto255 group for the CPU oracle (test infrastructure, see eg_oracle.h).
 * Extended twisted-Edwards arithmetic (RFC 8032 5.1.4, a = -1) and the ristretto255 encoding
 * (RFC 9496 4.3).  Replaces curve25519-dalek's RistrettoPoint / CompressedRistretto /
 * RISTRETTO_BASEPOINT_TABLE / (Vartime)MultiscalarMul as used by src/group/ristretto.rs:72-146.
 * Scalar multiplication uses the same algorithm shapes as the reference backend (width-5 wNAF
 * Straus for variable bases, width-8 wNAF table for the basepoint) so that it is a fair CPU baseline;
 * results do not depend on the algorithm because encodings are canonical.
 */
#include "eg_oracle.h"
#include <string.h>

int eo_fe_iszero(const eo_fe *f);
int eo_fe_isnegative(const eo_fe *f);
int eo_fe_eq(const eo_fe *a, const eo_fe *b);
const eo_fe *eo_fe_sqrt_m1(void);

static const eo_fe FE_ONE = {{1, 0, 0, 0, 0}};
static const eo_fe FE_ZERO = {{0, 0, 0, 0, 0}};

/* constants derived at first use from their defining equations (no transcribed magic numbers) */
static struct {
    int ready;
    eo_fe d, d2, invsqrt_a_minus_d;
    eo_pt G;
} C;

static void fe_from_u64(eo_fe *h, uint64_t x) {
    h->v[0] = x & ((1ULL << 51) - 1); h->v[1] = x >> 51; h->v[2] = h->v[3] = h->v[4] = 0;
}

static void constants_init(void) {
    if (C.ready) return;
    eo_fe a, b, t;
    /* d = -121665/121666 */
    fe_from_u64(&a, 121665); fe_from_u64(&b, 121666);
    eo_fe_invert(&t, &b);
    eo_fe_mul(&t, &t, &a);
    eo_fe_neg(&C.d, &t);
    eo_fe_add(&C.d2, &C.d, &C.d);
    /* 1/sqrt(a - d) = 1/sqrt(-1 - d), non-negative root */
    eo_fe amd;
    eo_fe_neg(&amd, &FE_ONE);
    eo_fe_sub(&amd, &amd, &C.d);
    eo_fe_sqrt_ratio_i(&C.invsqrt_a_minus_d, &FE_ONE, &amd);
    /* base point: y = 4/5, x = the even root of (y^2-1)/(d y^2+1) (RFC 8032 5.1) */
    eo_fe y, y2, u, v, x;
    fe_from_u64(&a, 4); fe_from_u64(&b, 5);
    eo_fe_invert(&t, &b);
    eo_fe_mul(&y, &t, &a);
    eo_fe_sq(&y2, &y);
    eo_fe_sub(&u, &y2, &FE_ONE);
    eo_fe_mul(&v, &C.d, &y2);
    eo_fe_add(&v, &v, &FE_ONE);
    eo_fe_sqrt_ratio_i(&x, &u, &v);          /* non-negative (even) root */
    C.G.X = x; C.G.Y = y; C.G.Z = FE_ONE;
    eo_fe_mul(&C.G.T, &x, &y);
    C.ready = 1;
}

void eo_pt_identity(eo_pt *p) { p->X = FE_ZERO; p->Y = FE_ONE; p->Z = FE_ONE; p->T = FE_ZERO; }
void eo_pt_generator(eo_pt *p) { constants_init(); *p = C.G; }

/* add-2008-hwcd-3 (unified, complete for a=-1 with non-square d) */
void eo_pt_add(eo_pt *r, const eo_pt *p, const eo_pt *q) {
    constants_init();
    eo_fe a, b, c, d, e, f, g, h, t;
    eo_fe_sub(&a, &p->Y, &p->X); eo_fe_sub(&t, &q->Y, &q->X); eo_fe_mul(&a, &a, &t);
    eo_fe_add(&b, &p->Y, &p->X); eo_fe_add(&t, &q->Y, &q->X); eo_fe_mul(&b, &b, &t);
    eo_fe_mul(&c, &p->T, &q->T); eo_fe_mul(&c, &c, &C.d2);
    eo_fe_mul(&d, &p->Z, &q->Z); eo_fe_add(&d, &d, &d);
    eo_fe_sub(&e, &b, &a); eo_fe_sub(&f, &d, &c); eo_fe_add(&g, &d, &c); eo_fe_add(&h, &b, &a);
    eo_fe_mul(&r->X, &e, &f); eo_fe_mul(&r->Y, &g, &h); eo_fe_mul(&r->T, &e, &h); eo_fe_mul(&r->Z, &f, &g);
}

void eo_pt_neg(eo_pt *r, const eo_pt *p) {
    eo_fe_neg(&r->X, &p->X); r->Y = p->Y; r->Z = p->Z; eo_fe_neg(&r->T, &p->T);
}

void eo_pt_sub(eo_pt *r, const eo_pt *p, const eo_pt *q) {
    eo_pt n;
    eo_pt_neg(&n, q);
    eo_pt_add(r, p, &n);
}

/* dbl-2008-hwcd */
void eo_pt_double(eo_pt *r, const eo_pt *p) {
    eo_fe a, b, c, e, f, g, h, t;
    eo_fe_sq(&a, &p->X); eo_fe_sq(&b, &p->Y);
    eo_fe_sq(&c, &p->Z); eo_fe_add(&c, &c, &c);
    eo_fe_add(&t, &p->X, &p->Y); eo_fe_sq(&t, &t);
    eo_fe_sub(&e, &t, &a); eo_fe_sub(&e, &e, &b);     /* E = (X+Y)^2 - A - B */
    eo_fe_sub(&g, &b, &a);                             /* G = D + B = B - A  (D = -A) */
    eo_fe_sub(&f, &g, &c);                             /* F = G - C */
    eo_fe_add(&h, &a, &b); eo_fe_neg(&h, &h);          /* H = D - B = -(A + B) */
    eo_fe_mul(&r->X, &e, &f); eo_fe_mul(&r->Y, &g, &h); eo_fe_mul(&r->T, &e, &h); eo_fe_mul(&r->Z, &f, &g);
}

/* RFC 9496 4.3.1 */
int eo_pt_decode(eo_pt *p, const uint8_t sb[32]) {
    constants_init();
    eo_fe s, ss, u1, u2, u2s, v, t, inv, denx, deny, x, y;
    uint8_t chk[32];
    eo_fe_frombytes(&s, sb);
    eo_fe_tobytes(chk, &s);
    if (memcmp(chk, sb, 32) != 0) return 0;    /* non-canonical (>= p or bit 255 set) */
    if (sb[0] & 1) return 0;                   /* negative */
    eo_fe_sq(&ss, &s);
    eo_fe_sub(&u1, &FE_ONE, &ss);
    eo_fe_add(&u2, &FE_ONE, &ss);
    eo_fe_sq(&u2s, &u2);
    eo_fe_sq(&t, &u1); eo_fe_mul(&t, &t, &C.d); eo_fe_neg(&t, &t);
    eo_fe_sub(&v, &t, &u2s);                   /* v = -(d u1^2) - u2^2 */
    eo_fe_mul(&t, &v, &u2s);
    int was_square = eo_fe_sqrt_ratio_i(&inv, &FE_ONE, &t);
    eo_fe_mul(&denx, &inv, &u2);
    eo_fe_mul(&deny, &inv, &denx); eo_fe_mul(&deny, &deny, &v);
    eo_fe_add(&t, &s, &s); eo_fe_mul(&x, &t, &denx);
    if (eo_fe_isnegative(&x)) eo_fe_neg(&x, &x);
    eo_fe_mul(&y, &u1, &deny);
    eo_fe_mul(&t, &x, &y);
    if (!was_square || eo_fe_isnegative(&t) || eo_fe_iszero(&y)) return 0;
    p->X = x; p->Y = y; p->Z = FE_ONE; p->T = t;
    return 1;
}

/* RFC 9496 4.3.2 */
void eo_pt_encode(uint8_t out[32], const eo_pt *p) {
    constants_init();
    eo_fe u1, u2, t, inv, den1, den2, zinv, ix, iy, ench, x, y, deninv, s;
    eo_fe_add(&u1, &p->Z, &p->Y); eo_fe_sub(&t, &p->Z, &p->Y); eo_fe_mul(&u1, &u1, &t);
    eo_fe_mul(&u2, &p->X, &p->Y);
    eo_fe_sq(&t, &u2); eo_fe_mul(&t, &t, &u1);
    eo_fe_sqrt_ratio_i(&inv, &FE_ONE, &t);
    eo_fe_mul(&den1, &inv, &u1);
    eo_fe_mul(&den2, &inv, &u2);
    eo_fe_mul(&zinv, &den1, &den2); eo_fe_mul(&zinv, &zinv, &p->T);
    eo_fe_mul(&ix, &p->X, eo_fe_sqrt_m1());
    eo_fe_mul(&iy, &p->Y, eo_fe_sqrt_m1());
    eo_fe_mul(&ench, &den1, &C.invsqrt_a_minus_d);
    eo_fe_mul(&t, &p->T, &zinv);
    int rotate = eo_fe_isnegative(&t);
    if (rotate) { x = iy; y = ix; deninv = ench; } else { x = p->X; y = p->Y; deninv = den2; }
    eo_fe_mul(&t, &x, &zinv);
    if (eo_fe_isnegative(&t)) eo_fe_neg(&y, &y);
    eo_fe_sub(&t, &p->Z, &y);
    eo_fe_mul(&s, &deninv, &t);
    if (eo_fe_isnegative(&s)) eo_fe_neg(&s, &s);
    eo_fe_tobytes(out, &s);
}

int eo_pt_is_identity(const eo_pt *p) {
    /* ristretto equality with (0,1): X*1 == Y*0 or X*0 == Y*1 */
    return eo_fe_iszero(&p->X) || eo_fe_iszero(&p->Y);
}

int eo_pt_eq(const eo_pt *p, const eo_pt *q) {
    eo_fe a, b;
    eo_fe_mul(&a, &p->X, &q->Y); eo_fe_mul(&b, &p->Y, &q->X);
    if (eo_fe_eq(&a, &b)) return 1;
    eo_fe_mul(&a, &p->X, &q->X); eo_fe_mul(&b, &p->Y, &q->Y);
    return eo_fe_eq(&a, &b);
}

/* ---------------------------------------------------------------- scalar multiplication */

typedef struct { eo_fe ypx, ymx, z, t2d; } cached_pt;     /* (Y+X, Y-X, Z, 2dT) */
typedef struct { eo_fe ypx, ymx, xy2d; } niels_pt;        /* affine (y+x, y-x, 2dxy) */

static void to_cached(cached_pt *c, const eo_pt *p) {
    eo_fe_add(&c->ypx, &p->Y, &p->X); eo_fe_sub(&c->ymx, &p->Y, &p->X);
    c->z = p->Z; eo_fe_mul(&c->t2d, &p->T, &C.d2);
}

static void add_cached(eo_pt *r, const eo_pt *p, const cached_pt *q, int negate) {
    eo_fe a, b, c, d, e, f, g, h, t;
    eo_fe_sub(&a, &p->Y, &p->X); eo_fe_add(&b, &p->Y, &p->X);
    if (!negate) { eo_fe_mul(&a, &a, &q->ymx); eo_fe_mul(&b, &b, &q->ypx); }
    else         { eo_fe_mul(&a, &a, &q->ypx); eo_fe_mul(&b, &b, &q->ymx); }
    eo_fe_mul(&c, &p->T, &q->t2d);
    if (negate) eo_fe_neg(&c, &c);
    eo_fe_mul(&d, &p->Z, &q->z); eo_fe_add(&d, &d, &d);
    eo_fe_sub(&e, &b, &a); eo_fe_sub(&f, &d, &c); eo_fe_add(&g, &d, &c); eo_fe_add(&h, &b, &a);
    eo_fe_mul(&r->X, &e, &f); eo_fe_mul(&r->Y, &g, &h); eo_fe_mul(&r->T, &e, &h); eo_fe_mul(&r->Z, &f, &g);
    (void)t;
}

static void add_niels(eo_pt *r, const eo_pt *p, const niels_pt *q, int negate) {
    eo_fe a, b, c, d, e, f, g, h;
    eo_fe_sub(&a, &p->Y, &p->X); eo_fe_add(&b, &p->Y, &p->X);
    if (!negate) { eo_fe_mul(&a, &a, &q->ymx); eo_fe_mul(&b, &b, &q->ypx); }
    else         { eo_fe_mul(&a, &a, &q->ypx); eo_fe_mul(&b, &b, &q->ymx); }
    eo_fe_mul(&c, &p->T, &q->xy2d);
    if (negate) eo_fe_neg(&c, &c);
    eo_fe_add(&d, &p->Z, &p->Z);
    eo_fe_sub(&e, &b, &a); eo_fe_sub(&f, &d, &c); eo_fe_add(&g, &d, &c); eo_fe_add(&h, &b, &a);
    eo_fe_mul(&r->X, &e, &f); eo_fe_mul(&r->Y, &g, &h); eo_fe_mul(&r->T, &e, &h); eo_fe_mul(&r->Z, &f, &g);
}

/* width-w non-adjacent form, digits in naf[0..255], odd in (-2^(w-1), 2^(w-1)) */
static void compute_naf(int8_t naf[257], const eo_sc *s, int w) {
    uint64_t x[5] = {s->v[0], s->v[1], s->v[2], s->v[3], 0};
    memset(naf, 0, 257);
    const int width = 1 << w, half = width >> 1;
    int pos = 0;
    unsigned carry = 0;
    while (pos < 257) {
        int idx = pos >> 6, bit = pos & 63;
        uint64_t bits;
        if (bit <= 64 - w) bits = x[idx] >> bit;
        else bits = (x[idx] >> bit) | (idx < 4 ? x[idx + 1] << (64 - bit) : 0);
        unsigned window = carry + (unsigned)(bits & (uint64_t)(width - 1));
        if ((window & 1) == 0) { pos += 1; continue; }
        if (window < (unsigned)half) { carry = 0; naf[pos] = (int8_t)window; }
        else { carry = 1; naf[pos] = (int8_t)((int)window - width); }
        pos += w;
    }
}

static niels_pt G_NAF8[64];   /* odd multiples 1G, 3G, ..., 127G in affine Niels form */
static int g_naf8_ready = 0;

static void g_table_init(void) {
    if (g_naf8_ready) return;
    constants_init();
    eo_pt g2, cur = C.G;
    eo_pt_double(&g2, &C.G);
    for (int i = 0; i < 64; i++) {
        eo_fe zi, x, y;
        eo_fe_invert(&zi, &cur.Z);
        eo_fe_mul(&x, &cur.X, &zi); eo_fe_mul(&y, &cur.Y, &zi);
        eo_fe_add(&G_NAF8[i].ypx, &y, &x); eo_fe_sub(&G_NAF8[i].ymx, &y, &x);
        eo_fe_mul(&G_NAF8[i].xy2d, &x, &y); eo_fe_mul(&G_NAF8[i].xy2d, &G_NAF8[i].xy2d, &C.d2);
        eo_pt_add(&cur, &cur, &g2);
    }
    g_naf8_ready = 1;
}

#define EO_MAX_TERMS 17      /* SumOfSquaresProof::verify with 15 ciphertexts: 15 + 2 terms (proofs.c) */

/* r = sum s_i P_i + g*G  (g may be NULL): Straus with shared doublings */
static void straus(eo_pt *r, const eo_sc *scalars, const eo_pt *points, size_t n, const eo_sc *g) {
    constants_init();
    int8_t nafs[EO_MAX_TERMS][257];
    int8_t gnaf[257];
    cached_pt tables[EO_MAX_TERMS][8];
    for (size_t k = 0; k < n; k++) {
        compute_naf(nafs[k], &scalars[k], 5);
        eo_pt p2, cur = points[k];
        eo_pt_double(&p2, &points[k]);
        for (int i = 0; i < 8; i++) { to_cached(&tables[k][i], &cur); if (i < 7) eo_pt_add(&cur, &cur, &p2); }
    }
    if (g) { g_table_init(); compute_naf(gnaf, g, 8); }
    int top = 256;
    for (; top >= 0; top--) {
        int any = g && gnaf[top];
        for (size_t k = 0; k < n && !any; k++) any = nafs[k][top] != 0;
        if (any) break;
    }
    eo_pt acc;
    eo_pt_identity(&acc);
    for (int i = top; i >= 0; i--) {
        eo_pt_double(&acc, &acc);
        for (size_t k = 0; k < n; k++) {
            int d = nafs[k][i];
            if (d > 0) add_cached(&acc, &acc, &tables[k][d >> 1], 0);
            else if (d < 0) add_cached(&acc, &acc, &tables[k][(-d) >> 1], 1);
        }
        if (g) {
            int d = gnaf[i];
            if (d > 0) add_niels(&acc, &acc, &G_NAF8[d >> 1], 0);
            else if (d < 0) add_niels(&acc, &acc, &G_NAF8[(-d) >> 1], 1);
        }
    }
    *r = acc;
}

void eo_pt_multi_mul(eo_pt *r, const eo_sc *scalars, const eo_pt *points, size_t n) {
    if (n <= EO_MAX_TERMS) { straus(r, scalars, points, n, NULL); return; }
    eo_pt rest;                                    /* e.g. PublicKeySet::from_participants with a threshold above 17 */
    straus(r, scalars, points, EO_MAX_TERMS, NULL);
    eo_pt_multi_mul(&rest, scalars + EO_MAX_TERMS, points + EO_MAX_TERMS, n - EO_MAX_TERMS);
    eo_pt_add(r, r, &rest);
}

void eo_pt_double_mul_generator(eo_pt *r, const eo_sc *a, const eo_pt *A, const eo_sc *b) {
    straus(r, a, A, 1, b);
}

void eo_pt_mul_generator(eo_pt *r, const eo_sc *k) {
    straus(r, NULL, NULL, 0, k);
}

void eo_pt_mul(eo_pt *r, const eo_sc *k, const eo_pt *p) {
    straus(r, k, p, 1, NULL);
}

/* ---------------------------------------------------------------- byte-level helpers */

int eo_point_decode_check(const uint8_t s[32]) {
    eo_pt p;
    return eo_pt_decode(&p, s);
}

int eo_point_mul_bytes(uint8_t out[32], const uint8_t scalar[32], const uint8_t point[32]) {
    eo_pt p; eo_sc k;
    if (!eo_pt_decode(&p, point) || !eo_sc_from_canonical(&k, scalar)) return 0;
    eo_pt_mul(&p, &k, &p);
    eo_pt_encode(out, &p);
    return 1;
}

void eo_point_mul_generator_bytes(uint8_t out[32], const uint8_t scalar[32]) {
    eo_pt p; eo_sc k;
    eo_sc_from_canonical(&k, scalar);
    eo_pt_mul_generator(&p, &k);
    eo_pt_encode(out, &p);
}

int eo_point_add_bytes(uint8_t out[32], const uint8_t a[32], const uint8_t b[32]) {
    eo_pt p, q;
    if (!eo_pt_decode(&p, a) || !eo_pt_decode(&q, b)) return 0;
    eo_pt_add(&p, &p, &q);
    eo_pt_encode(out, &p);
    return 1;
}

int eo_point_sub_bytes(uint8_t out[32], const uint8_t a[32], const uint8_t b[32]) {
    eo_pt p, q;
    if (!eo_pt_decode(&p, a) || !eo_pt_decode(&q, b)) return 0;
    eo_pt_sub(&p, &p, &q);
    eo_pt_encode(out, &p);
    return 1;
}
