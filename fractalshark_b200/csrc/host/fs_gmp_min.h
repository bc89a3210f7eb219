// fs_gmp_min.h -- the handful of GMP 6 mpf entry points the input generator needs, declared by hand:
// this image ships the GMP runtime (libgmp.so.10) but no gmp.h.  ABI per the GMP 6 manual
// (__mpf_struct {int _mp_prec; int _mp_size; long _mp_exp; mp_limb_t *_mp_d;}).
#pragma once
#include <stddef.h>

extern "C" {
typedef unsigned long fs_mp_limb_t;
typedef struct {
    int _mp_prec;
    int _mp_size;
    long _mp_exp;
    fs_mp_limb_t *_mp_d;
} fs_mpf_struct;
typedef fs_mpf_struct fs_mpf_t[1];

void __gmpf_init2(fs_mpf_struct *, unsigned long);
void __gmpf_clear(fs_mpf_struct *);
int __gmpf_set_str(fs_mpf_struct *, const char *, int);
void __gmpf_set(fs_mpf_struct *, const fs_mpf_struct *);
void __gmpf_set_ui(fs_mpf_struct *, unsigned long);
void __gmpf_set_d(fs_mpf_struct *, double);
void __gmpf_add(fs_mpf_struct *, const fs_mpf_struct *, const fs_mpf_struct *);
void __gmpf_sub(fs_mpf_struct *, const fs_mpf_struct *, const fs_mpf_struct *);
void __gmpf_mul(fs_mpf_struct *, const fs_mpf_struct *, const fs_mpf_struct *);
void __gmpf_div(fs_mpf_struct *, const fs_mpf_struct *, const fs_mpf_struct *);
void __gmpf_div_ui(fs_mpf_struct *, const fs_mpf_struct *, unsigned long);
void __gmpf_mul_2exp(fs_mpf_struct *, const fs_mpf_struct *, unsigned long);
void __gmpf_div_2exp(fs_mpf_struct *, const fs_mpf_struct *, unsigned long);
double __gmpf_get_d(const fs_mpf_struct *);
double __gmpf_get_d_2exp(long *, const fs_mpf_struct *);
int __gmpf_cmp(const fs_mpf_struct *, const fs_mpf_struct *);
}

#define fs_mpf_init2 __gmpf_init2
#define fs_mpf_clear __gmpf_clear
#define fs_mpf_set_str __gmpf_set_str
#define fs_mpf_set __gmpf_set
#define fs_mpf_set_ui __gmpf_set_ui
#define fs_mpf_set_d __gmpf_set_d
#define fs_mpf_add __gmpf_add
#define fs_mpf_sub __gmpf_sub
#define fs_mpf_mul __gmpf_mul
#define fs_mpf_div __gmpf_div
#define fs_mpf_div_ui __gmpf_div_ui
#define fs_mpf_mul_2exp __gmpf_mul_2exp
#define fs_mpf_div_2exp __gmpf_div_2exp
#define fs_mpf_get_d __gmpf_get_d
#define fs_mpf_get_d_2exp __gmpf_get_d_2exp
#define fs_mpf_cmp __gmpf_cmp
static inline int fs_mpf_sgn(const fs_mpf_struct *f) { return f->_mp_size < 0 ? -1 : (f->_mp_size > 0); }
