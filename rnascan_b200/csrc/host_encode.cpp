// Host-side symbol encoding (CPU threads).  The reference does this implicitly, per window:
// Seq.transcribe()/upper() (rnascan.py:191-193), the character switch of _pwm.c:41-63 and
// the dict lookup of matrix.py:36-41.  Here it happens once, while packing FASTA records
// into the device symbol stream.
#include <stdint.h>
#include <thread>
#include <vector>
#include <algorithm>
#include <cmath>
#include "../../include/rnascan_b200.h"

void rs_set_error(const char *fmt, ...);        // capi.cu

namespace {
struct Luts {
    uint8_t rna[256], ss[256];
    Luts()
    {
        for (int i = 0; i < 256; i++) { rna[i] = RS_RNA_OTHER; ss[i] = RS_SS_OTHER; }
        const char *r = "ACGU";
        for (int k = 0; k < 4; k++) { rna[(uint8_t)r[k]] = k; rna[(uint8_t)(r[k] | 0x20)] = k; }
        rna[(uint8_t)'T'] = 3; rna[(uint8_t)'t'] = 3;
        const char *s = "BEHLMRT";
        for (int k = 0; k < 7; k++) { ss[(uint8_t)s[k]] = k; ss[(uint8_t)(s[k] | 0x20)] = k | 8; }
    }
};
const Luts g_luts;

void run(const uint8_t *text, int64_t n, uint8_t *codes, const uint8_t *lut)
{
    unsigned hw = std::thread::hardware_concurrency();
    int64_t nt = std::max<int64_t>(1, std::min<int64_t>(hw ? hw : 1, n / (1 << 20)));
    auto work = [=](int64_t a, int64_t b) { for (int64_t i = a; i < b; i++) codes[i] = lut[text[i]]; };
    if (nt == 1) { work(0, n); return; }
    std::vector<std::thread> th;
    int64_t per = (n + nt - 1) / nt;
    for (int64_t t = 0; t < nt; t++) th.emplace_back(work, t * per, std::min(n, (t + 1) * per));
    for (auto &x : th) x.join();
}
}  // namespace

extern "C" int rs_host_encode_rna(const uint8_t *text, int64_t n, uint8_t *codes)
{
    if (n < 0 || (n > 0 && (!text || !codes))) return RS_ERR_INVALID;
    run(text, n, codes, g_luts.rna);
    return RS_OK;
}

extern "C" int rs_host_encode_struct(const uint8_t *text, int64_t n, uint8_t *codes)
{
    if (n < 0 || (n > 0 && (!text || !codes))) return RS_ERR_INVALID;
    run(text, n, codes, g_luts.ss);
    return RS_OK;
}

// The alphabet layout: index of the upper-cased byte in `letters` (bits 0-4), bit 5 for a lower-case byte (scored,
// not counted: str.upper() before scoring, matrix.py:36-41, but a case-sensitive Seq.count, rnascan.py:450-453),
// 0x1F for any other byte.  Letters: 1..31 distinct ASCII characters, none of them lower-case a-z (a lower-case
// letter would need two indices in one code).
extern "C" int rs_host_encode_alpha(const uint8_t *text, int64_t n, const uint8_t *letters, int n_letters,
                                    uint8_t *codes)
{
    if (n < 0 || (n > 0 && (!text || !codes))) return RS_ERR_INVALID;
    if (!letters || n_letters < 1 || n_letters > 31) {
        rs_set_error("alphabet of %d letters: 1..31 are supported", n_letters);
        return RS_ERR_INVALID;
    }
    uint8_t lut[256];
    std::fill(lut, lut + 256, (uint8_t)RS_ALPHA_OTHER);
    for (int k = 0; k < n_letters; k++) {
        const uint8_t c = letters[k];
        if (c >= 128 || (c >= 'a' && c <= 'z') || lut[c] != RS_ALPHA_OTHER) {
            rs_set_error("alphabet letter %d (byte %d) is not a distinct ASCII character outside a-z", k, (int)c);
            return RS_ERR_INVALID;
        }
        lut[c] = (uint8_t)k;
    }
    for (int c = 'a'; c <= 'z'; c++)
        if (lut[c - 32] != RS_ALPHA_OTHER) lut[c] = (uint8_t)(lut[c - 32] | RS_ALPHA_LOWER);
    run(text, n, codes, lut);
    return RS_OK;
}

// log2-odds of a normalised PFM against a background, in the arithmetic of CPython's
// math.log(p / b, 2) = log(p / b) / log(2.0) (Biopython log_odds, called at rnascan.py:248):
// p == 0 -> -inf; b == 0 -> +inf (p > 0) or NaN.  prob and out are [W][A] row-major, bg is [A]
// (already normalised to sum 1 by the caller, as Biopython does).
extern "C" int rs_host_log_odds(const double *prob, const double *bg, int W, int A, double *out)
{
    if (!prob || !bg || !out || W < 0 || A < 1) return RS_ERR_INVALID;
    const double ln2 = std::log(2.0);
    for (int i = 0; i < W; i++)
        for (int a = 0; a < A; a++) {
            const double p = prob[i * A + a], b = bg[a];
            double v;
            if (b > 0) v = p > 0 ? std::log(p / b) / ln2 : -INFINITY;
            else       v = p > 0 ? INFINITY : NAN;
            out[i * A + a] = v;
        }
    return RS_OK;
}
