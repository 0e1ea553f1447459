// Plan management, error reporting and small utilities of the grates_b200 C ABI.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <vector>
#include "gb_common.cuh"

static thread_local char g_err[512] = "";
static thread_local long long g_launches = 0;

int gb_set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
void gb_count_launch(int n) { g_launches += n; }

extern "C" int gb_version(void) { return GB_VERSION; }
extern "C" const char* gb_last_error(void) { return g_err; }
extern "C" int64_t gb_launch_count(int reset) {
    long long v = g_launches;
    if (reset) g_launches = 0;
    return v;
}

// Stream-ordered scratch memory (gb_scratch) comes from a pool the library owns, one per device: its release threshold
// keeps the multi-GB temporaries of covariance propagation / filtering between calls (the default threshold of 0 returns
// them to the driver at every synchronisation: milliseconds per GB on the next call) without touching the attributes of
// the device's default pool, which belongs to the process (torch, other libraries).  gb_trim() hands the memory back.
static std::mutex g_pool_mutex;
static cudaMemPool_t g_pools[64] = {};

cudaMemPool_t gb_scratch_pool(int device) {
    if (device < 0 || device >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (!g_pools[device]) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        cudaMemPool_t pool = nullptr;
        if (cudaMemPoolCreate(&pool, &props) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        unsigned long long keep = ~0ULL;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        g_pools[device] = pool;
    }
    return g_pools[device];
}

void gb_retain_pool_memory(int device) { (void)gb_scratch_pool(device); }

extern "C" int gb_trim(int device) {
    GB_REQUIRE(device >= 0 && device < 64, "gb_trim: device %d out of range", device);
    cudaMemPool_t pool = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        pool = g_pools[device];
    }
    if (!pool) return GB_OK;
    GB_CUDA(cudaSetDevice(device));
    GB_CUDA(cudaDeviceSynchronize());
    GB_CUDA(cudaMemPoolTrimTo(pool, 0));
    return GB_OK;
}

extern "C" int gb_device_count(int* count) {
    GB_REQUIRE(count != nullptr, "gb_device_count: count is NULL");
    GB_CUDA(cudaGetDeviceCount(count));
    return GB_OK;
}

template <typename T>
static int upload(T** d, const std::vector<T>& h) {
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(d), h.size() * sizeof(T)));
    GB_CUDA(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return GB_OK;
}

void gb_recursion_tables(int nmax, int npts, const double* sin_theta, std::vector<double>& ra,
                         std::vector<double>& rb, std::vector<double>& rc, std::vector<double>& pmm) {
    const int L = nmax + 1;
    // Recursion coefficients, evaluated exactly as utilities.py:46,52,54 (IEEE double, same
    // operation order), so that the device recursion reproduces the reference table bit for bit.
    ra.assign((size_t)L * L, 0.0);
    rb.assign((size_t)L * L, 0.0);
    rc.assign(L, 0.0);
    for (int n = 0; n < L; ++n) rc[n] = std::sqrt((double)(2 * n + 1));
    for (int n = 2; n < L; ++n)
        for (int m = 0; m <= n - 2; ++m) {
            const double dn = n, dm = m;
            ra[(size_t)n * L + m] = std::sqrt((2.0 * dn - 1.0) / (dn - dm) * (2.0 * dn + 1.0) / (dn + dm));
            rb[(size_t)n * L + m] =
                std::sqrt((2.0 * dn + 1.0) / (2.0 * dn - 3.0) * (dn - dm - 1.0) / (dn - dm) * (dn + dm - 1.0) / (dn + dm));
        }
    // Sectorial seeds P_mm(theta_i) (utilities.py:37,39,41-43): O(npts * L) values, the only part
    // of the Legendre triangle that is tabulated; everything below the diagonal is recomputed on
    // the fly inside the kernels.
    pmm.assign((size_t)npts * L, 0.0);
    for (int i = 0; i < npts; ++i) {
        double* row = &pmm[(size_t)i * L];
        row[0] = 1.0;
        if (L > 1) row[1] = std::sqrt(3.0) * sin_theta[i];
        for (int n = 2; n < L; ++n) {
            const double dn = n;
            const double f = std::sqrt((2.0 * dn + 1.0) / (2.0 * dn));
            const double fs = f * sin_theta[i];
            row[n] = fs * row[n - 1];
        }
    }
}

extern "C" int gb_plan_create(gb_plan** plan, int nmax, int nlat, int nlon, const double* cos_theta,
                              const double* sin_theta, const double* kn, const double* cos_mlon,
                              const double* sin_mlon, int device) {
    GB_REQUIRE(plan != nullptr, "gb_plan_create: plan is NULL");
    *plan = nullptr;
    GB_REQUIRE(nmax >= 0 && nmax <= 2047, "gb_plan_create: nmax=%d out of range [0, 2047]", nmax);
    GB_REQUIRE(nlat >= 1 && nlon >= 1, "gb_plan_create: empty grid (%d x %d)", nlat, nlon);
    GB_REQUIRE(cos_theta && sin_theta && kn && cos_mlon && sin_mlon, "gb_plan_create: NULL table pointer");
    int ndev = 0;
    GB_CUDA(cudaGetDeviceCount(&ndev));
    GB_REQUIRE(device >= 0 && device < ndev, "gb_plan_create: device %d not available (%d visible)", device, ndev);
    GB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    GB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return gb_set_error(GB_ERR_UNSUPPORTED, "gb_plan_create: device %d is sm_%d%d; this library is built for sm_100a",
                            device, prop.major, prop.minor);

    gb_retain_pool_memory(device);
    gb_plan* p = new gb_plan();
    p->device = device;
    p->nmax = nmax;
    p->L = nmax + 1;
    p->nlat = nlat;
    p->nlon = nlon;
    p->kpad = (2 * p->L + 3) / 4 * 4;
    p->nlp = (nlon + 7) / 8 * 8;
    p->sm_count = prop.multiProcessorCount;
    const int L = p->L;

    std::vector<double> ra, rb, rc, pmm;
    gb_recursion_tables(nmax, nlat, sin_theta, ra, rb, rc, pmm);
    std::vector<double> trig((size_t)p->kpad * p->nlp, 0.0);
    for (int m = 0; m < L; ++m)
        for (int j = 0; j < nlon; ++j) {
            trig[(size_t)(2 * m) * p->nlp + j] = cos_mlon[(size_t)m * nlon + j];
            if (m > 0) trig[(size_t)(2 * m + 1) * p->nlp + j] = sin_mlon[(size_t)m * nlon + j];
        }
    std::vector<double> ct(cos_theta, cos_theta + nlat), knv(kn, kn + (size_t)nlat * L);

    // Equatorial symmetry: parallel nlat-1-i mirrors parallel i (cos(theta) changes sign; sin(theta), and with it the
    // sectorial seeds, and the radius-dependent degree factors are the same), and the folded stage 1 derives the southern
    // parallels from the northern recursion, P_nm(pi - theta) = (-1)^(n-m) P_nm(theta).  The reference's own tables are
    // mirror images only to rounding (arccos next to the poles), so the shortcut is gated on a measurement: the zonal
    // functions -- the ones that are large at the poles and most sensitive to cos(theta) -- are run for both
    // hemispheres with the kernels' recursion, and the fold is used only if no degree differs by more than 2e-13 of its
    // largest value (0.5 deg grid: 5e-14; a 0.25 deg grid: 1e-12, not folded), i.e. ten times below the parity bar.
    {
        bool fold = (nlat % 2 == 0) && nlat >= 2 && L >= 2;
        const int nh = nlat / 2;
        std::vector<double> diff((size_t)nh * L, 0.0), scale(L, 0.0);
        std::vector<char> seed_bad(nh, 0);
        for (int i = 0; i < nh && fold; ++i) {
            const int j = nlat - 1 - i;
            double n2 = 1.0, s2 = 1.0, n1 = rc[1] * ct[i], s1 = rc[1] * ct[j];
            for (int n = 0; n < L; ++n) {
                double pn, ps;
                if (n == 0) { pn = 1.0; ps = 1.0; }
                else if (n == 1) { pn = n1; ps = s1; }
                else {
                    pn = ra[(size_t)n * L] * ct[i] * n1 - rb[(size_t)n * L] * n2;
                    ps = ra[(size_t)n * L] * ct[j] * s1 - rb[(size_t)n * L] * s2;
                    n2 = n1; n1 = pn; s2 = s1; s1 = ps;
                }
                const double vn = pn * knv[(size_t)i * L + n], vs = ((n & 1) ? -ps : ps) * knv[(size_t)j * L + n];
                diff[(size_t)i * L + n] = std::fabs(vn - vs);
                scale[n] = std::max(scale[n], std::fabs(vn));
                const double pa = pmm[(size_t)i * L + n], pb = pmm[(size_t)j * L + n];
                if (std::fabs(pa - pb) > 2e-13 * (n + 1) * std::fabs(pa) + 1e-200) seed_bad[i] = 1;   // (underflow next to the poles)
            }
        }
        // Parallels that fail the gate are next to the poles (the reference's arccos): up to two leading tiles of 32
        // parallels per hemisphere are left to the unfolded stage, everything else is folded.
        int last_bad = -1;
        for (int i = 0; i < nh && fold; ++i) {
            bool bad = seed_bad[i] != 0;
            for (int n = 0; n < L && !bad; ++n)
                if (diff[(size_t)i * L + n] > 2e-13 * scale[n]) bad = true;
            if (bad) last_bad = i;
        }
        int cap = last_bad < 0 ? 0 : (last_bad / 32 + 1) * 32;
        if (cap > 64 || (cap > 0 && (nlat < 128 || nh - cap < 32))) fold = false;
        p->fold_ns = fold ? 1 : 0;
        p->fold_cap = fold ? cap : 0;
    }

    // Four-fold longitude symmetry: with h = nlon/2, q = nlon/4 and mu = lon[h + j'] in (0, pi/2),
    //   lon[nlon-1-j'] = pi - mu,  lon[h-1-j'] = -mu,  lon[j'] = mu - pi.
    // Checked on the tables themselves (they are what the kernels multiply with).
    std::vector<int> krow_id(p->kpad), krow_sym(p->kpad, 0);
    for (int k = 0; k < p->kpad; ++k) krow_id[k] = k;
    std::vector<double> trig_q;
    {
        bool sym = (nlon % 8 == 0);   // first quadrant must hold an even number of meridians
        const int h = nlon / 2, q = nlon / 4;
        for (int m = 0; m < L && sym; ++m) {
            // numpy evaluates cos(m * lon): the product is rounded (half an ulp of |m lon| <= m pi) and lon
            // itself carries half an ulp of pi, so mirrored table entries differ by a few (m+1) * 1e-15
            const double tol = 4.0 * (m + 1) * 2.220446049250313e-16 * 3.141592653589793;
            const double sg = (m & 1) ? -1.0 : 1.0;
            const double* c = cos_mlon + (size_t)m * nlon;
            const double* s = sin_mlon + (size_t)m * nlon;
            for (int j = 0; j < q; ++j) {
                const double cq = c[h + j], sq = s[h + j];
                if (std::fabs(c[nlon - 1 - j] - sg * cq) > tol || std::fabs(s[nlon - 1 - j] + sg * sq) > tol ||
                    std::fabs(c[h - 1 - j] - cq) > tol || std::fabs(s[h - 1 - j] + sq) > tol ||
                    std::fabs(c[j] - sg * cq) > tol || std::fabs(s[j] - sg * sq) > tol) {
                    sym = false;
                    break;
                }
            }
        }
        p->sym = sym ? 1 : 0;
        if (sym) {
            p->nq = q;
            p->nqp = (q + 7) / 8 * 8;
            const int cnt[4] = {nmax / 2 + 1, (nmax + 1) / 2, nmax / 2, (nmax + 1) / 2};
            for (int g = 0; g < 4; ++g) p->grp_off[g + 1] = p->grp_off[g] + (cnt[g] + 3) / 4 * 4;
            p->kpad_s = p->grp_off[4] + 4;
            trig_q.assign((size_t)p->kpad_s * p->nqp, 0.0);
            for (int m = 0; m < L; ++m) {
                const int rc_row = p->grp_off[m & 1] + m / 2;
                krow_sym[2 * m] = rc_row;
                int rs_row = p->kpad_s - 1;   // (m = 0, sin) does not exist: dummy row
                if (m > 0) rs_row = p->grp_off[2 + (m & 1)] + ((m & 1) ? m / 2 : m / 2 - 1);
                krow_sym[2 * m + 1] = rs_row;
                for (int j = 0; j < q; ++j) {
                    trig_q[(size_t)rc_row * p->nqp + j] = cos_mlon[(size_t)m * nlon + h + j];
                    if (m > 0) trig_q[(size_t)rs_row * p->nqp + j] = sin_mlon[(size_t)m * nlon + h + j];
                }
            }
            for (int k = 2 * L; k < p->kpad; ++k) krow_sym[k] = p->kpad_s - 1;
        }
    }

    // Eight-fold symmetry: the first-quadrant meridians mirror about pi/4, mu' = pi/2 - mu = lon[h + q - 1 - j], where
    //   m = 0 (4): cos(m mu') =  cos(m mu), sin(m mu') = -sin(m mu)      m = 1 (4): cos(m mu') =  sin(m mu), sin(m mu') =  cos(m mu)
    //   m = 2 (4): cos(m mu') = -cos(m mu), sin(m mu') =  sin(m mu)      m = 3 (4): cos(m mu') = -sin(m mu), sin(m mu') = -cos(m mu)
    // so the even orders split once more (half their multiply-adds) and the odd orders are contracted with the octant's
    // cosine AND sine row (same multiply-adds, shared coefficient fragments).  Checked on the tables, as above.
    std::vector<int> krow_oct(p->kpad, 0);
    std::vector<double> trig_o_t;
    if (p->sym && nlon % 16 == 0) {
        const int h = nlon / 2, q = nlon / 4, no = nlon / 8;
        bool oct = true;
        for (int m = 0; m < L && oct; ++m) {
            const double tol = 4.0 * (m + 1) * 2.220446049250313e-16 * 3.141592653589793;
            const double* c = cos_mlon + (size_t)m * nlon;
            const double* s = sin_mlon + (size_t)m * nlon;
            for (int j = 0; j < no; ++j) {
                const double cm = c[h + j], sm = s[h + j], cp = c[h + q - 1 - j], sp = s[h + q - 1 - j];
                double ec, es;
                switch (m & 3) {
                    case 0: ec = cm; es = -sm; break;
                    case 1: ec = sm; es = cm; break;
                    case 2: ec = -cm; es = sm; break;
                    default: ec = -sm; es = -cm; break;
                }
                if (std::fabs(cp - ec) > tol || std::fabs(sp - es) > tol) {
                    oct = false;
                    break;
                }
            }
        }
        p->oct = oct ? 1 : 0;
        if (oct) {
            p->no = no;
            // group sizes: orders 0, 4, .. | 2, 6, .. (cosine coefficients); 4, 8, .. | 2, 6, .. (sine); odd orders (cos), (sin)
            int cnt[6] = {0, 0, 0, 0, 0, 0};
            for (int m = 0; m < L; ++m) {
                if ((m & 3) == 0) { ++cnt[0]; if (m > 0) ++cnt[2]; }
                else if ((m & 3) == 2) { ++cnt[1]; ++cnt[3]; }
                else { ++cnt[4]; ++cnt[5]; }
            }
            for (int g = 0; g < 6; ++g) p->ogrp_off[g + 1] = p->ogrp_off[g] + (cnt[g] + 3) / 4 * 4;
            p->kpad_o = p->ogrp_off[6] + 4;
            const int nop = (no + GB_Q_TN - 1) / GB_Q_TN * GB_Q_TN;
            std::vector<double> t1((size_t)p->kpad_o * nop, 0.0), t2((size_t)p->kpad_o * nop, 0.0);
            int fill[6] = {0, 0, 0, 0, 0, 0};
            for (int m = 0; m < L; ++m) {
                const double* c = cos_mlon + (size_t)m * nlon + h;
                const double* s = sin_mlon + (size_t)m * nlon + h;
                int rc_row, rs_row = p->kpad_o - 1;           // (m = 0, sin) does not exist: dummy row
                if ((m & 1) == 0) {
                    const int gc = (m & 3) == 0 ? 0 : 1, gs = gc + 2;
                    rc_row = p->ogrp_off[gc] + fill[gc]++;
                    if (m > 0) rs_row = p->ogrp_off[gs] + fill[gs]++;
                    for (int j = 0; j < no; ++j) {
                        t1[(size_t)rc_row * nop + j] = c[j];
                        if (m > 0) t1[(size_t)rs_row * nop + j] = s[j];
                    }
                } else {
                    const double sg = (m & 3) == 1 ? 1.0 : -1.0;
                    rc_row = p->ogrp_off[4] + fill[4]++;
                    rs_row = p->ogrp_off[5] + fill[5]++;
                    for (int j = 0; j < no; ++j) {
                        t1[(size_t)rc_row * nop + j] = c[j];          // A_m cos(m mu)           -> CO(mu)
                        t2[(size_t)rc_row * nop + j] = sg * s[j];     // A_m (+-) sin(m mu)      -> CO(pi/2 - mu)
                        t1[(size_t)rs_row * nop + j] = s[j];          // B_m sin(m mu)           -> SO(mu)
                        t2[(size_t)rs_row * nop + j] = sg * c[j];     // B_m (+-) cos(m mu)      -> SO(pi/2 - mu)
                    }
                }
                krow_oct[2 * m] = rc_row;
                krow_oct[2 * m + 1] = rs_row;
            }
            for (int k = 2 * L; k < p->kpad; ++k) krow_oct[k] = p->kpad_o - 1;
            // tiles of 32 octant meridians, both tables side by side; the columns of a warp's 16-column slab interleaved as
            // in the quadrant tiles (a lane's two fragments are four consecutive meridians)
            p->n_otiles = nop / GB_Q_TN;
            trig_o_t.assign((size_t)p->n_otiles * 2 * p->kpad_o * GB_Q_LDB, 0.0);
            for (int t = 0; t < p->n_otiles; ++t)
                for (int tb = 0; tb < 2; ++tb)
                    for (int k = 0; k < p->kpad_o; ++k)
                        for (int cc = 0; cc < GB_Q_TN; ++cc) {
                            const int slab = cc / 16, tc = cc % 16;
                            const int src = t * GB_Q_TN + slab * 16 + 4 * ((tc % 8) / 2) + 2 * (tc / 8) + (tc % 2);
                            trig_o_t[(((size_t)t * 2 + tb) * p->kpad_o + k) * GB_Q_LDB + cc] =
                                (tb ? t2 : t1)[(size_t)k * nop + src];
                        }
        }
    }

    // tiled + padded copies of the longitude tables (one bulk copy per pipeline stage)
    p->ab_rows = p->kpad > p->kpad_s ? p->kpad : p->kpad_s;
    if (p->kpad_o > p->ab_rows) p->ab_rows = p->kpad_o;
    p->n_ntiles = (p->nlp + GB_S2_TN - 1) / GB_S2_TN;
    std::vector<double> trig_t((size_t)p->n_ntiles * p->kpad * GB_S2_LDB, 0.0);
    for (int t = 0; t < p->n_ntiles; ++t)
        for (int k = 0; k < p->kpad; ++k)
            for (int c = 0; c < GB_S2_TN && t * GB_S2_TN + c < p->nlp; ++c)
                trig_t[((size_t)t * p->kpad + k) * GB_S2_LDB + c] = trig[(size_t)k * p->nlp + t * GB_S2_TN + c];
    std::vector<double> trig_q_t;
    if (p->sym) {
        p->n_qtiles = (p->nqp + GB_Q_TN - 1) / GB_Q_TN;
        trig_q_t.assign((size_t)p->n_qtiles * p->kpad_s * GB_Q_LDB, 0.0);
        // Inside every 16-column slab of a warp the columns are interleaved so that a lane's two DMMA fragments
        // (tile columns 2q, 2q+1 and 8+2q, 9+2q) are FOUR CONSECUTIVE meridians 4q .. 4q+3: one 32-byte store per
        // output row and lane (gb_fourier_stage2_sym)
        for (int t = 0; t < p->n_qtiles; ++t)
            for (int k = 0; k < p->kpad_s; ++k)
                for (int c = 0; c < GB_Q_TN; ++c) {
                    const int slab = c / 16, tc = c % 16;
                    const int src = t * GB_Q_TN + slab * 16 + 4 * ((tc % 8) / 2) + 2 * (tc / 8) + (tc % 2);
                    if (src < p->nqp)
                        trig_q_t[((size_t)t * p->kpad_s + k) * GB_Q_LDB + c] = trig_q[(size_t)k * p->nqp + src];
                }
    }

    // stage-1 tables (see gb_common.cuh)
    p->nlat_pad = (nlat + GB_T1_TM - 1) / GB_T1_TM * GB_T1_TM;
    p->lpad = (L + GB_T1_KC - 1) / GB_T1_KC * GB_T1_KC;
    std::vector<double> ct_pad(p->nlat_pad, 0.0), kn_t((size_t)(L + GB_T1_KC) * p->nlat_pad, 0.0),
        pmm_t((size_t)L * p->nlat_pad, 0.0), rec_a((size_t)L * p->lpad, 0.0), rec_b((size_t)L * p->lpad, 0.0);
    for (int i = 0; i < nlat; ++i) {
        ct_pad[i] = ct[i];
        for (int n = 0; n < L; ++n) {
            kn_t[(size_t)n * p->nlat_pad + i] = knv[(size_t)i * L + n];
            pmm_t[(size_t)n * p->nlat_pad + i] = pmm[(size_t)i * L + n];
        }
    }
    for (int m = 0; m < L; ++m)
        for (int n = m + 1; n < L; ++n) {
            // (a ct) p1 - 0 * p2 at n = m+1 is bit-identical to utilities.py:46
            rec_a[(size_t)m * p->lpad + (n - m)] = (n == m + 1) ? rc[n] : ra[(size_t)n * L + m];
            rec_b[(size_t)m * p->lpad + (n - m)] = (n == m + 1) ? 0.0 : rb[(size_t)n * L + m];
        }

    // first table row of every order in the tiled Legendre table / tiled X (orders padded to 8 rows)
    std::vector<int> roff(L + 1, 0);
    for (int m = 0; m < L; ++m) roff[m + 1] = roff[m] + ((L - m + 7) & ~7);
    p->ptab_rtot = roff[L];

    int rc_ = GB_OK;
    if ((rc_ = upload(&p->d_ptab_roff, roff)) || (rc_ = upload(&p->d_ct_pad, ct_pad)) || (rc_ = upload(&p->d_kn_t, kn_t)) || (rc_ = upload(&p->d_pmm_t, pmm_t)) ||
        (rc_ = upload(&p->d_rec_a, rec_a)) || (rc_ = upload(&p->d_rec_b, rec_b)) ||
        (rc_ = upload(&p->d_trig_t, trig_t)) || (p->sym && (rc_ = upload(&p->d_trig_q_t, trig_q_t))) ||
        (rc_ = upload(&p->d_ct, ct)) || (rc_ = upload(&p->d_kn, knv)) || (rc_ = upload(&p->d_pmm, pmm)) ||
        (rc_ = upload(&p->d_ra, ra)) || (rc_ = upload(&p->d_rb, rb)) || (rc_ = upload(&p->d_rc, rc)) ||
        (rc_ = upload(&p->d_trig, trig)) ||
        (rc_ = upload(&p->d_krow_id, krow_id)) || (rc_ = upload(&p->d_krow_sym, krow_sym)) ||
        (p->oct && ((rc_ = upload(&p->d_krow_oct, krow_oct)) || (rc_ = upload(&p->d_trig_o_t, trig_o_t)))) ||
        (p->sym && (rc_ = upload(&p->d_trig_q, trig_q)))) {
        gb_plan_destroy(p);
        return rc_;
    }
    *plan = p;
    return GB_OK;
}

extern "C" int gb_plan_info(const gb_plan* plan, int* nmax, int* nlat, int* nlon, int* device) {
    GB_REQUIRE(plan != nullptr, "gb_plan_info: plan is NULL");
    if (nmax) *nmax = plan->nmax;
    if (nlat) *nlat = plan->nlat;
    if (nlon) *nlon = plan->nlon;
    if (device) *device = plan->device;
    return GB_OK;
}

extern "C" int gb_plan_is_symmetric(const gb_plan* plan) { return (plan && plan->sym) ? (plan->oct ? 2 : 1) : 0; }

extern "C" int gb_plan_is_folded(const gb_plan* plan) { return (plan && plan->fold_ns) ? 1 + plan->fold_cap / 32 : 0; }

extern "C" int gb_plan_destroy(gb_plan* p) {
    if (!p) return GB_OK;
    cudaSetDevice(p->device);
    cudaFree(p->d_ct); cudaFree(p->d_kn); cudaFree(p->d_pmm); cudaFree(p->d_ra); cudaFree(p->d_rb);
    cudaFree(p->d_rc); cudaFree(p->d_trig);
    cudaFree(p->d_ct_pad); cudaFree(p->d_kn_t); cudaFree(p->d_pmm_t); cudaFree(p->d_rec_a); cudaFree(p->d_rec_b);
    cudaFree(p->d_krow_id); cudaFree(p->d_krow_sym); cudaFree(p->d_trig_q);
    cudaFree(p->d_krow_oct); cudaFree(p->d_trig_o_t);
    cudaFree(p->d_trig_t); cudaFree(p->d_trig_q_t); cudaFree(p->d_x); cudaFree(p->d_ab);
    cudaFree(p->d_io_in); cudaFree(p->d_io_out[0]); cudaFree(p->d_io_out[1]);
    cudaFree(p->d_lon_ops); cudaFree(p->d_lat_ops); cudaFree(p->d_lat_off);
    cudaFree(p->d_ana_w_t); cudaFree(p->d_ana_kmap); cudaFree(p->d_ana_vf);
    cudaFree(p->d_ana_lat_t); cudaFree(p->d_ana_lat_m); cudaFree(p->d_ana_lat_n); cudaFree(p->d_ana_gt);
    delete[] p->h_lat_off;
    gb_cov_layout_free(p);
    for (auto& t : p->d_ptab) cudaFree(t);
    cudaFree(p->d_ptab_roff);
    if (p->ws_free) cudaEventDestroy(p->ws_free);
    if (p->prof_ev) {
        for (int i = 0; i < p->prof_capacity * 4; ++i) cudaEventDestroy(p->prof_ev[i]);
        delete[] p->prof_ev;
    }
    if (p->s_compute) cudaStreamDestroy(p->s_compute);
    if (p->s_copy) cudaStreamDestroy(p->s_copy);
    for (auto& e : p->ev)
        if (e) cudaEventDestroy(e);
    delete p;
    return GB_OK;
}

int gb_plan_acquire(gb_plan* p, cudaStream_t st) {
    if (p->ws_used && p->ws_stream != st) {
        if (!p->ws_free) GB_CUDA(cudaEventCreateWithFlags(&p->ws_free, cudaEventDisableTiming));
        // everything queued on the previous call's stream so far includes that call's last kernel
        if (cudaEventRecord(p->ws_free, p->ws_stream) != cudaSuccess || cudaStreamWaitEvent(st, p->ws_free, 0) != cudaSuccess) {
            cudaGetLastError();                       // e.g. the other stream no longer exists
            GB_CUDA(cudaDeviceSynchronize());
        }
    }
    p->ws_stream = st;
    p->ws_used = 1;
    return GB_OK;
}

// Grow the synthesis / analysis workspace to hold n_epochs (never shrinks).
int gb_plan_ensure_workspace(gb_plan* p, int n_epochs) {
    if (n_epochs <= p->ws_epochs) return GB_OK;
    GB_CUDA(cudaSetDevice(p->device));
    GB_CUDA(cudaDeviceSynchronize());
    cudaFree(p->d_x); p->d_x = nullptr;
    cudaFree(p->d_ab); p->d_ab = nullptr;
    p->ws_epochs = 0;
    const long long m = (long long)n_epochs * p->nlat;
    const long long mpad = (m + 127) / 128 * 128;
    // X holds either the order-wise layout or the tiled one (80- or 240-column tiles + 4 pad columns, gb_pack.cu)
    const size_t cols = 2 * (size_t)n_epochs;
    const size_t tiled = (size_t)p->ptab_rtot * std::max({((cols + 79) / 80) * 84, ((cols + 119) / 120) * 124, ((cols + 239) / 240) * 244});
    const size_t x_elems = std::max((size_t)p->L * (p->L + 1) / 2 * cols, tiled);
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_x), x_elems * sizeof(double)));
    p->x_elems = x_elems;
    p->x_layout_key = 0;
    const size_t ab_elems = (size_t)(mpad / GB_TM) * p->ab_rows * GB_LDA;
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ab), ab_elems * sizeof(double)));
    // padding rows and padded columns must stay finite (they meet zero trig rows / masked stores)
    GB_CUDA(cudaMemset(p->d_ab, 0, ab_elems * sizeof(double)));
    GB_CUDA(cudaDeviceSynchronize());
    p->ws_epochs = n_epochs;
    p->ws_mpad = mpad;
    return GB_OK;
}

extern "C" int gb_plan_set_profiling(gb_plan* p, int capacity) {
    GB_REQUIRE(p != nullptr && capacity >= 0, "gb_plan_set_profiling: bad argument");
    GB_CUDA(cudaSetDevice(p->device));
    if (p->prof_ev) {
        GB_CUDA(cudaDeviceSynchronize());
        for (int i = 0; i < p->prof_capacity * 4; ++i) cudaEventDestroy(p->prof_ev[i]);
        delete[] p->prof_ev;
        p->prof_ev = nullptr;
    }
    p->prof_capacity = 0;
    p->prof_count = 0;
    if (capacity > 0) {
        p->prof_ev = new cudaEvent_t[(size_t)capacity * 4];
        for (int i = 0; i < capacity * 4; ++i) GB_CUDA(cudaEventCreate(&p->prof_ev[i]));
        p->prof_capacity = capacity;
    }
    return GB_OK;
}

extern "C" int gb_plan_stage_times(gb_plan* p, double* ms, int max_calls, int* n_calls) {
    GB_REQUIRE(p != nullptr && ms != nullptr && n_calls != nullptr, "gb_plan_stage_times: NULL argument");
    const int n = p->prof_count < max_calls ? p->prof_count : max_calls;
    for (int c = 0; c < n; ++c) {
        cudaEvent_t* ev = p->prof_ev + (size_t)c * 4;
        GB_CUDA(cudaEventSynchronize(ev[3]));
        for (int s = 0; s < 3; ++s) {
            float t = 0.f;
            GB_CUDA(cudaEventElapsedTime(&t, ev[s], ev[s + 1]));
            ms[c * 3 + s] = t;
        }
    }
    *n_calls = n;
    p->prof_count = 0;
    return GB_OK;
}

extern "C" int gb_host_alloc(void** ptr, uint64_t bytes) {
    GB_REQUIRE(ptr != nullptr, "gb_host_alloc: ptr is NULL");
    GB_CUDA(cudaMallocHost(ptr, bytes ? bytes : 1));
    return GB_OK;
}
extern "C" int gb_host_free(void* ptr) {
    if (ptr) GB_CUDA(cudaFreeHost(ptr));
    return GB_OK;
}

// ---------------------------------------------------------------------------------------------
// FP64 pipe probes (roofline denominators)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gb_probe_dmma(double* out, int iters, double a, double b) {
    double acc[8][2];
#pragma unroll
    for (int c = 0; c < 8; ++c) { acc[c][0] = threadIdx.x * 1e-9; acc[c][1] = c; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < 8; ++c) gb::dmma_884(acc[c][0], acc[c][1], a, b);
    }
    double s = 0;
#pragma unroll
    for (int c = 0; c < 8; ++c) s += acc[c][0] + acc[c][1];
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void __launch_bounds__(256) gb_probe_dfma(double* out, int iters, double a, double b) {
    double acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = threadIdx.x * 1e-9 + c;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] = fma(acc[c], a, b);
    }
    double s = 0;
#pragma unroll
    for (int c = 0; c < 8; ++c) s += acc[c];
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" int gb_probe_fp64_peak(int device, double* dmma_tflops, double* dfma_tflops) {
    GB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    GB_CUDA(cudaGetDeviceProperties(&prop, device));
    const int grid = prop.multiProcessorCount * 4;
    double* out = nullptr;
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&out), (size_t)grid * 256 * sizeof(double)));
    cudaEvent_t e0, e1;
    GB_CUDA(cudaEventCreate(&e0));
    GB_CUDA(cudaEventCreate(&e1));
    const int iters = 4000;
    float ms = 0.f;
    double best_mma = 0, best_fma = 0;
    for (int rep = 0; rep < 6; ++rep) {
        GB_CUDA(cudaEventRecord(e0));
        gb_probe_dmma<<<grid, 256>>>(out, iters, 1.0000001, 1e-9);
        GB_CUDA(cudaEventRecord(e1));
        GB_CUDA(cudaEventSynchronize(e1));
        GB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double t1 = 2.0 * 256 * 8 * (double)iters * 8.0 * grid / (ms * 1e-3) / 1e12;
        if (rep > 0 && t1 > best_mma) best_mma = t1;
        GB_CUDA(cudaEventRecord(e0));
        gb_probe_dfma<<<grid, 256>>>(out, iters * 4, 1.0000001, 1e-9);
        GB_CUDA(cudaEventRecord(e1));
        GB_CUDA(cudaEventSynchronize(e1));
        GB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double t2 = 2.0 * 8 * (double)iters * 4 * 256.0 * grid / (ms * 1e-3) / 1e12;
        if (rep > 0 && t2 > best_fma) best_fma = t2;
    }
    GB_CUDA(cudaGetLastError());
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    if (dmma_tflops) *dmma_tflops = best_mma;
    if (dfma_tflops) *dfma_tflops = best_fma;
    return GB_OK;
}
