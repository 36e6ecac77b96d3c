// capi.cpp — the extern "C" boundary of libmpcf.so (see include/mpcf.h for what each entry replaces).
#include <cmath>
#include <cstdint>
#include <cstring>
#include <mutex>
#include <new>
#include <string>

#include "kernels.cuh"
#include "model.hpp"

using namespace mpcf;

struct mpcf_model {
    HostModel h;
    Family fam = FAM_GENERIC64;
    // static-family parameter block (largest variant), filled for the family in use
    StaticParams<12> sp12;
    StaticParams<6> chain6[2];  // forest12x6: the two arms as stand-alone 6-DOF chains
    StaticParams<14> sp14;
    StaticParams<7> sp7, chain7[2];  // chain7 / forest14x7 (the reference's Centauro layout: 2 x 7 arms)
    StaticParams<6> sp6;
    StaticParams<3> sp3;
    // device copy of the generic blob, uploaded lazily on first launch (model creation needs no GPU)
    mutable std::mutex mu;
    mutable double *d_dbl = nullptr;
    mutable int *d_int = nullptr;
    mutable bool dirty = true;
    mutable int device = -1;  // device holding the uploaded blob (run-time-topology families)
    int fd_status = 0;  // 0 unknown, 1 ok, -1 singular
    CoupleHost couple;  // coupled fatigue of a two-arm model (mpcf_model_set_coupling)
    int npat = 0;       // size of the ancestor pattern sum_k (depth_k + 1): packed storage of the tree Jacobian pipeline
};

static thread_local std::string g_err;
static int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}
extern "C" const char *mpcf_last_error(void) { return g_err.c_str(); }
extern "C" long mpcf_launch_count(void) { return launch_count(); }

extern "C" void mpcf_opts_default(mpcf_opts *o)
{
    if (!o) return;
    const double Ra = 10.0, Rh = 2.0, Rth = 300.0 * 9.0 / 309.0, Cth = 15.0, ktau = 40.0;
    const double tth = Rth * Cth;
    o->armature = 0.0;
    o->gravity[0] = 0.0; o->gravity[1] = 0.0; o->gravity[2] = -9.81;
    o->lambda = 1.0 / tth;
    o->kappa = Rth / tth;
    o->ctau = Ra / (ktau * ktau);
    o->cv = 1.0 / Rh;
}

// joints [first, first + N) of the host model as a stand-alone parameter block
template <int N>
static void fill_static(const HostModel &h, StaticParams<N> &p, int first = 0)
{
    for (int i = 0; i < N; ++i) {
        const int g = first + i;
        std::memcpy(p.Rp[i], &h.Rp[9 * g], 9 * sizeof(double));
        std::memcpy(p.pp[i], &h.pp[3 * g], 3 * sizeof(double));
        p.mass[i] = h.mass[g];
        std::memcpy(p.mc[i], &h.mc[3 * g], 3 * sizeof(double));
        std::memcpy(p.Io[i], &h.Io[6 * g], 6 * sizeof(double));
        p.arm[i] = h.arm[g];
        std::memcpy(p.fat[i], &h.fat[4 * g], 4 * sizeof(double));
    }
    std::memcpy(p.grav, h.grav, sizeof p.grav);
    p.fence0 = 0;
}

static bool is_forest(const HostModel &h, int L)
{
    if (h.n % L) return false;
    for (int i = 0; i < h.n; ++i) {
        if (h.jtype[i] != 0) return false;
        if (h.parent[i] != ((i % L == 0) ? -1 : i - 1)) return false;
    }
    return true;
}

static void refresh(mpcf_model *m)
{
    const HostModel &h = m->h;
    if (h.n == 3 && is_forest(h, 3)) { m->fam = FAM_CHAIN3; fill_static(h, m->sp3); }
    else if (h.n == 6 && is_forest(h, 6)) { m->fam = FAM_CHAIN6; fill_static(h, m->sp6); }
    else if (h.n == 12 && is_forest(h, 6)) {
        m->fam = FAM_FOREST12x6;
        fill_static(h, m->sp12);
        for (int c = 0; c < 2; ++c) fill_static(h, m->chain6[c], 6 * c);
    }
    else if (h.n == 7 && is_forest(h, 7)) { m->fam = FAM_CHAIN7; fill_static(h, m->sp7); }
    else if (h.n == 14 && is_forest(h, 7)) {
        m->fam = FAM_FOREST14x7;
        fill_static(h, m->sp14);
        for (int c = 0; c < 2; ++c) fill_static(h, m->chain7[c], 7 * c);
    }
    else m->fam = h.n <= 16 ? FAM_GENERIC16 : FAM_GENERIC64;
    {
        std::vector<int> depth(h.n, 0);
        m->npat = 0;
        for (int j = 0; j < h.n; ++j) {
            depth[j] = h.parent[j] < 0 ? 0 : depth[h.parent[j]] + 1;
            m->npat += depth[j] + 1;
        }
    }
    m->dirty = true;
    m->fd_status = 0;
}

static int finish_create(mpcf_model *m, int rc, const std::string &err, mpcf_model **out)
{
    if (rc != MPCF_OK) {
        delete m;
        return fail(rc, err);
    }
    refresh(m);
    *out = m;
    return MPCF_OK;
}

extern "C" int mpcf_model_create_from_urdf(const char *xml, size_t len, const mpcf_opts *opts, mpcf_model **out)
{
    if (!xml || !out) return fail(MPCF_EINVAL, "null argument");
    *out = nullptr;
    mpcf_opts o;
    if (opts) o = *opts; else mpcf_opts_default(&o);
    mpcf_model *m = new (std::nothrow) mpcf_model();
    if (!m) return fail(MPCF_EINVAL, "out of memory");
    std::string err;
    int rc;
    try { rc = parse_urdf(xml, len, o, m->h, err); }
    catch (const std::exception &e) { rc = MPCF_EPARSE; err = e.what(); }
    return finish_create(m, rc, err, out);
}

extern "C" int mpcf_model_create_synthetic(int kind, int ndof, unsigned long long seed, const mpcf_opts *opts, mpcf_model **out)
{
    if (!out) return fail(MPCF_EINVAL, "null argument");
    *out = nullptr;
    mpcf_opts o;
    if (opts) o = *opts; else mpcf_opts_default(&o);
    mpcf_model *m = new (std::nothrow) mpcf_model();
    if (!m) return fail(MPCF_EINVAL, "out of memory");
    std::string err;
    int rc;
    try { rc = make_synthetic(kind, ndof, seed, o, m->h, err); }
    catch (const std::exception &e) { rc = MPCF_EINVAL; err = e.what(); }
    return finish_create(m, rc, err, out);
}

extern "C" int mpcf_model_destroy(mpcf_model *m)
{
    if (!m) return MPCF_OK;
    if (m->d_dbl) cudaFree(m->d_dbl);
    if (m->d_int) cudaFree(m->d_int);
    delete m;
    return MPCF_OK;
}

extern "C" int mpcf_model_info(const mpcf_model *m, int *nq, int *nv, int *nbody, int *nframe)
{
    if (!m) return fail(MPCF_EINVAL, "null model");
    if (nq) *nq = m->h.n;
    if (nv) *nv = m->h.n;
    if (nbody) *nbody = m->h.n;
    if (nframe) *nframe = (int)m->h.fparent.size();
    return MPCF_OK;
}

extern "C" int mpcf_frame_id(const mpcf_model *m, const char *name)
{
    if (!m || !name) return fail(MPCF_EINVAL, "null argument");
    for (size_t i = 0; i < m->h.frame_names.size(); ++i)
        if (m->h.frame_names[i] == name) return (int)i;
    return fail(MPCF_EFRAME, std::string("unknown frame '") + name + "'");
}

extern "C" const char *mpcf_joint_name(const mpcf_model *m, int j)
{
    if (!m || j < 0 || j >= m->h.n) return nullptr;
    return m->h.joint_names[j].c_str();
}
extern "C" const char *mpcf_frame_name(const mpcf_model *m, int f)
{
    if (!m || f < 0 || f >= (int)m->h.frame_names.size()) return nullptr;
    return m->h.frame_names[f].c_str();
}
extern "C" const char *mpcf_model_kernel_family(const mpcf_model *m)
{
    if (!m) return nullptr;
    switch (m->fam) {
    case FAM_CHAIN3: return "chain3";
    case FAM_CHAIN6: return "chain6";
    case FAM_FOREST12x6: return "forest12x6";
    case FAM_CHAIN7: return "chain7";
    case FAM_FOREST14x7: return "forest14x7";
    case FAM_GENERIC16: return "generic16";
    default: return "generic64";
    }
}

extern "C" long mpcf_model_export(const mpcf_model *m, const char *field, void *out, size_t cap)
{
    if (!m || !field || !out) return fail(MPCF_EINVAL, "null argument");
    const HostModel &h = m->h;
    const void *src = nullptr;
    size_t bytes = 0;
    std::string f(field);
    auto dv = [&](const std::vector<double> &v) { src = v.data(); bytes = v.size() * sizeof(double); };
    auto iv = [&](const std::vector<int> &v) { src = v.data(); bytes = v.size() * sizeof(int); };
    if (f == "parent") iv(h.parent);
    else if (f == "jtype") iv(h.jtype);
    else if (f == "fparent") iv(h.fparent);
    else if (f == "jcontinuous") iv(h.jcontinuous);
    else if (f == "Rp") dv(h.Rp);
    else if (f == "pp") dv(h.pp);
    else if (f == "mass") dv(h.mass);
    else if (f == "mc") dv(h.mc);
    else if (f == "Io") dv(h.Io);
    else if (f == "arm") dv(h.arm);
    else if (f == "fat") dv(h.fat);
    else if (f == "fR") dv(h.fR);
    else if (f == "fp") dv(h.fp);
    else if (f == "q_lo") dv(h.q_lo);
    else if (f == "q_hi") dv(h.q_hi);
    else if (f == "v_max") dv(h.v_max);
    else if (f == "tau_max") dv(h.tau_max);
    else if (f == "grav") { src = h.grav; bytes = sizeof h.grav; }
    else return fail(MPCF_EINVAL, "unknown field '" + f + "'");
    if (bytes > cap) return fail(MPCF_EINVAL, "buffer too small for field '" + f + "'");
    std::memcpy(out, src, bytes);
    return (long)bytes;
}

extern "C" int mpcf_model_set_armature(mpcf_model *m, const double *arm)
{
    if (!m || !arm) return fail(MPCF_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(m->mu);
    for (int i = 0; i < m->h.n; ++i) m->h.arm[i] = arm[i];
    refresh(m);
    return MPCF_OK;
}
extern "C" int mpcf_model_set_fatigue(mpcf_model *m, const double *rows)
{
    if (!m || !rows) return fail(MPCF_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(m->mu);
    for (int i = 0; i < 4 * m->h.n; ++i) m->h.fat[i] = rows[i];
    refresh(m);
    return MPCF_OK;
}

extern "C" int mpcf_model_set_coupling(mpcf_model *m, const mpcf_coupling *c)
{
    if (!m) return fail(MPCF_EINVAL, "null model");
    std::lock_guard<std::mutex> lk(m->mu);
    if (!c) { m->couple = CoupleHost{}; return MPCF_OK; }
    const int L = family_chain_len(m->fam);
    if (family_chains(m->fam) != 2) return fail(MPCF_EINVAL, "coupled fatigue needs a two-arm model (kernel families forest12x6 / forest14x7)");
    if (!(c->weight >= 0.0)) return fail(MPCF_EINVAL, "box weight must be >= 0");
    CoupleHost ch;
    ch.on = true;
    ch.weight = c->weight;
    for (int a = 0; a < 2; ++a) {
        const int fr = c->ee_frame[a];
        if (fr < 0 || fr >= (int)m->h.fparent.size()) return fail(MPCF_EFRAME, "coupling: end-effector frame index out of range");
        const int j = m->h.fparent[fr];
        if (j < a * L || j >= (a + 1) * L) return fail(MPCF_EFRAME, "coupling: ee_frame[" + std::to_string(a) + "] is not carried by arm " + std::to_string(a));
        ch.ee_joint[a] = j - a * L;
        std::memcpy(ch.ee_p[a], &m->h.fp[3 * fr], 3 * sizeof(double));
    }
    m->couple = ch;
    return MPCF_OK;
}

// ---- launch plumbing ----
static int cuda_fail(cudaError_t e, const char *what)
{
    return fail(MPCF_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

static int get_launch_model(const mpcf_model *m, LaunchModel &lm)
{
    const HostModel &h = m->h;
    lm.fam = m->fam;
    lm.n = h.n;
    lm.static_params = nullptr;
    lm.chain_params = nullptr;
    lm.blob = GenericBlob{nullptr, nullptr, h.n};
    switch (m->fam) {
    case FAM_CHAIN3: lm.static_params = lm.chain_params = &m->sp3; return MPCF_OK;
    case FAM_CHAIN6: lm.static_params = lm.chain_params = &m->sp6; return MPCF_OK;
    case FAM_FOREST12x6: lm.static_params = &m->sp12; lm.chain_params = m->chain6; return MPCF_OK;
    case FAM_CHAIN7: lm.static_params = lm.chain_params = &m->sp7; return MPCF_OK;
    case FAM_FOREST14x7: lm.static_params = &m->sp14; lm.chain_params = m->chain7; return MPCF_OK;
    default: break;
    }
    std::lock_guard<std::mutex> lk(m->mu);
    int dev = 0;
    cudaGetDevice(&dev);
    if (!m->dirty && m->device != dev)
        return fail(MPCF_EINVAL, "model constants were uploaded to device " + std::to_string(m->device) + "; create one model handle per device");
    if (m->dirty) {
        const int n = h.n;
        std::vector<double> d;
        d.reserve(blob_doubles(n));
        auto app = [&](const std::vector<double> &v) { d.insert(d.end(), v.begin(), v.end()); };
        app(h.Rp); app(h.pp); app(h.mass); app(h.mc); app(h.Io); app(h.arm); app(h.fat);
        d.insert(d.end(), h.grav, h.grav + 3);
        std::vector<int> ii(h.parent);
        ii.insert(ii.end(), h.jtype.begin(), h.jtype.end());
        std::vector<int> keep(n, 0);  // link i's (v, a) are needed after link i + 1 has been visited
        for (int j = 0; j < n; ++j)
            if (h.parent[j] >= 0 && h.parent[j] != j - 1) keep[h.parent[j]] = 1;
        ii.insert(ii.end(), keep.begin(), keep.end());
        std::vector<int> depth(n, 0), rowptr(n + 1, 0);  // packed ancestor storage of the tree Jacobian pipeline
        for (int j = 0; j < n; ++j) depth[j] = h.parent[j] < 0 ? 0 : depth[h.parent[j]] + 1;
        for (int j = 0; j < n; ++j) rowptr[j + 1] = rowptr[j] + depth[j] + 1;
        ii.insert(ii.end(), depth.begin(), depth.end());
        ii.insert(ii.end(), rowptr.begin(), rowptr.end());
        cudaError_t e;
        // a setter re-dirtied an uploaded model: kernels queued on any stream may still read the old blob
        if (m->d_dbl && m->device == dev) cudaDeviceSynchronize();
        if (m->d_dbl && m->device != dev) {  // first use on another device: the old buffers belong to m->device
            return fail(MPCF_EINVAL, "model constants were uploaded to device " + std::to_string(m->device) + "; create one model handle per device");
        }
        if (!m->d_dbl && (e = cudaMalloc(&m->d_dbl, d.size() * sizeof(double))) != cudaSuccess) return cuda_fail(e, "cudaMalloc(model)");
        if (!m->d_int && (e = cudaMalloc(&m->d_int, ii.size() * sizeof(int))) != cudaSuccess) return cuda_fail(e, "cudaMalloc(model)");
        // synchronous copies: the model is immutable afterwards and may be used from any stream
        if ((e = cudaMemcpy(m->d_dbl, d.data(), d.size() * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess) return cuda_fail(e, "cudaMemcpy(model)");
        if ((e = cudaMemcpy(m->d_int, ii.data(), ii.size() * sizeof(int), cudaMemcpyHostToDevice)) != cudaSuccess) return cuda_fail(e, "cudaMemcpy(model)");
        m->dirty = false;
        m->device = dev;
    }
    lm.blob.dbl = m->d_dbl;
    lm.blob.ints = m->d_int;
    return MPCF_OK;
}

// Forward dynamics needs D_i = S_i^T IA_i S_i + armature_i > 0.  The articulated inertia IA_i is bounded ABOVE by the
// composite rigid inertia of the subtree (IA_i <= Ic_i), so a zero composite inertia about a joint axis at q = 0 is a
// sufficient reason to refuse (the shipped Pilz flange: mass at the joint origin, zero tensor), not a guarantee that every
// configuration is regular: the kernels themselves turn a non-positive pivot into NaN outputs (dyn.cuh: fd_crba / aba).
static int check_forward_dynamics(const mpcf_model *cm)
{
    mpcf_model *m = const_cast<mpcf_model *>(cm);
    std::lock_guard<std::mutex> lk(m->mu);
    if (m->fd_status == 0) {
        const HostModel &h = m->h;
        const int n = h.n;
        std::vector<double> cm_(n), cmc(3 * n), cI(9 * n);
        for (int i = 0; i < n; ++i) {
            cm_[i] = h.mass[i];
            for (int k = 0; k < 3; ++k) cmc[3 * i + k] = h.mc[3 * i + k];
            const double *o = &h.Io[6 * i];
            double I[9] = {o[0], o[1], o[2], o[1], o[3], o[4], o[2], o[4], o[5]};
            std::memcpy(&cI[9 * i], I, sizeof I);
        }
        int status = 1;
        for (int i = n - 1; i >= 0; --i) {
            const double D = (h.jtype[i] == 0 ? cI[9 * i + 8] : cm_[i]) + h.arm[i];
            if (!(D > 0.0)) status = -1;
            const int p = h.parent[i];
            if (p < 0) continue;
            const double *R = &h.Rp[9 * i], *t = &h.pp[3 * i];
            double a[3], RI[9], RIRt[9];
            for (int r = 0; r < 3; ++r) a[r] = R[3 * r] * cmc[3 * i] + R[3 * r + 1] * cmc[3 * i + 1] + R[3 * r + 2] * cmc[3 * i + 2];
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) RI[3 * r + c] = R[3 * r] * cI[9 * i + c] + R[3 * r + 1] * cI[9 * i + 3 + c] + R[3 * r + 2] * cI[9 * i + 6 + c];
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) RIRt[3 * r + c] = RI[3 * r] * R[3 * c] + RI[3 * r + 1] * R[3 * c + 1] + RI[3 * r + 2] * R[3 * c + 2];
            const double ap = a[0] * t[0] + a[1] * t[1] + a[2] * t[2], tt = t[0] * t[0] + t[1] * t[1] + t[2] * t[2];
            const double dg = 2 * ap + cm_[i] * tt;
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c)
                    cI[9 * p + 3 * r + c] += RIRt[3 * r + c] - (a[r] * t[c] + t[r] * a[c] + cm_[i] * t[r] * t[c]) + (r == c ? dg : 0.0);
            for (int k = 0; k < 3; ++k) cmc[3 * p + k] += a[k] + cm_[i] * t[k];
            cm_[p] += cm_[i];
        }
        m->fd_status = status;
    }
    if (m->fd_status < 0)
        return fail(MPCF_ESINGULAR, "forward dynamics is singular: a joint has zero articulated inertia about its axis; set an armature");
    return MPCF_OK;
}

#define PROLOGUE(cond_args)                                              \
    if (!model) return fail(MPCF_EINVAL, "null model");                  \
    if (U < 0) return fail(MPCF_EINVAL, "negative batch size");          \
    if (U > 0 && !(cond_args)) return fail(MPCF_EINVAL, "null array argument"); \
    LaunchModel lm;                                                      \
    if (int rc = get_launch_model(model, lm)) return rc;                 \
    cudaStream_t st = static_cast<cudaStream_t>(stream);

static int frame_arg(const mpcf_model *m, int frame, FrameArg &fa)
{
    const HostModel &h = m->h;
    if (frame < 0 || frame >= (int)h.fparent.size()) return fail(MPCF_EFRAME, "frame index out of range");
    fa.joint = h.fparent[frame];
    std::memcpy(fa.R, &h.fR[9 * frame], sizeof fa.R);
    std::memcpy(fa.p, &h.fp[3 * frame], sizeof fa.p);
    return MPCF_OK;
}

static int done(cudaError_t e, const char *what) { return e == cudaSuccess ? MPCF_OK : cuda_fail(e, what); }

extern "C" int mpcf_rnea_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *qdd, double *tau,
                               void *stream)
{
    PROLOGUE(q && qd && tau)
    return done(launch_rnea(lm, U, q, qd, qdd, tau, st), "rnea_batch");
}

extern "C" int mpcf_fk_batch(const mpcf_model *model, int frame, long U, const double *q, double *pos, double *rot, void *stream)
{
    PROLOGUE(q && pos && rot)
    FrameArg fa;
    if (int rc = frame_arg(model, frame, fa)) return rc;
    return done(launch_fk(lm, fa, U, q, pos, rot, st), "fk_batch");
}

extern "C" int mpcf_frame_jac_batch(const mpcf_model *model, int frame, long U, const double *q, double *J, void *stream)
{
    PROLOGUE(q && J)
    FrameArg fa;
    if (int rc = frame_arg(model, frame, fa)) return rc;
    return done(launch_jac(lm, fa, U, q, J, st), "frame_jac_batch");
}

extern "C" int mpcf_frame_jac_t_wrench_batch(const mpcf_model *model, int frame, long U, const double *q, const double *W,
                                             double *out, void *stream)
{
    PROLOGUE(q && W && out)
    EeArgs ee;
    ee.nee = 1;
    if (int rc = frame_arg(model, frame, ee.f[0])) return rc;
    ZohArg zoh{};
    return done(launch_node_eval(lm, ee, 1.0, U, q, nullptr, nullptr, W, nullptr, 0.0, zoh, out, nullptr, nullptr, true, st),
                "frame_jac_t_wrench_batch");
}

extern "C" int mpcf_node_eval_ref_batch(const mpcf_model *model, int nee, const int *ee_frames, double wsign, long U, const double *q,
                                        const double *qd, const double *qdd, const double *W, const double *T, double h,
                                        double *tau, double *qnext, double *Tnext, void *stream)
{
    PROLOGUE(q && qd && tau)
    if (nee < 0 || nee > MPCF_MAX_EE) return fail(MPCF_EINVAL, "nee out of range (0..MPCF_MAX_EE)");
    if (nee > 0 && (!ee_frames || (U > 0 && !W))) return fail(MPCF_EINVAL, "end-effector frames / wrenches missing");
    if (Tnext && !T && U > 0) return fail(MPCF_EINVAL, "Tnext requested without T");
    EeArgs ee;
    ee.nee = nee;
    for (int e = 0; e < nee; ++e)
        if (int rc = frame_arg(model, ee_frames[e], ee.f[e])) return rc;
    ZohArg zoh{};
    for (int i = 0; i < model->h.n; ++i) zoh.a[i] = std::exp(-model->h.fat[4 * i] * h);
    return done(launch_node_eval(lm, ee, wsign, U, q, qd, qdd, W, T, h, zoh, tau, qnext, Tnext, false, st), "node_eval_ref_batch");
}

extern "C" int mpcf_node_eval_ref_jvp_batch(const mpcf_model *model, int nee, const int *ee_frames, double wsign, long U, const double *q,
                                            const double *qd, const double *qdd, const double *W, double *dtau_dq, double *dtau_dqd,
                                            void *stream)
{
    PROLOGUE(q && qd && dtau_dq && dtau_dqd)
    if (nee < 0 || nee > MPCF_MAX_EE) return fail(MPCF_EINVAL, "nee out of range (0..MPCF_MAX_EE)");
    if (nee > 0 && (!ee_frames || (U > 0 && !W))) return fail(MPCF_EINVAL, "end-effector frames / wrenches missing");
    EeArgs ee;
    ee.nee = nee;
    for (int e = 0; e < nee; ++e)
        if (int rc = frame_arg(model, ee_frames[e], ee.f[e])) return rc;
    return done(launch_node_eval_jvp(lm, ee, wsign, U, q, qd, qdd, W, dtau_dq, dtau_dqd, st), "node_eval_ref_jvp_batch");
}

extern "C" int mpcf_aba_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau, double *qdd,
                              void *stream)
{
    PROLOGUE(q && qd && tau && qdd)
    if (int rc = check_forward_dynamics(model)) return rc;
    return done(launch_aba(lm, U, q, qd, tau, qdd, st), "aba_batch");
}

extern "C" int mpcf_step_rk4_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                                   const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn, void *stream)
{
    PROLOGUE(q && qd && tau && f && qn && qdn && fn)
    if (int rc = check_forward_dynamics(model)) return rc;
    if (!model->couple.on || U == 0) return done(launch_step(lm, U, q, qd, tau, f, dt, dt_u, qn, qdn, fn, st), "step_rk4_batch");
    // coupled fatigue: heating torque from a pre-kernel into stream-ordered scratch (no synchronisation)
    double *theat = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&theat), (size_t)model->h.n * U * sizeof(double), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMallocAsync(heating torque)");
    e = launch_couple(lm, model->couple, U, U, q, f, tau, theat, U, 0, dt, dt_u, nullptr, 0, st);
    if (e == cudaSuccess) e = launch_step(lm, U, q, qd, tau, f, dt, dt_u, qn, qdn, fn, st, theat);
    const cudaError_t e2 = cudaFreeAsync(theat, st);
    return done(e != cudaSuccess ? e : e2, "step_rk4_batch (coupled)");
}

extern "C" int mpcf_rollout_rk4_batch(const mpcf_model *model, long B, int N, const double *q0, const double *qd0, const double *f0,
                                      const double *tau, double dt, double *qt, double *qdt, double *ft, void *stream)
{
    const long U = B;
    PROLOGUE(q0 && qd0 && f0 && tau && qt && qdt && ft)
    if (N <= 0) return fail(MPCF_EINVAL, "N must be positive");
    if (model->couple.on) return fail(MPCF_EINVAL, "the rollout entry does not support coupled fatigue: use mpcf_step_rk4_batch per step");
    if (int rc = check_forward_dynamics(model)) return rc;
    return done(launch_rollout(lm, B, N, q0, qd0, f0, tau, dt, qt, qdt, ft, st), "rollout_rk4_batch");
}

// Workspace of the analytic Jacobian pipeline: (16 n + 12 n^2) doubles per unit, processed in chunks of at most
// 2^20 units, so the request is bounded (4.4 GB for n = 6) however large U is.
static const long kJvpChunkUnits = 1L << 20;
extern "C" size_t mpcf_step_rk4_jvp_workspace_bytes(const mpcf_model *model, long U)
{
    if (!model || U <= 0) return 0;
    LaunchModel lm;
    lm.fam = model->fam;
    lm.n = model->h.n;
    if (tree_jvp_supported(lm)) return tree_jvp_workspace_bytes(model->h.n, model->npat, U);
    if (!jvp2_supported(lm)) return 0;
    long units = U < kJvpChunkUnits ? U : kJvpChunkUnits;
    units = (units + 31) / 32 * 32;
    return (size_t)units * jvp_ws_bytes_per_unit(lm);
}

// The step-derivative entries' workspace: the caller's, checked (128-byte aligned, at least one 32-unit tile), or one from the
// device's stream-ordered memory pool sized for U units (no synchronisation; the pool keeps the block after the first call, so
// steady-state calls cost two pool look-ups).  *owned: the caller frees it with cudaFreeAsync.  Models without a workspace
// pipeline need none.
static int get_workspace(const mpcf_model *model, const LaunchModel &lm, long U, void *workspace, size_t workspace_bytes, cudaStream_t st,
                         const char *alloc_what, double **ws, size_t *bytes, bool *owned)
{
    *ws = nullptr; *bytes = 0; *owned = false;
    const bool tree = tree_jvp_supported(lm);
    if (!tree && !jvp2_supported(lm)) return MPCF_OK;
    if (workspace) {
        const size_t min_ws = tree ? tree_jvp_workspace_bytes(model->h.n, model->npat, 32) : 32 * jvp_ws_bytes_per_unit(lm);
        // the chain-rule kernel streams the workspace with cp.async.bulk: 16-byte aligned global addresses; chunk offsets
        // are multiples of 256 B, so the base decides.  128 keeps every plane on a full cache line.
        if (reinterpret_cast<uintptr_t>(workspace) % 128) return fail(MPCF_EINVAL, "workspace must be 128-byte aligned");
        if (workspace_bytes < min_ws) return fail(MPCF_EINVAL, "workspace too small: see mpcf_step_rk4_jvp_workspace_bytes");
        *ws = static_cast<double *>(workspace);
        *bytes = workspace_bytes;
        return MPCF_OK;
    }
    *bytes = mpcf_step_rk4_jvp_workspace_bytes(model, U);
    const cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(ws), *bytes, st);
    if (e != cudaSuccess) return cuda_fail(e, alloc_what);
    *owned = true;
    return MPCF_OK;
}

// analytic pipeline on `cnt` units (plane strides ld / ld_jac), with the coupled-fatigue pre / post kernels around it when the
// model has a coupling (heating torque in stream-ordered scratch: no synchronisation)
static cudaError_t run_pipeline(const mpcf_model *model, const LaunchModel &lm, long cnt, long ld, const double *q, const double *qd,
                                const double *tau, const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn,
                                double *jac, long ld_jac, double *ws, size_t ws_bytes, cudaStream_t st)
{
    if (tree_jvp_supported(lm))
        return launch_step_jvp_tree(lm, model->npat, ld, cnt, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, ld_jac, ws, ws_bytes, st);
    if (!model->couple.on) return launch_step_jvp_ws(lm, ld, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, ws, ws_bytes, st, cnt, ld_jac);
    double *theat = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&theat), (size_t)model->h.n * cnt * sizeof(double), st);
    if (e != cudaSuccess) return e;
    e = launch_couple(lm, model->couple, cnt, ld, q, f, tau, theat, cnt, 0, dt, dt_u, nullptr, 0, st);
    if (e == cudaSuccess) e = launch_step_jvp_ws(lm, ld, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, ws, ws_bytes, st, cnt, ld_jac, theat, cnt);
    if (e == cudaSuccess) e = launch_couple(lm, model->couple, cnt, ld, q, f, tau, theat, cnt, 1, dt, dt_u, jac, ld_jac, st);
    const cudaError_t e2 = cudaFreeAsync(theat, st);
    return e != cudaSuccess ? e : e2;
}

// the dual-number sweep kernel (3n + 1 seeds): every family; the cross-check of the analytic pipeline and the path of the
// run-time-topology families
extern "C" int mpcf_step_rk4_jvp_dual_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                                            const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn,
                                            double *jac, void *stream)
{
    PROLOGUE(q && qd && tau && f && jac)
    if ((qn || qdn || fn) && !(qn && qdn && fn)) return fail(MPCF_EINVAL, "qn/qdn/fn must be all set or all NULL");
    if (int rc = check_forward_dynamics(model)) return rc;
    if (model->couple.on) return fail(MPCF_EINVAL, "the dual-number entry does not support coupled fatigue");
    return done(launch_step_jvp(lm, U, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, st), "step_rk4_jvp_dual_batch");
}

extern "C" int mpcf_step_rk4_jvp_ws_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                                          const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn,
                                          double *jac, void *workspace, size_t workspace_bytes, void *stream)
{
    PROLOGUE(q && qd && tau && f && jac)
    if ((qn || qdn || fn) && !(qn && qdn && fn)) return fail(MPCF_EINVAL, "qn/qdn/fn must be all set or all NULL");
    if (int rc = check_forward_dynamics(model)) return rc;
    if (!jvp2_supported(lm) && !tree_jvp_supported(lm))  // run-time topology with n > 40: no workspace pipeline; the workspace argument is ignored
        return done(launch_step_jvp(lm, U, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, st), "step_rk4_jvp_batch");
    if (U == 0) return MPCF_OK;
    double *ws;
    size_t bytes;
    bool owned;
    if (int rc = get_workspace(model, lm, U, workspace, workspace_bytes, st, "cudaMallocAsync(jvp workspace)", &ws, &bytes, &owned)) return rc;
    const cudaError_t e = run_pipeline(model, lm, U, U, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, U, ws, bytes, st);
    const cudaError_t e2 = owned ? cudaFreeAsync(ws, st) : cudaSuccess;
    return done(e != cudaSuccess ? e : e2, owned ? "step_rk4_jvp_batch" : "step_rk4_jvp_ws_batch");
}

// Unit-range form: `cnt` units whose input / state planes have stride `ld` (base pointers already shifted to the range) and a
// Jacobian buffer with plane stride `ld_jac` (>= cnt): lets a caller sweep a batch much larger than the Jacobian it can
// hold by reusing one chunk-sized Jacobian buffer (config C5: 1,048,576 scenarios x 100 nodes on one GPU).
extern "C" int mpcf_step_rk4_jvp_strided_batch(const mpcf_model *model, long cnt, long ld, const double *q, const double *qd,
                                               const double *tau, const double *f, double dt, const double *dt_u, double *qn,
                                               double *qdn, double *fn, double *jac, long ld_jac, void *workspace,
                                               size_t workspace_bytes, void *stream)
{
    const long U = cnt;
    PROLOGUE(q && qd && tau && f && jac)
    if (ld < cnt || ld_jac < cnt) return fail(MPCF_EINVAL, "plane strides must be >= cnt");
    if ((qn || qdn || fn) && !(qn && qdn && fn)) return fail(MPCF_EINVAL, "qn/qdn/fn must be all set or all NULL");
    if (int rc = check_forward_dynamics(model)) return rc;
    if (cnt == 0) return MPCF_OK;
    if (!jvp2_supported(lm) && !tree_jvp_supported(lm))
        return done(launch_step_jvp(lm, ld, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, st, cnt, ld_jac), "step_rk4_jvp_strided_batch");
    if (!workspace) return fail(MPCF_EINVAL, "the strided entry needs a caller workspace (mpcf_step_rk4_jvp_workspace_bytes)");
    double *ws;
    size_t bytes;
    bool owned;  // false: the caller's workspace is never replaced
    if (int rc = get_workspace(model, lm, cnt, workspace, workspace_bytes, st, "cudaMallocAsync(jvp workspace)", &ws, &bytes, &owned)) return rc;
    return done(run_pipeline(model, lm, cnt, ld, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, ld_jac, ws, bytes, st), "step_rk4_jvp_strided_batch");
}

extern "C" int mpcf_step_rk4_jvp_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                                       const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn,
                                       double *jac, void *stream)
{
    return mpcf_step_rk4_jvp_ws_batch(model, U, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, nullptr, 0, stream);
}

// ---- reverse mode ----
// step VJP on `cnt` units whose state / torque planes have stride `ld` (the adjoint, addend and output strides travel in `a`)
static cudaError_t run_vjp(const mpcf_model *model, const LaunchModel &lm, long cnt, long ld, const double *q, const double *qd, const double *tau,
                           const double *f, double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn, double *ws,
                           size_t ws_bytes, cudaStream_t st)
{
    if (tree_jvp_supported(lm)) return launch_step_vjp_tree(lm, model->npat, ld, cnt, q, qd, tau, f, dt, dt_u, a, qn, qdn, fn, ws, ws_bytes, st);
    if (jvp2_supported(lm)) return launch_step_vjp_ws(lm, ld, cnt, q, qd, tau, f, dt, dt_u, a, qn, qdn, fn, ws, ws_bytes, st);
    return launch_step_vjp_dual(lm, ld, cnt, q, qd, tau, f, dt, dt_u, a, qn, qdn, fn, st);
}

extern "C" int mpcf_step_rk4_vjp_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau, const double *f,
                                       double dt, const double *dt_u, const double *lq, const double *lqd, const double *lf, double *gq,
                                       double *gqd, double *gtau, double *gf, double *gdt, double *qn, double *qdn, double *fn, void *workspace,
                                       size_t workspace_bytes, void *stream)
{
    PROLOGUE(q && qd && tau && f && gq && gqd && gtau && gf)
    if ((qn || qdn || fn) && !(qn && qdn && fn)) return fail(MPCF_EINVAL, "qn/qdn/fn must be all set or all NULL");
    if (model->couple.on) return fail(MPCF_EINVAL, "the reverse-mode entries do not support coupled fatigue");
    if (int rc = check_forward_dynamics(model)) return rc;
    if (U == 0) return MPCF_OK;
    VjpArgs a;
    a.lq = lq; a.lqd = lqd; a.lf = lf; a.ldl = U;
    a.lda = U;
    a.gq = gq; a.gqd = gqd; a.gf = gf; a.ldg = U;
    a.gtau = gtau; a.ldgt = U;
    a.gdt = gdt;
    double *ws;
    size_t bytes;
    bool owned;
    if (int rc = get_workspace(model, lm, U, workspace, workspace_bytes, st, "cudaMallocAsync(vjp workspace)", &ws, &bytes, &owned)) return rc;
    const cudaError_t e = run_vjp(model, lm, U, U, q, qd, tau, f, dt, dt_u, a, qn, qdn, fn, ws, bytes, st);
    const cudaError_t e2 = owned ? cudaFreeAsync(ws, st) : cudaSuccess;
    return done(e != cudaSuccess ? e : e2, "step_rk4_vjp_batch");
}

// Adjoint of the rollout: one step VJP per node, k = N-1 .. 0, on the node's B contiguous units (plane stride N B).  lambda_k =
// g_x(lambda_{k+1}) + dL/dx_k alternates between the g*0 outputs and an O(B) scratch buffer, so that node 0 writes dL/dx_0 into
// the outputs; the step at node 0 reads x_0 (stride B) and a stride-B copy of tau's node-0 columns.
extern "C" int mpcf_rollout_rk4_vjp_batch(const mpcf_model *model, long B, int N, const double *q0, const double *qd0, const double *f0,
                                          const double *tau, double dt, const double *qt, const double *qdt, const double *ft, const double *gqt,
                                          const double *gqdt, const double *gft, double *gtau, double *gq0, double *gqd0, double *gf0,
                                          void *workspace, size_t workspace_bytes, void *stream)
{
    const long U = B;
    PROLOGUE(q0 && qd0 && f0 && tau && qt && qdt && ft && gtau && gq0 && gqd0 && gf0)
    if (N <= 0) return fail(MPCF_EINVAL, "N must be positive");
    if (model->couple.on) return fail(MPCF_EINVAL, "the reverse-mode entries do not support coupled fatigue");
    if (int rc = check_forward_dynamics(model)) return rc;
    if (B == 0) return MPCF_OK;
    const int n = model->h.n;
    const long NB = (long)N * B;
    double *ws;
    size_t bytes;
    bool owned;
    if (int rc = get_workspace(model, lm, B, workspace, workspace_bytes, st, "cudaMallocAsync(vjp workspace)", &ws, &bytes, &owned)) return rc;
    double *scr = nullptr;  // [3n][B] adjoint of the odd nodes | [n][B] tau of node 0
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&scr), (size_t)4 * n * B * sizeof(double), st);
    if (e != cudaSuccess) {
        if (owned) cudaFreeAsync(ws, st);
        return cuda_fail(e, "cudaMallocAsync(rollout adjoint scratch)");
    }
    double *tau0 = scr + (size_t)3 * n * B;
    if (N > 1) e = cudaMemcpy2DAsync(tau0, B * sizeof(double), tau, NB * sizeof(double), B * sizeof(double), n, cudaMemcpyDeviceToDevice, st);
    auto sh = [](const double *p, long off) { return p ? p + off : p; };
    for (int k = N - 1; k >= 0 && e == cudaSuccess; --k) {
        VjpArgs a;
        if (k == N - 1) {  // lambda_N = dL/dx_N = trajectory entry N - 1
            a.lq = sh(gqt, (long)k * B); a.lqd = sh(gqdt, (long)k * B); a.lf = sh(gft, (long)k * B); a.ldl = NB;
        } else {
            const bool even = (k + 1) % 2 == 0;
            a.lq = even ? gq0 : scr; a.lqd = even ? gqd0 : scr + (size_t)n * B; a.lf = even ? gf0 : scr + (size_t)2 * n * B; a.ldl = B;
        }
        if (k > 0) { a.aq = sh(gqt, (long)(k - 1) * B); a.aqd = sh(gqdt, (long)(k - 1) * B); a.af = sh(gft, (long)(k - 1) * B); }
        a.lda = NB;
        const bool even = k % 2 == 0;
        a.gq = even ? gq0 : scr; a.gqd = even ? gqd0 : scr + (size_t)n * B; a.gf = even ? gf0 : scr + (size_t)2 * n * B; a.ldg = B;
        a.gtau = gtau + (long)k * B; a.ldgt = NB;
        if (k == 0)
            e = run_vjp(model, lm, B, B, q0, qd0, N > 1 ? tau0 : tau, f0, dt, nullptr, a, nullptr, nullptr, nullptr, ws, bytes, st);
        else {
            const long off = (long)(k - 1) * B;
            e = run_vjp(model, lm, B, NB, qt + off, qdt + off, tau + (long)k * B, ft + off, dt, nullptr, a, nullptr, nullptr, nullptr, ws, bytes, st);
        }
    }
    cudaError_t e2 = cudaFreeAsync(scr, st);
    if (owned) {
        const cudaError_t e3 = cudaFreeAsync(ws, st);
        if (e2 == cudaSuccess) e2 = e3;
    }
    return done(e != cudaSuccess ? e : e2, "rollout_rk4_vjp_batch");
}

// ---- second order ----
extern "C" int mpcf_step_rk4_hess_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                                        const double *f, double dt, const double *dt_u, const double *lq, const double *lqd,
                                        const double *lf, double *H, void *stream)
{
    PROLOGUE(q && qd && tau && f && H)
    if (model->couple.on) return fail(MPCF_EINVAL, "the second-order entries do not support coupled fatigue");
    if (int rc = check_forward_dynamics(model)) return rc;
    HessArgs h;
    h.lq = lq; h.lqd = lqd; h.lf = lf;
    h.H = H;
    return done(launch_step_hess(lm, U, q, qd, tau, f, dt, dt_u, h, st), "step_rk4_hess_batch");
}

extern "C" int mpcf_step_rk4_hvp_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                                       const double *f, double dt, const double *dt_u, const double *lq, const double *lqd,
                                       const double *lf, const double *vq, const double *vqd, const double *vtau, const double *vf,
                                       const double *vdt, double *hq, double *hqd, double *htau, double *hf, double *hdt,
                                       double *jq, double *jqd, double *jf, void *stream)
{
    PROLOGUE(q && qd && tau && f && hq && hqd && htau && hf)
    if ((jq || jqd || jf) && !(jq && jqd && jf)) return fail(MPCF_EINVAL, "jq/jqd/jf must be all set or all NULL");
    if (model->couple.on) return fail(MPCF_EINVAL, "the second-order entries do not support coupled fatigue");
    if (int rc = check_forward_dynamics(model)) return rc;
    HessArgs h;
    h.lq = lq; h.lqd = lqd; h.lf = lf;
    h.vq = vq; h.vqd = vqd; h.vtau = vtau; h.vf = vf; h.vdt = vdt;
    h.hq = hq; h.hqd = hqd; h.htau = htau; h.hf = hf; h.hdt = hdt;
    h.jq = jq; h.jqd = jqd; h.jf = jf;
    return done(launch_step_hvp(lm, U, q, qd, tau, f, dt, dt_u, h, st), "step_rk4_hvp_batch");
}

extern "C" int mpcf_fd_derivs_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau, double *A,
                                    double *B, double *C, void *stream)
{
    PROLOGUE(q && qd && tau && A && B && C)
    if (int rc = check_forward_dynamics(model)) return rc;
    return done(launch_fd_derivs(lm, U, q, qd, tau, A, B, C, st), "fd_derivs_batch");
}

extern "C" int mpcf_rnea_derivs_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *qdd, double *dtau_dq,
                                      double *dtau_dqd, double *M, void *stream)
{
    PROLOGUE(q && qd && dtau_dq && dtau_dqd && M)
    return done(launch_rnea_derivs(lm, U, q, qd, qdd, dtau_dq, dtau_dqd, M, st), "rnea_derivs_batch");
}

extern "C" int mpcf_cost_residual_batch(const mpcf_model *model, long B, int N, const double *q, const double *qd, const double *f,
                                        const double *tau, const double *qn, const double *qdn, const double *fn, double dt,
                                        double w_qd, double w_tau, double tau0, double alpha, double tau_floor, double f_max,
                                        double *out, void *stream)
{
    if (!model) return fail(MPCF_EINVAL, "null model");
    if (B < 0 || N <= 0) return fail(MPCF_EINVAL, "bad B / N");
    if (B > 0 && !(q && qd && f && tau && qn && qdn && fn && out)) return fail(MPCF_EINVAL, "null array argument");
    CostArgs c{dt, w_qd, w_tau, tau0, alpha, tau_floor, f_max};
    return done(launch_cost_residual(model->h.n, B, N, q, qd, f, tau, qn, qdn, fn, c, out, static_cast<cudaStream_t>(stream)),
                "cost_residual_batch");
}

extern "C" int mpcf_cost_residual_table_batch(const mpcf_model *model, long B, int N, const double *q, const double *qd, const double *f,
                                              const double *tau, const double *qn, const double *qdn, const double *fn, double w_qd,
                                              double w_tau, const double *bound_table, double f_max, double *out, long ld_out,
                                              void *stream)
{
    if (!model) return fail(MPCF_EINVAL, "null model");
    if (B < 0 || N <= 0) return fail(MPCF_EINVAL, "bad B / N");
    if (ld_out <= 0) ld_out = B;
    if (ld_out < B) return fail(MPCF_EINVAL, "ld_out must be >= B");
    if (B > 0 && !(q && qd && f && tau && qn && qdn && fn && out && bound_table)) return fail(MPCF_EINVAL, "null array argument");
    if ((size_t)2 * model->h.n * N * sizeof(double) > 200 * 1024) return fail(MPCF_ELIMIT, "bound table exceeds 200 KB of shared memory (2 n N doubles)");
    return done(launch_cost_residual_table(model->h.n, B, N, q, qd, f, tau, qn, qdn, fn, w_qd, w_tau, f_max, bound_table, out, ld_out,
                                           static_cast<cudaStream_t>(stream)),
                "cost_residual_table_batch");
}

extern "C" int mpcf_ocp_rows_count(const mpcf_model *model)
{
    if (!model) return fail(MPCF_EINVAL, "null model");
    const int arms = family_chains(model->fam);
    if (arms == 0) return fail(MPCF_EINVAL, "the fused OCP rows need a compile-time family (chain3/6/7: one arm, forest12x6/14x7: two arms)");
    return (arms == 2 ? 26 : 3) + 3 * model->h.n;
}

extern "C" int mpcf_ocp_rows_count_arms(const mpcf_model *model, int narm)
{
    if (!model) return fail(MPCF_EINVAL, "null model");
    if (narm != 1 && narm != 2) return fail(MPCF_EINVAL, "ocp rows: narm must be 1 or 2");
    const int arms = family_chains(model->fam);
    if (arms != 0 && narm != arms)
        return fail(MPCF_EINVAL, "ocp rows: this compile-time family has " + std::to_string(arms) + " arm(s), not " + std::to_string(narm));
    return (narm == 2 ? 26 : 3) + 3 * model->h.n;
}

extern "C" int mpcf_ocp_rows_batch(const mpcf_model *model, const mpcf_rows_opts *o, long B, int N, const double *q, const double *qd,
                                   const double *F, const double *T, const double *q_last, const double *T_last, const double *rel_pos0,
                                   const double *rel_ori0, double *rows, double *cost, double *dtau_dF, double *dT_dtau, double *kin_jac,
                                   void *stream)
{
    const long U = B * (long)N;
    PROLOGUE(q && qd && F && rows && cost)
    if (!o || B < 0 || N <= 0) return fail(MPCF_EINVAL, "bad options / B / N");
    const int arms = family_chains(model->fam), L = family_chain_len(model->fam);
    // run-time trees: one arm when ee_frame[1] < 0, two otherwise; the frames may sit anywhere in the tree (shared ancestors,
    // world-fixed).  Compile-time families: the arm count and the arm carrying each frame are fixed by the family.
    const bool tree = arms == 0;
    RowsHost h;
    h.narm = tree ? (o->ee_frame[1] < 0 ? 1 : 2) : arms;
    h.N = N; h.B = B;
    for (int a = 0; a < h.narm; ++a) {
        const int fr = o->ee_frame[a];
        if (fr < 0 || fr >= (int)model->h.fparent.size()) return fail(MPCF_EFRAME, "ocp rows: end-effector frame index out of range");
        const int j = model->h.fparent[fr];  // -1: world-fixed frame
        if (!tree && (j < a * L || j >= (a + 1) * L))
            return fail(MPCF_EFRAME, "ocp rows: ee_frame[" + std::to_string(a) + "] is not carried by arm " + std::to_string(a));
        h.ee_joint[a] = j;
        std::memcpy(h.ee_p[a], &model->h.fp[3 * fr], 3 * sizeof(double));
        std::memcpy(h.ee_R[a], &model->h.fR[9 * fr], 9 * sizeof(double));
    }
    h.wsign = o->wsign; h.dist2_ref = o->dist2_ref; h.mu = o->mu; h.w_box = o->w_box; h.w_qd = o->w_qd; h.w_F = o->w_F; h.h = o->h;
    std::memcpy(h.fdes, o->fdes, sizeof h.fdes);
    std::memcpy(h.p_ref, o->p_ref, sizeof h.p_ref);
    return done(launch_ocp_rows(lm, h, q, qd, F, T, q_last, T_last, rel_pos0, rel_ori0, rows, cost, dtau_dF, dT_dtau, kin_jac, st), "ocp_rows_batch");
}

extern "C" int mpcf_probe_fp64(long iters, int blocks, double *out, void *stream)
{
    if (iters <= 0 || blocks <= 0 || !out) return fail(MPCF_EINVAL, "bad probe arguments");
    return done(launch_fp64_probe(iters, blocks, out, static_cast<cudaStream_t>(stream)), "probe_fp64");
}

// Pitched host<->device copies for the host-facing pipeline (scenario-chunk slices of SoA planes).
// kind: 1 = host->device, 2 = device->host.  Host memory should be pinned for the copy to be asynchronous.
extern "C" int mpcf_memcpy2d_async(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width_bytes, size_t height,
                                   int kind, void *stream)
{
    if (!dst || !src) return fail(MPCF_EINVAL, "null pointer");
    if (kind != 1 && kind != 2) return fail(MPCF_EINVAL, "kind must be 1 (H2D) or 2 (D2H)");
    if (width_bytes == 0 || height == 0) return MPCF_OK;
    return done(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width_bytes, height,
                                  kind == 1 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)),
                "memcpy2d_async");
}

extern "C" int mpcf_gather_planes(const double *src, long ld_src, const int *plane_map, int nplanes, long U, double *dst, void *stream)
{
    if (nplanes < 0 || U < 0 || ld_src < U) return fail(MPCF_EINVAL, "bad sizes");
    if (nplanes > 0 && U > 0 && !(src && plane_map && dst)) return fail(MPCF_EINVAL, "null array argument");
    if (nplanes > 65535) return fail(MPCF_ELIMIT, "at most 65535 planes per call");
    if ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) % 16) return fail(MPCF_EINVAL, "src and dst must be 16-byte aligned");
    return done(launch_gather_planes(src, dst, plane_map, nplanes, U, ld_src, static_cast<cudaStream_t>(stream)), "gather_planes");
}

// Per-kernel timing of the analytic Jacobian pipeline (diagnostics for bench.py; not thread-safe, off by default).
extern "C" int mpcf_profile_enable(int on)
{
    jvp_profile_enable(on != 0);
    return MPCF_OK;
}
extern "C" int mpcf_profile_read(double *ms3, long *launches)
{
    if (!ms3 || !launches) return fail(MPCF_EINVAL, "null argument");
    return jvp_profile_read(ms3, launches);
}
