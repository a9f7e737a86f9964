// Batched, variable-size multi-site evaluation (dgp_batch_* of include/dgp.h): the B200 replacement of the reference's
// one-worker-per-site map (examples/nwqn-loadest-example/nwqn-loadest-example.py:156-157) for sites that share a model.
//
// Every launch of the single-site schedule (dgp_api.cu, DESIGN.md 4.5) covers ALL sites of the batch: the tile engine
// maps tile index -> (site, tile) through a per-launch prefix table passed by value (BatchTab), the diagonal-block
// kernel runs one CTA per site, the memory-bound helpers take the site from the grid.  Per-site arrays are slabs
// [site][ld][ld] / [site][ld] with one 3-D tensor map per matrix (site = third TMA coordinate).
//
// Sites of different size are END-ALIGNED: with NB = max nb and panels of pw block columns, site i starts at global block
// step off_i = floor((NB - nb_i) / pw) pw, so that at every global step all active sites have (almost) the same trailing
// matrix left, all finish together, and the latency-bound chain (diagonal block -> panel solve -> in-panel update) is paid
// once per global step for the whole batch instead of once per site.  Panels of a site still start at its local block 0, so
// every tile sees exactly the operations (and operand order) of the single-site schedule: results are bit-identical.
//
// Included at the end of dgp_api.cu (uses its launch helpers).
#pragma once

struct dgp_batch_s {
  int device = 0, sms = 148;
  cudaStream_t stream = nullptr, stream_hi = nullptr, stream_lo = nullptr, stream_t2 = nullptr;
  bool own_stream = false;
  cudaEvent_t ev_lo[2] = {nullptr, nullptr};
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> evs;
  bool timing = false;
  int max_sites = 0, max_pad = 0, max_n = 0;
  int G = 0, NB = 0;
  long long ld = 0;
  int n[DGP_BATCH_MAX] = {0}, nb[DGP_BATCH_MAX] = {0}, off[DGP_BATCH_MAX] = {0}, order[DGP_BATCH_MAX] = {0};
  bool have_train = false, pending = false;
  // have_T[s]: the last evaluation was a dgp_batch_factorize and site s factorised (info == 0): L^-1 in the lower triangle
  // of its A slab and alpha are what dgp_batch_predict reads.  Cleared by set_train and by every nlml_grad launch (LAUUM
  // overwrites T).
  bool have_T[DGP_BATCH_MAX] = {false};
  // have_eval[s]: the last evaluation (nlml_grad or factorize) finished and site s had info == 0: alpha and U = L^-T are
  // resident, which is what the mean-only prediction and dgp_batch_mean_functional_grad read.  Cleared by set_train and
  // by every launch.
  bool have_eval[DGP_BATCH_MAX] = {false};
  dgp_spec spec, user_spec;
  SiteDims sd;
  double *A = nullptr, *L = nullptr, *U = nullptr;
  double *X = nullptr, *y = nullptr, *noise = nullptr, *Xw = nullptr, *r = nullptr, *z = nullptr, *alpha = nullptr;
  double *theta = nullptr, *scal = nullptr, *gpart = nullptr, *zpart = nullptr, *jitv = nullptr;
  double *h_theta = nullptr, *h_scal = nullptr, *h_jit = nullptr;  // pinned
  CUtensorMap tmA, tmL, tmU;
  L8Work l8;   // residue buffers of the INT8 LAUUM (sites of L8_MIN_NPAD padded points or more, one site at a time)
  // prediction slabs (dgp_batch_predict), allocated by the first prediction on the handle and kept (chunk = DGP_BATCH_CHUNK):
  // Kx [max_sites][chunk][max_pad], mean / variance partials [max_sites][max_nb | 2 max_nb][chunk], inputs and features
  // [max_sites][chunk][8], means / mu / var [max_sites][chunk]; pinned staging of the inputs and of mu / var
  double *Kx = nullptr, *Xs = nullptr, *Xws = nullptr, *means = nullptr, *dot = nullptr, *vpart = nullptr;
  double *mu = nullptr, *var = nullptr;
  double *h_xs = nullptr, *h_mu = nullptr, *h_var = nullptr;  // pinned
  CUtensorMap tmKx;
  // adjoint slabs (dgp_batch_mean_functional_grad), allocated by its first call and kept: c [max_sites][chunk], v / gamma
  // and the intermediate U'v [max_sites][max_pad], its row-block partials [max_sites][max_nb][max_pad], the contraction
  // partials [max_sites][mfg_pstride], results [max_sites][1 + DGP_MAX_THETA]; pinned staging of c and of the results
  double *cvec = nullptr, *vvec = nullptr, *tmpz = nullptr, *gam = nullptr, *gzpart = nullptr, *wpart = nullptr, *mfg = nullptr;
  double *h_c = nullptr, *h_mfg = nullptr;  // pinned
  long long mfg_pstride = 0;
  long long launches = 0;
  double last_ms[4] = {0, 0, 0, 0};
  std::string err;
};
typedef struct dgp_batch_s* dgp_batch_t;

// slab [sites][rows][ld] (rows = ld: the per-site matrices; the prediction chunk: the cross-covariance slab)
static int make_map3(dgp_batch_t h, CUtensorMap* m, double* base, long long ld, long long rows, int sites) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) DGP_FAIL(h, -3, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {(cuuint64_t)ld, (cuuint64_t)rows, (cuuint64_t)sites};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 8, (cuuint64_t)rows * (cuuint64_t)ld * 8};
  cuuint32_t box[3] = {BK, 64, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) DGP_FAIL(h, -3, "cuTensorMapEncodeTiled (3-D) failed (%d) ld=%lld sites=%d", (int)r, ld, sites);
  return 0;
}

namespace {
struct TabBuilder {
  BatchTab t;
  int total = 0;
  bool any_first = false;
  explicit TabBuilder(dgp_batch_t b) {
    memset(&t, 0, sizeof(t));
    t.ld = b->ld;
    t.jitv = b->jitv;
  }
  void add(int site, int step, int nb, int n, int a0, int a1, int a2, int ntiles) {
    if (ntiles <= 0) return;
    BatchEnt& e = t.e[t.count++];
    e.tile0 = total; e.site = site; e.step = step; e.nb = nb; e.n = n; e.aux0 = a0; e.aux1 = a1; e.aux2 = a2;
    total += ntiles;
  }
};

GemmArgs b_args(dgp_batch_t b, int mode, double* C, double sign, int ntiles) {
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.mode = mode; g.nb = b->NB; g.n = 0;
  g.ntiles = ntiles; g.C = C; g.ldc = b->ld; g.sign = sign;
  g.Xw = b->Xw; g.noise = b->noise; g.theta = b->theta; g.part = b->gpart;
  return g;
}

// one rank-(128 kb) update launch over the sites of `tb` (M_TRAIL_COL entries); half_limit: largest tile count that still
// runs on 64-row half tiles
int b_launch_trail(dgp_batch_t b, const TabBuilder& tb, cudaStream_t st, int half_limit, bool pdl) {
  if (tb.total <= 0) return 0;
  GemmArgs g = b_args(b, M_TRAIL_COL, b->A, -1.0, tb.total);
  if (tb.any_first) return launch_gemm<INIT_COV, EPI_STORE>(b, b->tmL, b->tmL, g, st, pdl, &tb.t);
  if (tb.total <= half_limit) return launch_gemm<INIT_LOAD, EPI_STORE, 4>(b, b->tmL, b->tmL, g, st, pdl, &tb.t);
  return launch_gemm<INIT_LOAD, EPI_STORE>(b, b->tmL, b->tmL, g, st, pdl, &tb.t);
}

int b_ensure_events(dgp_batch_t b, size_t count) {
  while (b->evs.size() < count) {
    cudaEvent_t e;
    CK(b, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    b->evs.push_back(e);
  }
  return 0;
}

// Two-level right-looking Cholesky with look-ahead (potrf_core of dgp_api.cu) over all sites, end-aligned.
struct BInvProgress;
int b_trtri_advance(dgp_batch_t b, BInvProgress& ip, int Fg);
int b_eager(dgp_batch_t b, BInvProgress* ip, cudaEvent_t ev_panel, int pe);

int b_potrf(dgp_batch_t b, BInvProgress* eager) {
  const int G = b->G, NB = b->NB;
  constexpr int pw = PANEL_BLOCKS, sw = STRIP_BLOCKS;
  const long long ld = b->ld;
  cudaStream_t T = b->stream, P = b->stream_hi, T2 = b->stream_t2;
  const int npanels = (NB + pw - 1) / pw;
  int rc;
  bool any2 = false;
  if ((rc = b_ensure_events(b, 3 * (size_t)npanels + 3))) return rc;
  auto ev_panel = [&](int p) { return b->evs[3 * p]; };
  auto ev_cols = [&](int p) { return b->evs[3 * p + 1]; };
  auto ev_col0 = [&](int p) { return b->evs[3 * p + 2]; };
  k_cov_col0_b<<<dim3(4 * NB, 1, G), 256, 0, T>>>(b->spec, b->sd, b->theta, b->Xw, b->noise, b->jitv, b->A);
  b->launches++;
  CK(b, cudaGetLastError());
  CK(b, cudaEventRecord(ev_cols(0), T));
  CK(b, cudaStreamWaitEvent(P, ev_cols(0), 0));
  // standalone generator (as in potrf_core): the sites with more than DGP_PREGEN_MIN_NB block columns get their
  // whole lower triangle written on the low-priority stream while the first diagonal blocks are factored, and their first
  // updates read it like any later one.  The same sites by the same rule as the single-site engine: bit-identical results.
  bool pre[DGP_BATCH_MAX];
  bool any_pre = false, wP = false, wT = false, w2 = false;
  for (int i = 0; i < G; i++) {
    pre[i] = b->nb[i] > DGP_PREGEN_MIN_NB;
    any_pre |= pre[i];
  }
  cudaEvent_t ev_gen = b->evs[3 * (size_t)npanels + 1];
  if (any_pre) {
    CK(b, cudaStreamWaitEvent(b->stream_lo, ev_cols(0), 0));
    k_cov_lower_b<<<dim3(4 * NB, NB - 1, G), 256, 0, b->stream_lo>>>(b->spec, b->sd, b->theta, b->Xw, b->noise, b->jitv, b->A,
                                                                            DGP_PREGEN_MIN_NB);
    b->launches++;
    CK(b, cudaGetLastError());
    CK(b, cudaEventRecord(ev_gen, b->stream_lo));
  }
  const int slots = 2 * b->sms;
  for (int p = 0; p < npanels; p++) {
    const int pb = p * pw, pe = (pb + pw < NB) ? pb + pw : NB;
    if (p > 0) CK(b, cudaStreamWaitEvent(P, ev_col0(p), 0));
    // ---- the latency-bound chain of the panel, stream P
    for (int t = pb; t < pe; t++) {
      P2Batch pk;
      memset(&pk, 0, sizeof(pk));
      pk.slab = ld * ld;
      TabBuilder trsm(b), inp(b);
      for (int k = 0; k < G; k++) {
        const int i = b->order[k], s = t - b->off[i], nbi = b->nb[i];
        if (s < 0 || s >= nbi) continue;
        pk.site[pk.count] = (short)i; pk.step[pk.count] = (short)s; pk.count++;
        const int m = nbi - s - 1;
        trsm.add(i, s, nbi, b->n[i], 0, 1, 0, 2 * m);
        const int lpe = (pe - b->off[i] < nbi) ? pe - b->off[i] : nbi;
        if (s + 1 < lpe) {   // right-looking, like the single-site engine: the two must agree for bit-identical results
          const int w = lpe - s - 1;
          const bool first = (s == 0) && !pre[i];
          inp.add(i, s, nbi, b->n[i], (s + 1) | (w << 16), 1, first ? 0 : 1, m * 2 * w);
          inp.any_first |= first && m > 0;
        }
      }
      if (pk.count == 0) continue;
      // dependent launch behind the in-panel update of the previous block column (same stream, nothing in between)
      CK(b, launch_ex(k_potf2_v2, pk.count, P2_THREADS, (size_t)P2_SMEM, P, t > pb, (const double*)b->A, b->L, b->U, ld,
                      (double*)nullptr, b->scal, 0, b->A, 0, pk));
      b->launches++;
      if (trsm.total > 0) {  // panel solve: L[i, s] = A[i, s] T_ss', T_ss read from the diagonal block of the work matrix
        GemmArgs g = b_args(b, M_TRSM, b->L, 1.0, trsm.total);
        if (2 * trsm.total <= slots) { if ((rc = launch_gemm<INIT_ZERO, EPI_STORE, 4>(b, b->tmA, b->tmA, g, P, true, &trsm.t))) return rc; }
        else if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(b, b->tmA, b->tmA, g, P, true, &trsm.t))) return rc;
      }
      if (inp.total > 0) {   // rank-128 update of the panel's own remaining columns
        const bool waited = (t == pb && p > 0);
        if (waited) CK(b, cudaStreamWaitEvent(P, ev_cols(p), 0));
        const bool gen_wait = any_pre && !wP;
        if (gen_wait) { wP = true; CK(b, cudaStreamWaitEvent(P, ev_gen, 0)); }
        if ((rc = b_launch_trail(b, inp, P, b->sms, !waited && !gen_wait))) return rc;
      }
    }
    CK(b, cudaEventRecord(ev_panel(p), P));
    CK(b, cudaStreamWaitEvent(T, ev_panel(p), 0));
    if (any_pre && !wT) { wT = true; CK(b, cudaStreamWaitEvent(T, ev_gen, 0)); }
    if (eager != nullptr && pe < NB && (rc = b_eager(b, eager, ev_panel(p), pe))) return rc;
    // ---- rank-(128 pw) update right of the panel.  Column strips on two streams (potrf_core of dgp_api.cu): fixed strips
    // of `sw` block columns in the end-aligned (global) column numbering, strip j always on stream j mod 2; the next panel's
    // columns are the head of their strip: first column | its other columns | the rest of the strip.
    const int j0 = pe / sw;
    bool used2 = false;
    auto strip_stream = [&](int j) -> cudaStream_t {
      if ((j & 1) == 0) return T;
      if (!used2) { used2 = true; cudaStreamWaitEvent(T2, ev_panel(p), 0); }
      if (any_pre && !w2) { w2 = true; cudaStreamWaitEvent(T2, ev_gen, 0); }
      return T2;
    };
    cudaStream_t S0 = strip_stream(j0);
    TabBuilder ta(b), tb2(b), tr(b);
    int jmax = j0;
    for (int k = 0; k < G; k++) {
      const int i = b->order[k], nbi = b->nb[i], lpb = pb - b->off[i];
      if (lpb < 0 || lpb >= nbi) continue;
      const int lpe = (pe - b->off[i] < nbi) ? pe - b->off[i] : nbi;
      if (lpe >= nbi) continue;
      const int kb = lpe - lpb, ne = (lpe + pw < nbi) ? lpe + pw : nbi, w = ne - lpe, m = nbi - lpe;
      const bool first = (lpb == 0) && !pre[i];
      const int a2 = first ? 0 : 1;
      ta.add(i, lpb, nbi, b->n[i], lpe | (1 << 16), kb, a2, m * 2);
      ta.any_first |= first;
      if (w > 1) { tb2.add(i, lpb, nbi, b->n[i], (lpe + 1) | ((w - 1) << 16), kb, a2, (m - 1) * 2 * (w - 1)); tb2.any_first |= first; }
      const int e0 = ((j0 + 1) * sw - b->off[i] < nbi) ? (j0 + 1) * sw - b->off[i] : nbi;   // local end of the near strip
      if (ne < e0) { tr.add(i, lpb, nbi, b->n[i], ne | ((e0 - ne) << 16), kb, a2, (nbi - ne) * 2 * (e0 - ne)); tr.any_first |= first; }
      const int jl = (b->off[i] + nbi - 1) / sw;   // last global strip this site reaches
      if (jl > jmax) jmax = jl;
    }
    if ((rc = b_launch_trail(b, ta, S0, slots, false))) return rc;
    if (p + 1 < npanels) CK(b, cudaEventRecord(ev_col0(p + 1), S0));
    if ((rc = b_launch_trail(b, tb2, S0, slots, false))) return rc;
    if (p + 1 < npanels) CK(b, cudaEventRecord(ev_cols(p + 1), S0));
    if ((rc = b_launch_trail(b, tr, S0, slots, false))) return rc;
    for (int j = j0 + 1; j <= jmax; j++) {
      TabBuilder ts(b);
      for (int k = 0; k < G; k++) {
        const int i = b->order[k], nbi = b->nb[i], lpb = pb - b->off[i];
        if (lpb < 0 || lpb >= nbi) continue;
        const int lpe = (pe - b->off[i] < nbi) ? pe - b->off[i] : nbi;
        const int o = j * sw - b->off[i];
        if (lpe >= nbi || o >= nbi) continue;
        const int wj = (o + sw < nbi) ? sw : nbi - o;
        const bool first = (lpb == 0) && !pre[i];
        ts.add(i, lpb, nbi, b->n[i], o | (wj << 16), lpe - lpb, first ? 0 : 1, (nbi - o) * 2 * wj);
        ts.any_first |= first;
      }
      if (ts.total > 0 && (rc = b_launch_trail(b, ts, strip_stream(j), slots, false))) return rc;
    }
    if (used2) any2 = true;
  }
  if (any2) {  // the caller continues on T
    CK(b, cudaEventRecord(b->evs[3 * (size_t)npanels], T2));
    CK(b, cudaStreamWaitEvent(T, b->evs[3 * (size_t)npanels], 0));
  }
  return 0;
}

// U = L^-T by recursive doubling, all sites per launch, stream W.  b_trtri_advance(Fg): every merge whose block range lies
// inside the block columns that are final once the global step Fg is reached (site i: its first Fg - off_i columns) and has
// not been launched yet (trtri_advance of dgp_api.cu); Fg >= NB: everything that is left.  want_T: also transpose the last
// level, so that T = L^-1 is complete in the lower triangle of the A slab (dgp_batch_factorize, for the prediction).
struct BInvProgress {
  short done[16][DGP_BATCH_MAX];
  bool want_T;
  cudaStream_t W;
};

int b_trtri_advance(dgp_batch_t b, BInvProgress& ip, int Fg) {
  const int G = b->G, NB = b->NB;
  int rc, lv = 0;
  for (int hb = 1; hb < NB; hb *= 2, lv++) {
    TabBuilder tb(b);
    PairRange prg;
    memset(&prg, 0, sizeof(prg));
    int tmax = 0;
    for (int k = 0; k < G; k++) {
      const int i = b->order[k], nbi = b->nb[i];
      if (nbi <= hb) continue;
      const int npairs = (nbi - hb + 2 * hb - 1) / (2 * hb);
      const int F = Fg >= NB ? nbi : Fg - b->off[i];
      const int avail = F >= nbi ? npairs : (F > 0 ? F / (2 * hb) : 0);
      const int pr0 = ip.done[lv][i], cnt = avail - pr0;
      if (cnt <= 0) continue;
      // merges the size rule sends to the INT8 tensor cores leave the shared table and run one site at a time
      int pe = pr0;
      const size_t so = (size_t)i * (size_t)b->ld * (size_t)b->ld;
      for (; pe < avail && inv_emulated(hb, pair_w2(nbi, hb, pe)); pe++)
        if ((rc = inv_merge_i8(b, b->l8, b->max_pad, b->A + so, b->L + so, b->U + so, b->ld, pe * 2 * hb, hb,
                               pair_w2(nbi, hb, pe), ip.W))) return rc;
      tb.add(i, pe, nbi, b->n[i], hb, avail - pe, 0, (avail - pe) * hb * 2 * hb);
      if (ip.want_T || 2 * hb < nbi) {
        prg.pr0[i] = (short)pr0; prg.cnt[i] = (short)cnt;
        if (cnt * 16 * hb * hb > tmax) tmax = cnt * 16 * hb * hb;
      }
      ip.done[lv][i] = (short)avail;
    }
    if (tb.total > 0) {   // (none when every merge of the level went to the INT8 tensor cores; the transposes still run)
      GemmArgs gm = b_args(b, M_INV_M, b->A, 1.0, tb.total);
      if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(b, b->tmU, b->tmL, gm, ip.W, false, &tb.t))) return rc;
      GemmArgs gu = b_args(b, M_INV_U, b->U, -1.0, tb.total);
      if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(b, b->tmA, b->tmA, gu, ip.W, false, &tb.t))) return rc;
    }
    if (tmax > 0) {
      k_transpose_pairs_b<<<dim3(tmax, G), 256, 0, ip.W>>>(b->sd, prg, b->U, b->A, hb);
      b->launches++;
      CK(b, cudaGetLastError());
    }
  }
  return 0;
}

int b_eager(dgp_batch_t b, BInvProgress* ip, cudaEvent_t ev_panel, int pe) {
  if ((pe & 7) != 0) return 0;
  CK(b, cudaStreamWaitEvent(ip->W, ev_panel, 0));
  return b_trtri_advance(b, *ip, pe);
}

// the rest of the inverse, then z = U'r, alpha = U z
int b_trtri(dgp_batch_t b, BInvProgress& ip) {
  const int G = b->G, NB = b->NB;
  cudaStream_t W = ip.W;
  int rc;
  if ((rc = b_trtri_advance(b, ip, NB))) return rc;
  k_upperT_gemv_part_b<<<dim3(NB, NB, G), 256, 0, W>>>(b->sd, b->U, b->r, b->zpart);
  k_upperT_gemv_sum_b<<<dim3((unsigned)((b->ld + 255) / 256), G), 256, 0, W>>>(b->sd, b->zpart, b->z);
  k_upper_gemv_b<<<dim3((unsigned)(b->ld / 8), G), 256, 0, W>>>(b->sd, b->U, b->z, b->alpha);
  b->launches += 3;
  CK(b, cudaGetLastError());
  return 0;
}

// LAUUM -> Ky^-1 (lower tiles, over the dead T) and the gradient contraction W (.) dK/dtheta; all sites per launch.
// Sites the size rule of the single-site engine sends to the INT8 tensor cores go there one by one, the others share
// one DMMA launch.
int b_lauum_grad(dgp_batch_t b, cudaStream_t W) {
  TabBuilder tb(b);
  int rc;
  for (int k = 0; k < b->G; k++) {
    const int i = b->order[k];
    if (lauum_emulated(b->nb[i] * 128)) {
      const size_t so = (size_t)i * (size_t)b->ld * (size_t)b->ld;
      if ((rc = lauum_i8(b, b->l8, b->max_pad, b->U + so, b->A + so, b->ld, b->nb[i] * 128, W))) return rc;
    } else {
      tb.add(i, 0, b->nb[i], b->n[i], 0, 0, 0, lauum_slots(b->nb[i]));
    }
  }
  GemmArgs g = b_args(b, M_LAUUM, b->A, 1.0, tb.total);
  rc = launch_gemm<INIT_ZERO, EPI_STORE>(b, b->tmU, b->tmU, g, W, false, &tb.t);
  if (rc) return rc;
  k_grad_contract_b<<<b->sd.tile0[b->G], 128, 0, W>>>(b->spec, b->sd, b->theta, b->Xw, b->alpha, b->A, b->gpart);
  b->launches++;
  CK(b, cudaGetLastError());
  return 0;
}

// level 1: NLML + gradient (dgp_batch_nlml_grad); level 2: factorise for the prediction (dgp_batch_factorize: the inverse
// with its last level transposed, no LAUUM, no gradient), as evaluate_enqueue of dgp_api.cu
int b_enqueue(dgp_batch_t b, int level) {
  int rc;
  const int G = b->G;
  cudaStream_t T = b->stream, W = b->stream_lo ? b->stream_lo : b->stream;
  if (b->timing) CK(b, cudaEventRecord(b->ev[0], T));
  CK(b, cudaMemcpyAsync(b->theta, b->h_theta, sizeof(double) * DGP_MAX_THETA * G, cudaMemcpyHostToDevice, T));
  CK(b, cudaMemcpyAsync(b->jitv, b->h_jit, sizeof(double) * G, cudaMemcpyHostToDevice, T));
  k_features_b<<<dim3((unsigned)((b->ld + 255) / 256), G), 256, 0, T>>>(b->spec, b->sd, b->theta, b->X, b->y, b->Xw, b->r, b->scal);
  b->launches++;
  CK(b, cudaGetLastError());
  BInvProgress ip;
  memset(&ip, 0, sizeof(ip));
  ip.W = W;
  ip.want_T = (level == 2);
  // the merges of the inverse are released as the factorisation passes them at every size (unlike the single-site engine)
  if ((rc = b_potrf(b, W != T ? &ip : nullptr))) return rc;
  if (b->timing) CK(b, cudaEventRecord(b->ev[1], T));
  if (W != T) {
    CK(b, cudaEventRecord(b->ev_lo[0], T));
    CK(b, cudaStreamWaitEvent(W, b->ev_lo[0], 0));
  }
  if ((rc = b_trtri(b, ip))) return rc;
  if (b->timing) CK(b, cudaEventRecord(b->ev[2], W));
  if (level == 1 && (rc = b_lauum_grad(b, W))) return rc;
  if (b->timing) CK(b, cudaEventRecord(b->ev[3], W));
  if (W != T) {
    CK(b, cudaEventRecord(b->ev_lo[1], W));
    CK(b, cudaStreamWaitEvent(T, b->ev_lo[1], 0));
  }
  k_finish_b<<<dim3(b->spec.ntheta + 1, G), 256, 0, T>>>(b->spec, b->sd, b->theta, b->gpart, b->z, b->alpha, b->X, b->scal,
                                                          level == 1 ? 1 : 0);
  b->launches++;
  CK(b, cudaGetLastError());
  CK(b, cudaMemcpyAsync(b->h_scal, b->scal, sizeof(double) * SC_SIZE * G, cudaMemcpyDeviceToHost, T));
  if (b->timing) CK(b, cudaEventRecord(b->ev[4], T));
  return 0;
}

// Rows of every site's prediction grid per batched launch.  1024 keeps the cross-covariance slab at 1024 / (3 max_pad) of the
// training slabs (64 MB per site at n = 8192) while a launch of the variance GEMM still has 8 x 2 nb tiles per site, a full
// wave of the 2 x 148 CTA slots for a single site from 19 block columns (n > 2304) on; 2048 rows would only save the 4 launches per chunk.
constexpr int DGP_BATCH_CHUNK = 1024;

void b_predict_free(dgp_batch_t b) {
  double* bufs[] = {b->Kx, b->Xs, b->Xws, b->means, b->dot, b->vpart, b->mu, b->var};
  for (double* p : bufs) if (p) cudaFree(p);
  double* hbufs[] = {b->h_xs, b->h_mu, b->h_var};
  for (double* p : hbufs) if (p) cudaFreeHost(p);
  b->Kx = b->Xs = b->Xws = b->means = b->dot = b->vpart = b->mu = b->var = nullptr;
  b->h_xs = b->h_mu = b->h_var = nullptr;
}

void b_mfg_free(dgp_batch_t b) {
  double* bufs[] = {b->cvec, b->vvec, b->tmpz, b->gam, b->gzpart, b->wpart, b->mfg};
  for (double* p : bufs) if (p) cudaFree(p);
  if (b->h_c) cudaFreeHost(b->h_c);
  if (b->h_mfg) cudaFreeHost(b->h_mfg);
  b->cvec = b->vvec = b->tmpz = b->gam = b->gzpart = b->wpart = b->mfg = nullptr;
  b->h_c = b->h_mfg = nullptr;
}

// the prediction slabs, once per handle, for max_sites sites of up to max_n points (later calls allocate nothing)
int b_predict_alloc(dgp_batch_t b) {
  if (b->Kx) return 0;
  const size_t S = b->max_sites, C = DGP_BATCH_CHUNK, np = b->max_pad, nbm = np / 128;
  cudaError_t r = cudaSuccess;
  auto A = [&](double** p, size_t count) { if (r == cudaSuccess) r = cudaMalloc((void**)p, count * sizeof(double)); };
  auto H = [&](double** p, size_t count) { if (r == cudaSuccess) r = cudaMallocHost((void**)p, count * sizeof(double)); };
  A(&b->Kx, S * C * np); A(&b->dot, S * nbm * C); A(&b->vpart, S * 2 * nbm * C);
  A(&b->Xs, S * C * DGP_MAX_COLS); A(&b->Xws, S * C * DGP_XS); A(&b->means, S * C); A(&b->mu, S * C); A(&b->var, S * C);
  H(&b->h_xs, S * C * DGP_MAX_COLS); H(&b->h_mu, S * C); H(&b->h_var, S * C);
  if (r != cudaSuccess) {
    cudaGetLastError();
    b_predict_free(b);
    DGP_FAIL(b, -2, "dgp_batch_predict: allocation of the prediction slabs failed: %s", cudaGetErrorString(r));
  }
  return 0;
}

// the adjoint slabs, once per handle (the partials of a site: (chunk / 128 + nb) (2 nb) tiles at the largest m and n)
int b_mfg_alloc(dgp_batch_t b) {
  if (b->cvec) return 0;
  const size_t S = b->max_sites, C = DGP_BATCH_CHUNK, np = b->max_pad, nbm = np / 128;
  b->mfg_pstride = (long long)((C / 128 + nbm) * (np / 64) * DGP_MAX_THETA);
  cudaError_t r = cudaSuccess;
  auto A = [&](double** p, size_t count) { if (r == cudaSuccess) r = cudaMalloc((void**)p, count * sizeof(double)); };
  auto H = [&](double** p, size_t count) { if (r == cudaSuccess) r = cudaMallocHost((void**)p, count * sizeof(double)); };
  A(&b->cvec, S * C); A(&b->vvec, S * np); A(&b->tmpz, S * np); A(&b->gam, S * np); A(&b->gzpart, S * nbm * np);
  A(&b->wpart, S * (size_t)b->mfg_pstride); A(&b->mfg, S * (1 + DGP_MAX_THETA));
  H(&b->h_c, S * C); H(&b->h_mfg, S * (1 + DGP_MAX_THETA));
  if (r != cudaSuccess) {
    cudaGetLastError();
    b_mfg_free(b);
    DGP_FAIL(b, -2, "dgp_batch_mean_functional_grad: allocation of the adjoint slabs failed: %s", cudaGetErrorString(r));
  }
  return 0;
}
}  // namespace

extern "C" {

size_t dgp_batch_workspace_bytes(int max_sites, int max_n) {
  const size_t np = round_up(max_n > 0 ? max_n : 128, 128), S = max_sites > 0 ? max_sites : 1, nbm = np / 128;
  return S * (3 * np * np + np * (DGP_MAX_COLS + DGP_XS + 6) + nbm * (nbm + 1) * DGP_MAX_THETA + nbm * np + DGP_MAX_THETA + SC_SIZE + 1) * 8;
}

int dgp_batch_destroy(dgp_batch b) {
  if (!b) return 0;
  cudaSetDevice(b->device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  if (b->stream_hi) { cudaStreamSynchronize(b->stream_hi); cudaStreamDestroy(b->stream_hi); }
  if (b->stream_lo) { cudaStreamSynchronize(b->stream_lo); cudaStreamDestroy(b->stream_lo); }
  if (b->stream_t2) { cudaStreamSynchronize(b->stream_t2); cudaStreamDestroy(b->stream_t2); }
  for (int i = 0; i < 2; i++) if (b->ev_lo[i]) cudaEventDestroy(b->ev_lo[i]);
  for (int i = 0; i < 5; i++) if (b->ev[i]) cudaEventDestroy(b->ev[i]);
  for (cudaEvent_t e : b->evs) cudaEventDestroy(e);
  double* bufs[] = {b->A, b->L, b->U, b->X, b->y, b->noise, b->Xw, b->r, b->z, b->alpha, b->theta, b->scal, b->gpart, b->zpart, b->jitv};
  for (double* p : bufs) if (p) cudaFree(p);
  b_predict_free(b);
  b_mfg_free(b);
  b->l8.release();
  if (b->h_theta) cudaFreeHost(b->h_theta);
  if (b->h_scal) cudaFreeHost(b->h_scal);
  if (b->h_jit) cudaFreeHost(b->h_jit);
  if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
  delete b;
  return 0;
}

int dgp_batch_create(dgp_batch* out, int device, int max_sites, int max_n, void* stream) {
  dgp_batch_t nil = nullptr;
  if (!out || max_n <= 0 || max_sites < 1 || max_sites > DGP_BATCH_MAX)
    DGP_FAIL(nil, -1, "dgp_batch_create: bad arguments (1 <= max_sites <= %d)", DGP_BATCH_MAX);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    DGP_FAIL(nil, -2, "dgp_batch_create: no CUDA device (this engine has no CPU fallback)");
  if (cudaSetDevice(device) != cudaSuccess) DGP_FAIL(nil, -2, "dgp_batch_create: cannot select device %d", device);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) DGP_FAIL(nil, -2, "dgp_batch_create: libdgp is built for sm_100a (B200) only");
  dgp_batch_t b = new dgp_batch_s();
  b->device = device;
  b->sms = prop.multiProcessorCount;
  b->max_sites = max_sites; b->max_n = max_n; b->max_pad = round_up(max_n, 128);
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);
  if (stream) b->stream = (cudaStream_t)stream;
  else {
    cudaStreamCreateWithPriority(&b->stream, cudaStreamNonBlocking, (lo + hi) / 2);
    b->own_stream = true;
  }
  cudaStreamCreateWithPriority(&b->stream_lo, cudaStreamNonBlocking, lo);
  cudaStreamCreateWithPriority(&b->stream_hi, cudaStreamNonBlocking, hi);
  {
    int pr = (lo + hi) / 2;
    if (cudaStreamGetPriority(b->stream, &pr) != cudaSuccess) { cudaGetLastError(); pr = (lo + hi) / 2; }
    cudaStreamCreateWithPriority(&b->stream_t2, cudaStreamNonBlocking, pr);
  }
  const size_t np = b->max_pad, S = max_sites, nbm = np / 128;
  cudaError_t r = cudaSuccess;
  auto A = [&](double** p, size_t count) { if (r == cudaSuccess) r = cudaMalloc((void**)p, count * sizeof(double)); };
  A(&b->A, S * np * np); A(&b->L, S * np * np); A(&b->U, S * np * np);
  A(&b->X, S * np * DGP_MAX_COLS); A(&b->y, S * np); A(&b->noise, S * np); A(&b->Xw, S * np * DGP_XS);
  A(&b->r, S * np); A(&b->z, S * np); A(&b->alpha, S * np);
  A(&b->theta, S * DGP_MAX_THETA); A(&b->scal, S * SC_SIZE); A(&b->gpart, S * nbm * (nbm + 1) * DGP_MAX_THETA);
  A(&b->zpart, S * nbm * np); A(&b->jitv, S);
  if (r == cudaSuccess) r = cudaMallocHost((void**)&b->h_theta, S * DGP_MAX_THETA * sizeof(double));
  if (r == cudaSuccess) r = cudaMallocHost((void**)&b->h_scal, S * SC_SIZE * sizeof(double));
  if (r == cudaSuccess) r = cudaMallocHost((void**)&b->h_jit, S * sizeof(double));
  for (int i = 0; i < 5 && r == cudaSuccess; i++) r = cudaEventCreate(&b->ev[i]);
  for (int i = 0; i < 2 && r == cudaSuccess; i++) r = cudaEventCreateWithFlags(&b->ev_lo[i], cudaEventDisableTiming);
  if (r != cudaSuccess) {
    g_create_error = std::string("dgp_batch_create: allocation failed: ") + cudaGetErrorString(r);
    cudaGetLastError();
    dgp_batch_destroy(b);
    return -2;
  }
  cudaFuncSetAttribute(k_potf2_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM);
  *out = b;
  return 0;
}

const char* dgp_batch_last_error(dgp_batch b) { return b ? b->err.c_str() : g_create_error.c_str(); }

int dgp_batch_set_train(dgp_batch b, const dgp_spec* spec, int nsites, const int* n, const double* const* X,
                        const double* const* y, const double* const* noise) {
  if (!b) return -1;
  if (!spec || !n || !X || !y || !noise || nsites < 1 || nsites > b->max_sites)
    DGP_FAIL(b, -1, "dgp_batch_set_train: bad arguments (nsites=%d, max_sites=%d)", nsites, b->max_sites);
  int rc = check_spec(b, spec);
  if (rc) return rc;
  for (int i = 0; i < nsites; i++)
    if (n[i] < 1 || n[i] > b->max_n || !X[i] || !y[i] || !noise[i])
      DGP_FAIL(b, -1, "dgp_batch_set_train: site %d: n=%d (max_n=%d) or NULL data", i, n[i], b->max_n);
  CK(b, cudaSetDevice(b->device));
  if (b->pending) { CK(b, cudaStreamSynchronize(b->stream)); b->pending = false; }
  b->user_spec = *spec;
  b->spec = *spec;
  augment_spec(&b->spec);
  b->G = nsites;
  int npmax = 0;
  for (int i = 0; i < nsites; i++) {
    b->n[i] = n[i];
    b->nb[i] = round_up(n[i], 128) / 128;
    if (b->nb[i] * 128 > npmax) npmax = b->nb[i] * 128;
  }
  b->ld = npmax;
  b->NB = npmax / 128;
  const int pw = PANEL_BLOCKS;
  memset(&b->sd, 0, sizeof(b->sd));
  b->sd.count = nsites; b->sd.nbmax = b->NB; b->sd.ld = b->ld;
  for (int i = 0; i < nsites; i++) {
    b->off[i] = ((b->NB - b->nb[i]) / pw) * pw;
    b->sd.n[i] = b->n[i]; b->sd.nb[i] = b->nb[i];
    b->sd.tile0[i + 1] = b->sd.tile0[i] + b->nb[i] * (b->nb[i] + 1);
    b->order[i] = i;
  }
  // launch tables list the sites largest first (longest tiles of a launch start first)
  for (int i = 1; i < nsites; i++)
    for (int k = i; k > 0 && b->nb[b->order[k]] > b->nb[b->order[k - 1]]; k--) std::swap(b->order[k], b->order[k - 1]);
  const size_t ld = (size_t)b->ld, slab = ld * ld;
  cudaStream_t st = b->stream;
  CK(b, cudaMemsetAsync(b->L, 0, slab * nsites * 8, st));
  CK(b, cudaMemsetAsync(b->U, 0, slab * nsites * 8, st));
  CK(b, cudaMemsetAsync(b->noise, 0, ld * nsites * 8, st));
  CK(b, cudaMemsetAsync(b->X, 0, ld * nsites * DGP_MAX_COLS * 8, st));
  CK(b, cudaMemsetAsync(b->y, 0, ld * nsites * 8, st));
  for (int i = 0; i < nsites; i++) {
    CK(b, cudaMemcpyAsync(b->X + (size_t)i * ld * DGP_MAX_COLS, X[i], (size_t)n[i] * spec->ndim * 8, cudaMemcpyHostToDevice, st));
    CK(b, cudaMemcpyAsync(b->y + (size_t)i * ld, y[i], (size_t)n[i] * 8, cudaMemcpyHostToDevice, st));
    CK(b, cudaMemcpyAsync(b->noise + (size_t)i * ld, noise[i], (size_t)n[i] * 8, cudaMemcpyHostToDevice, st));
  }
  CK(b, cudaStreamSynchronize(st));
  for (int i = 0; i < DGP_BATCH_MAX; i++) b->have_T[i] = b->have_eval[i] = false;
  if ((rc = make_map3(b, &b->tmA, b->A, b->ld, b->ld, nsites))) return rc;
  if ((rc = make_map3(b, &b->tmL, b->L, b->ld, b->ld, nsites))) return rc;
  if ((rc = make_map3(b, &b->tmU, b->U, b->ld, b->ld, nsites))) return rc;
  b->have_train = true;
  return 0;
}

// level 1: dgp_batch_nlml_grad_launch; level 2: dgp_batch_factorize
static int b_launch(dgp_batch b, const double* theta, const double* jitter, int level) {
  if (!b) return -1;
  if (!b->have_train) DGP_FAIL(b, -1, "no training data: call dgp_batch_set_train first");
  if (!theta) DGP_FAIL(b, -1, "theta is NULL");
  if (b->pending) DGP_FAIL(b, -1, "an evaluation is already in flight: call dgp_batch_nlml_grad_wait first");
  CK(b, cudaSetDevice(b->device));
  for (int i = 0; i < DGP_BATCH_MAX; i++) b->have_T[i] = b->have_eval[i] = false;
  const int P = b->spec.ntheta;
  memset(b->h_theta, 0, sizeof(double) * DGP_MAX_THETA * b->G);
  for (int i = 0; i < b->G; i++) {
    memcpy(b->h_theta + (size_t)i * DGP_MAX_THETA, theta + (size_t)i * P, sizeof(double) * P);
    b->h_jit[i] = jitter ? jitter[i] : 0.0;
  }
  int rc = b_enqueue(b, level);
  if (rc) return rc;
  b->pending = true;
  return 0;
}

int dgp_batch_nlml_grad_launch(dgp_batch b, const double* theta, const double* jitter) {
  return b_launch(b, theta, jitter, 1);
}

int dgp_batch_nlml_grad_ready(dgp_batch b) {
  if (!b) return -1;
  if (!b->pending) DGP_FAIL(b, -1, "no evaluation in flight");
  CK(b, cudaSetDevice(b->device));
  const cudaError_t e = cudaStreamQuery(b->stream);
  if (e == cudaSuccess) return 1;
  if (e == cudaErrorNotReady) return 0;
  DGP_FAIL(b, -2, "cudaStreamQuery failed: %s", cudaGetErrorString(e));
}

int dgp_batch_nlml_grad_wait(dgp_batch b, double* nlml_out, double* grad_out, int* info_out) {
  if (!b) return -1;
  if (!b->pending) DGP_FAIL(b, -1, "no evaluation in flight");
  CK(b, cudaSetDevice(b->device));
  CK(b, cudaStreamSynchronize(b->stream));
  b->pending = false;
  if (b->timing) {
    float ms;
    for (int i = 0; i < 4; i++) { cudaEventElapsedTime(&ms, b->ev[i], b->ev[i + 1]); b->last_ms[i] = ms; }
  }
  const int P = b->spec.ntheta;
  int bad = 0;
  for (int i = 0; i < b->G; i++) {
    const double* sc = b->h_scal + (size_t)i * SC_SIZE;
    if (nlml_out) nlml_out[i] = sc[SC_NLML];
    if (grad_out) memcpy(grad_out + (size_t)i * P, sc + SC_GRAD, sizeof(double) * P);
    const int info = (int)sc[SC_INFO];
    if (info_out) info_out[i] = info;
    b->have_eval[i] = info == 0;
    if (info != 0) bad++;
  }
  return bad;
}

int dgp_batch_nlml_grad(dgp_batch b, const double* theta, const double* jitter, double* nlml_out, double* grad_out,
                        int* info_out) {
  int rc = dgp_batch_nlml_grad_launch(b, theta, jitter);
  if (rc) return rc;
  return dgp_batch_nlml_grad_wait(b, nlml_out, grad_out, info_out);
}

int dgp_batch_get_alpha(dgp_batch b, int site, double* alpha_out) {
  if (!b) return -1;
  if (!b->have_train || b->pending || site < 0 || site >= b->G || !alpha_out) DGP_FAIL(b, -1, "dgp_batch_get_alpha: bad arguments");
  CK(b, cudaSetDevice(b->device));
  CK(b, cudaMemcpyAsync(alpha_out, b->alpha + (size_t)site * b->ld, (size_t)b->n[site] * 8, cudaMemcpyDeviceToHost, b->stream));
  CK(b, cudaStreamSynchronize(b->stream));
  return 0;
}

int dgp_batch_factorize(dgp_batch b, const double* theta, const double* jitter, double* nlml_out, int* info_out) {
  int rc = b_launch(b, theta, jitter, 2);
  if (rc) return rc;
  if ((rc = dgp_batch_nlml_grad_wait(b, nlml_out, nullptr, info_out)) < 0) return rc;
  for (int i = 0; i < b->G; i++) b->have_T[i] = (int)b->h_scal[(size_t)i * SC_SIZE + SC_INFO] == 0;
  return rc;
}

// dgp_predict for every site of the batch, DGP_BATCH_CHUNK rows of every grid per launch: features of the chunk -> cross
// covariance + mean partials -> variance GEMM V'[i, c] = sum_k Kx[i, k] T[c, k] with row sums of squares (M_PREDVAR,
// EPI_SUMSQ) -> mu, var.  Per site, every tile and partial sums the same k range in the same order as the single-site
// prediction, and rows never mix: the results do not depend on the chunk or on which sites share a launch.
int dgp_batch_predict(dgp_batch b, const int* m, const double* const* Xs, double* const* mu_out, double* const* var_out) {
  if (!b) return -1;
  if (!b->have_train || !m || !Xs || !mu_out) DGP_FAIL(b, -1, "dgp_batch_predict: bad arguments");
  if (b->pending) DGP_FAIL(b, -1, "dgp_batch_predict: an evaluation is in flight: call dgp_batch_nlml_grad_wait first");
  const int G = b->G, C = DGP_BATCH_CHUNK, ndim = b->spec.ndim;
  int mmax = 0;
  for (int i = 0; i < G; i++) {
    if (m[i] < 0) DGP_FAIL(b, -1, "dgp_batch_predict: site %d: m = %d", i, m[i]);
    if (m[i] == 0) continue;
    if (!Xs[i] || !mu_out[i]) DGP_FAIL(b, -1, "dgp_batch_predict: site %d: NULL grid or output", i);
    const bool want_var = var_out != nullptr && var_out[i] != nullptr;
    if (want_var && !b->have_T[i])
      DGP_FAIL(b, -1, "dgp_batch_predict: site %d is not factorised: call dgp_batch_factorize first (again after every "
               "dgp_batch_set_train / dgp_batch_nlml_grad; a site whose factorisation failed cannot predict)", i);
    if (!want_var && !b->have_eval[i])
      DGP_FAIL(b, -1, "dgp_batch_predict: site %d has no successful evaluation: the mean needs dgp_batch_nlml_grad or "
               "dgp_batch_factorize first (again after every dgp_batch_set_train; a site whose evaluation failed cannot predict)", i);
    if (m[i] > mmax) mmax = m[i];
  }
  if (mmax == 0) return 0;
  CK(b, cudaSetDevice(b->device));
  int rc;
  if ((rc = b_predict_alloc(b))) return rc;
  if ((rc = make_map3(b, &b->tmKx, b->Kx, b->ld, C, G))) return rc;
  cudaStream_t st = b->stream;
  for (int m0 = 0; m0 < mmax; m0 += C) {
    PredChunk pc;
    memset(&pc, 0, sizeof(pc));
    TabBuilder tb(b);
    bool any_var = false;
    for (int k = 0; k < G; k++) {   // largest sites first in the GEMM's table, as in every other batched launch
      const int i = b->order[k];
      const int mc = m[i] - m0 < 0 ? 0 : (m[i] - m0 < C ? m[i] - m0 : C);
      if (mc == 0) continue;
      pc.m[i] = mc;
      pc.var[i] = var_out != nullptr && var_out[i] != nullptr;
      memcpy(b->h_xs + (size_t)i * C * DGP_MAX_COLS, Xs[i] + (size_t)m0 * ndim, (size_t)mc * ndim * 8);
      if (pc.var[i]) {
        const int rb = (mc + 127) / 128;
        tb.add(i, 0, b->nb[i], b->n[i], rb, C, 0, rb * 2 * b->nb[i]);
        any_var = true;
      }
    }
    CK(b, cudaMemcpyAsync(b->Xs, b->h_xs, (size_t)G * C * DGP_MAX_COLS * 8, cudaMemcpyHostToDevice, st));
    k_pred_features_b<<<dim3(C / 256, G), 256, 0, st>>>(b->spec, pc, b->theta, b->Xs, b->Xws, b->means, C);
    k_cov_rect_pred_b<<<dim3(C / 32, b->NB, G), 256, 0, st>>>(b->spec, b->sd, pc, b->theta, b->Xws, b->Xw, b->noise, b->alpha,
                                                              b->Kx, b->dot, C);
    b->launches += 2;
    CK(b, cudaGetLastError());
    if (any_var) {
      GemmArgs g = b_args(b, M_PREDVAR, nullptr, 1.0, tb.total);
      g.aux1 = C; g.part = b->vpart;
      if ((rc = launch_gemm<INIT_ZERO, EPI_SUMSQ>(b, b->tmKx, b->tmA, g, st, false, &tb.t))) return rc;
    }
    k_pred_finish_b<<<dim3(C / 256, G), 256, 0, st>>>(b->spec, b->sd, pc, b->theta, b->Xws, b->means, b->dot, b->vpart, b->mu,
                                                      b->var, C);
    b->launches++;
    CK(b, cudaGetLastError());
    CK(b, cudaMemcpyAsync(b->h_mu, b->mu, (size_t)G * C * 8, cudaMemcpyDeviceToHost, st));
    if (any_var) CK(b, cudaMemcpyAsync(b->h_var, b->var, (size_t)G * C * 8, cudaMemcpyDeviceToHost, st));
    CK(b, cudaStreamSynchronize(st));
    for (int i = 0; i < G; i++) {
      if (pc.m[i] == 0) continue;
      memcpy(mu_out[i] + m0, b->h_mu + (size_t)i * C, (size_t)pc.m[i] * 8);
      if (pc.var[i]) memcpy(var_out[i] + m0, b->h_var + (size_t)i * C, (size_t)pc.m[i] * 8);
    }
  }
  return 0;
}

// dgp_mean_functional_grad for every site of the batch, each step one launch over all sites: features, cross covariance
// and mu of the points (the prediction kernels on the chunk slabs; Kx is kept) -> v = Kx' c -> gamma = U (U' v) on the U
// slab (U = L^-T is intact after both evaluations: LAUUM writes Ky^-1 into A) -> both weighted contractions of dK/dtheta
// -> the per-site reductions.  alpha, z and zpart, which later predictions and evaluations read, are not touched.
int dgp_batch_mean_functional_grad(dgp_batch b, const int* m, const double* const* Xs, const double* const* c,
                                   double* val_out, double* grad_out) {
  if (!b) return -1;
  if (!b->have_train || !m || !Xs || !c || !val_out || !grad_out)
    DGP_FAIL(b, -1, "dgp_batch_mean_functional_grad: bad arguments (NULL pointer or no training data)");
  if (b->pending) DGP_FAIL(b, -1, "dgp_batch_mean_functional_grad: an evaluation is in flight: call dgp_batch_nlml_grad_wait first");
  const int G = b->G, C = DGP_BATCH_CHUNK, ndim = b->spec.ndim, P = b->spec.ntheta;
  MfgTab mt;
  memset(&mt, 0, sizeof(mt));
  for (int i = 0; i < G; i++) {
    if (m[i] < 0 || m[i] > C) DGP_FAIL(b, -1, "dgp_batch_mean_functional_grad: site %d: m = %d (0 <= m <= %d)", i, m[i], C);
    if (m[i] == 0) continue;
    if (!Xs[i] || !c[i]) DGP_FAIL(b, -1, "dgp_batch_mean_functional_grad: site %d: NULL points or weights", i);
    if (!b->have_eval[i])
      DGP_FAIL(b, -1, "dgp_batch_mean_functional_grad: site %d has no successful evaluation: call dgp_batch_nlml_grad or "
               "dgp_batch_factorize first (again after every dgp_batch_set_train; a site whose evaluation failed has no adjoint)", i);
    mt.m[i] = m[i];
  }
  for (int i = 0; i < G; i++) mt.tile0[i + 1] = mt.tile0[i] + (mt.m[i] == 0 ? 0 : ((mt.m[i] + 127) / 128 + b->nb[i]) * 2 * b->nb[i]);
  memset(val_out, 0, sizeof(double) * G);
  memset(grad_out, 0, sizeof(double) * G * P);
  if (mt.tile0[G] == 0) return 0;
  CK(b, cudaSetDevice(b->device));
  int rc;
  if ((rc = b_predict_alloc(b))) return rc;
  if ((rc = b_mfg_alloc(b))) return rc;
  cudaStream_t st = b->stream;
  PredChunk pk, pm;   // pk: write the cross covariance (kept for v = Kx' c); pm: the mean alone
  memset(&pk, 0, sizeof(pk));
  memset(&pm, 0, sizeof(pm));
  for (int i = 0; i < G; i++) {
    pk.m[i] = pm.m[i] = mt.m[i];
    pk.var[i] = mt.m[i] > 0;
    if (mt.m[i] == 0) continue;
    const int mpad = (mt.m[i] + 127) / 128 * 128;
    memcpy(b->h_xs + (size_t)i * C * DGP_MAX_COLS, Xs[i], (size_t)mt.m[i] * ndim * 8);
    memcpy(b->h_c + (size_t)i * C, c[i], (size_t)mt.m[i] * 8);
    memset(b->h_c + (size_t)i * C + mt.m[i], 0, (size_t)(mpad - mt.m[i]) * 8);
  }
  CK(b, cudaMemcpyAsync(b->Xs, b->h_xs, (size_t)G * C * DGP_MAX_COLS * 8, cudaMemcpyHostToDevice, st));
  CK(b, cudaMemcpyAsync(b->cvec, b->h_c, (size_t)G * C * 8, cudaMemcpyHostToDevice, st));
  const unsigned gl = (unsigned)((b->ld + 255) / 256);
  k_pred_features_b<<<dim3(C / 256, G), 256, 0, st>>>(b->spec, pk, b->theta, b->Xs, b->Xws, b->means, C);
  k_cov_rect_pred_b<<<dim3(C / 32, b->NB, G), 256, 0, st>>>(b->spec, b->sd, pk, b->theta, b->Xws, b->Xw, b->noise, b->alpha,
                                                            b->Kx, b->dot, C);
  k_pred_finish_b<<<dim3(C / 256, G), 256, 0, st>>>(b->spec, b->sd, pm, b->theta, b->Xws, b->means, b->dot, b->vpart, b->mu,
                                                    b->var, C);
  // gamma = Ky^-1 (Kx*' c) = U (U' v)
  k_colsum_weighted_b<<<dim3(gl, G), 256, 0, st>>>(b->sd, mt, b->Kx, b->cvec, b->vvec, C);
  k_upperT_gemv_part_b<<<dim3(b->NB, b->NB, G), 256, 0, st>>>(b->sd, b->U, b->vvec, b->gzpart);
  k_upperT_gemv_sum_b<<<dim3(gl, G), 256, 0, st>>>(b->sd, b->gzpart, b->tmpz);
  k_upper_gemv_b<<<dim3((unsigned)(b->ld / 8), G), 256, 0, st>>>(b->sd, b->U, b->tmpz, b->gam);
  // the two weighted contractions of dK/dtheta, then the per-site reductions
  k_wgrad_b<<<mt.tile0[G], 128, 0, st>>>(b->spec, b->sd, mt, b->theta, b->Xws, b->Xw, b->cvec, b->gam, b->alpha, b->wpart, C,
                                         b->mfg_pstride);
  k_mfg_finish_b<<<dim3(P + 1, G), 256, 0, st>>>(b->spec, b->sd, mt, b->theta, b->wpart, b->cvec, b->mu, b->Xs, b->gam,
                                                 b->alpha, b->X, b->mfg, C, b->mfg_pstride);
  b->launches += 9;
  CK(b, cudaGetLastError());
  CK(b, cudaMemcpyAsync(b->h_mfg, b->mfg, (size_t)G * (1 + DGP_MAX_THETA) * 8, cudaMemcpyDeviceToHost, st));
  CK(b, cudaStreamSynchronize(st));
  for (int i = 0; i < G; i++) {
    if (mt.m[i] == 0) continue;
    const double* o = b->h_mfg + (size_t)i * (1 + DGP_MAX_THETA);
    val_out[i] = o[0];
    memcpy(grad_out + (size_t)i * P, o + 1, sizeof(double) * P);
  }
  return 0;
}

long long dgp_batch_launch_count(dgp_batch b) { return b ? b->launches : 0; }
int dgp_batch_set_timing(dgp_batch b, int enable) { if (!b) return -1; b->timing = enable != 0; return 0; }
int dgp_batch_last_timing(dgp_batch b, double* ms4) {
  if (!b || !ms4) return -1;
  for (int i = 0; i < 4; i++) ms4[i] = b->last_ms[i];
  return 0;
}

}  // extern "C"
