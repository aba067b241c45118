// qlnlp_eval_body.cuh -- the body of the evaluator kernel (qlnlp_kernels.cuh), NOT a header: it is included inside
// eval_kernel and eval_prod_kernel, which define JM, FASTDIV, RAGGED and the launch record P.  Kept as one text so that
// both kernels run the same steps and the existing instantiations read their __grid_constant__ parameter directly
// (a device function taking it by reference or by value compiles to different code).
    constexpr bool WITH_JAC = JM != JM_NONE;
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x;

    // layout (RAGGED: sized for the largest horizon of the launch, P.c.N)
    double* const zbuf = smem;
    const unsigned mbar = smem_addr(zbuf + zbuf_len(P.c.N) - 1);      // 8-byte mbarrier behind the staged vector
    double* const fbuf = zbuf + zbuf_len(P.c.N);
    QlRagClass* const rc = reinterpret_cast<QlRagClass*>(fbuf + QL_FBUF);       // RAGGED: the class being evaluated
    double* const jb = fbuf + QL_FBUF + QL_RAGCLASS_BYTES / 8;
    // RAGGED launches mix classes: the record of the current evaluation's class lives in shared memory and is swapped
    // when the class changes (the caller orders the problems by class, so that happens a handful of times per warp)
    const QlClass& c = RAGGED ? rc->c : P.c;
    int cur_cls = -1;
    QlSeg* const plan = reinterpret_cast<QlSeg*>(jb + 2 * QL_JBUF);
    const unsigned zaddr = smem_addr(zbuf);
    const unsigned jaddr = smem_addr(jb);
    int tmpl0 = -1, tmpl1 = -1;        // template currently held by staging buffer 0 / 1
    unsigned segctr = 0;               // segments this warp has streamed so far: consecutive segments alternate between
                                       // the two staging buffers ACROSS evaluations too, so the bulk store that may still
                                       // be reading a buffer (wait_group.read 1) is never the buffer being rewritten
    // cost coefficients: from shared memory ([41][N], copied once per CTA) when the launch has room for it, else
    // from the field-major global table (L2)
    Consts<FASTDIV> K;
    if (!RAGGED) { K.g = c.g; K.mb = c.mb; K.mf = c.mf; K.Ib = c.Ib; K.rmb = P.rmb; K.rmf = P.rmf; K.rIb = P.rIb; }
    const double* cost = P.cost;
    const double* x0_def = P.x0_def;
    const double* xf_def = P.xf_def;
    const int* seg_begin = P.seg_begin;
    int npad = P.npad;
    auto cls_of = [&](long long t) -> int {           // class of the t-th evaluation of a RAGGED launch
        const long long i = P.index ? __ldg(P.index + t) : t;
        return P.cls_of ? __ldg(P.cls_of + i) : 0;
    };
    auto n_of = [&](long long t) -> int { return RAGGED ? __ldg(&P.classes[cls_of(t)].c.n_nlp) : P.c.n_nlp; };

    const bool zbulk = P.zbulk != 0;      // ragged launches: only when the caller guarantees aligned, padded Z rows
    auto zrow_of = [&](long long t) -> const double* {
        if (RAGGED) return P.io.Z + __ldg(P.z_off + (P.index ? __ldg(P.index + t) : t));
        return P.io.Z + t * P.io.ldz;
    };
    unsigned zphase = 0;                 // parity of the mbarrier phase the next wait completes
    if (zbulk) {
        if (lane == 0) mbar_init(mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        __syncwarp();
    }
    // Work distribution: evaluations are handed out through a global ticket counter, in index order, to whichever
    // warp is free.  Besides balancing the load this keeps the rows being written at any moment within a narrow,
    // advancing address window, which the memory system likes much better than the drifting round-robin pattern of a
    // static assignment (+5 % full / +10 % g+J throughput at B=65,536, profiles/r01_ablation.md section 7).
    auto take_issue = [&]() -> unsigned {             // lane 0 draws the ticket; nothing waits for the atomic yet
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(P.ticket, 1u);
        return t;
    };
    auto take_get = [&](unsigned t) -> long long { return (long long)__shfl_sync(0xffffffffu, t, 0); };
    auto take = [&]() -> long long { return take_get(take_issue()); };
    // Programmatic dependent launch (the launcher sets the attribute on request): the next grid on the stream may be
    // scheduled into the SM slots this grid's warps give up while they drain; everything of it that touches data a
    // predecessor may have written - the work counter first of all - comes after griddepcontrol.wait, which returns
    // when every prerequisite grid has completed and flushed.  Without the attribute both instructions are no-ops.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (JM == JM_BLOCK && !RAGGED) {
        // the segment plan lives in shared memory: one 16-byte record per segment (a table of the handle, written once)
        const int4* src = reinterpret_cast<const int4*>(P.segs);
        int4* dst = reinterpret_cast<int4*>(plan);
        for (int i = lane; i < P.nseg; i += QL_LANES) dst[i] = __ldg(src + i);
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    long long b = take();
    long long nb = P.B;
    if (b < P.B) stage_z(zrow_of(b), zaddr, mbar, n_of(b), lane, zbulk);

    while (b < P.B) {
        if (zbulk) { mbar_wait(mbar, zphase); zphase ^= 1u; }
        else cp_async_wait_all();
        __syncwarp();
        double fsum = 0.0;
        // The kernels without the SPARSE_BLOCK stream are latency-bound: they draw the next ticket now, so that the
        // atomic's round trip is hidden behind this evaluation (the SPARSE_BLOCK kernel has no register to spare for it).
        // With a cost / gradient part the ticket is only DRAWN here and read after the first pass's cost section, when
        // the atomic has returned.  The short g-only evaluation reads it at once: reading it late made that launch
        // bimodal (265 or 349 M evals/s from one process to the next, profiles/r02_kernel_ab.md), at once it is steady.
        const bool late_ticket = JM != JM_BLOCK && (P.io.f || P.io.grad);
        unsigned tkt = 0;
        if (JM != JM_BLOCK) tkt = take_issue();
        if (JM != JM_BLOCK && !late_ticket) nb = take_get(tkt);
        const long long pi = (RAGGED && P.index) ? __ldg(P.index + b) : b;      // problem number (f, x0, xf, offsets)
        if (RAGGED) {
            const int cid = P.cls_of ? __ldg(P.cls_of + pi) : 0;
            if (cid != cur_cls) {
                // swap the class record (and, for SPARSE_BLOCK, the segment plan) in; the staging buffers' constant
                // images belong to the old class
                if (P.bulk && lane == 0) bulk_wait_read<0>();      // stores in flight still read the staging buffers
                __syncwarp();
                const int4* src = reinterpret_cast<const int4*>(P.classes + cid);
                int4* dst = reinterpret_cast<int4*>(rc);
                if (lane < QL_RAGCLASS_BYTES / 16) dst[lane] = __ldg(src + lane);
                __syncwarp();
                if (JM == JM_BLOCK) {
                    const int4* ps = reinterpret_cast<const int4*>(rc->segs);
                    int4* pd = reinterpret_cast<int4*>(plan);
                    for (int i = lane; i < rc->nseg; i += QL_LANES) pd[i] = __ldg(ps + i);
                    __syncwarp();
                }
                tmpl0 = tmpl1 = -1;
                cur_cls = cid;
            }
            K.g = c.g; K.mb = c.mb; K.mf = c.mf; K.Ib = c.Ib; K.rmb = rc->rmb; K.rmf = rc->rmf; K.rIb = rc->rIb;
            cost = rc->cost; x0_def = rc->x0_def; xf_def = rc->xf_def; seg_begin = rc->seg_begin; npad = rc->npad;
        }
        const bool first_is_y1 = (c.init_mode == 1);    // contact-first reads y1 (mode 1) or y2 (mode 2)
        double* const grow = P.io.g ? P.io.g + (RAGGED ? __ldg(P.g_off + pi) : b * P.io.ldg) : nullptr;
        double* const gradrow = P.io.grad ? P.io.grad + (RAGGED ? __ldg(P.z_off + pi) : b * P.io.ldgrad) : nullptr;
        double* const jrow = (WITH_JAC && JM != JM_PROD) ? P.io.jac + (RAGGED ? __ldg(P.j_off + pi) : b * P.io.ldjac) : nullptr;
        // TMA bulk stores need 16-byte aligned rows: a launch-wide property for strided batches, per row when ragged
        const bool bulk = P.bulk != 0 && (!RAGGED || (reinterpret_cast<uintptr_t>(jrow) & 15) == 0);

        if (grow) {
            // boundary rows (constraints.jl:149-150) straight from the staged vector, one lane per row
            const double* x0 = P.io.x0 ? P.io.x0 + pi * QL_NX : x0_def;
            const double* xf = P.io.xf ? P.io.xf + pi * QL_NX : xf_def;
            if (lane < QL_NX) QL_GST(grow + lane, __dsub_rn(zbuf[lane], __ldg(x0 + lane)));
            if (lane < QL_NX - 1) QL_GST(grow + c.c_term + lane, __dsub_rn(zbuf[(c.N - 1) * QL_NZK + lane], __ldg(xf + lane)));
            __syncwarp();
        }
        for (int p = 0; p < c.npass; ++p) {
            const int k = p * QL_LANES + lane + 1;          // 1-based knot of this lane
            const bool act = k <= c.N;
            const bool has_u = k < c.N;
            const bool jump = has_u && (k == c.k_trans - 1);   // constraints.jl:29 / :190
            double* const zk = zbuf + (k - 1) * QL_NZK;
            // costs.jl:9-15 accumulates J knot by knot: the 32 terms of the PREVIOUS pass are added here, in order,
            // where few registers are live (every lane adds up the same sequence; only lane 0's copy is stored)
            if (P.io.f && p > 0) fsum = f_chain(fsum, fbuf);

            // ---- 1. my knot's slice of Z: x_k, u_k, x_{k+1} = zk[0..34], fetched with 128-bit shared loads (the knot
            // stride of 160 B makes 64-bit loads 4-way bank conflicted; 16-byte loads halve the wavefronts)
            double zin[36];
            {
                const double2* zk2 = reinterpret_cast<const double2*>(zk);
#pragma unroll
                for (int i = 0; i < 18; ++i) {
                    const bool ld = (i < 8) ? act : has_u;      // knot N reads x_N only (zk[15] is the padding element)
                    const double2 v = ld ? zk2[i] : make_double2(0.0, 0.0);
                    zin[2 * i] = v.x;
                    zin[2 * i + 1] = v.y;
                }
                if (!has_u) zin[QL_NX] = 0.0;
            }
            const double* const xk = zin;
            const double* const uk = zin + QL_NX;
            const double* const xnx = zin + QL_NZK;
            __syncwarp();       // every lane holds its inputs: this pass's slice of zbuf may be overwritten

            // ---- 2. cost and gradient (costs.jl:6-34, quadratic_cost.jl:44-52); gradient in place over Z
            double lane_term = -0.0;                // lanes without a knot add -0.0: x + (-0.0) == x bit for bit
            if (act && (P.io.f || gradrow)) {
                const double* ct = cost + (k - 1);
                const int np = npad;
                double cq[QL_NCOST];                // all loads first: their latency overlaps
#pragma unroll
                for (int i = 0; i < QL_NCOST; ++i) cq[i] = __ldg(ct + i * np);
                const double hk = uk[4];
                double hq = __dmul_rn(__dmul_rn(0.5, __dmul_rn(xk[0], cq[0])), xk[0]);     // 0.5*x'Q*x, folded left
                double dq = __dmul_rn(cq[15], xk[0]);                                       // q'x
#pragma unroll
                for (int i = 1; i < QL_NX; ++i) {
                    hq = __dadd_rn(hq, __dmul_rn(__dmul_rn(0.5, __dmul_rn(xk[i], cq[i])), xk[i]));
                    dq = __dadd_rn(dq, __dmul_rn(cq[15 + i], xk[i]));
                }
                // my knot's slice of the gradient goes in place over my (dead) slice of the staged Z, as 16-byte stores
                double2* const zk2 = reinterpret_cast<double2*>(zk);
                double gz[QL_NZK];
#pragma unroll
                for (int i = 0; i < QL_NX; ++i) {
                    const double gq = __dadd_rn(__dmul_rn(cq[i], xk[i]), cq[15 + i]);       // Q*x + q
                    gz[i] = has_u ? __dmul_rn(hk, gq) : gq;
                    if ((i & 1) && gradrow) zk2[i >> 1] = make_double2(gz[i - 1], gz[i]);
                }
                double term;
                if (has_u) {
                    double hr = __dmul_rn(__dmul_rn(0.5, __dmul_rn(uk[0], cq[30])), uk[0]);
                    double dr = __dmul_rn(cq[35], uk[0]);
#pragma unroll
                    for (int i = 1; i < QL_NU; ++i) {
                        hr = __dadd_rn(hr, __dmul_rn(__dmul_rn(0.5, __dmul_rn(uk[i], cq[30 + i])), uk[i]));
                        dr = __dadd_rn(dr, __dmul_rn(cq[35 + i], uk[i]));
                    }
                    // quirk Q1 (costs.jl:30): the h entry gets h*(R55*h + r5), not d(h*stagecost)/dh
#pragma unroll
                    for (int i = 0; i < QL_NU; ++i)
                        gz[QL_NX + i] = __dmul_rn(hk, __dadd_rn(__dmul_rn(cq[30 + i], uk[i]), cq[35 + i]));
                    // ((((0.5x'Qx + q'x) + 0.5u'Ru) + r'u) + c) * h
                    const double sc = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(hq, dq), hr), dr), cq[40]);
                    term = __dmul_rn(hk, sc);
                } else {
                    term = __dadd_rn(__dadd_rn(hq, dq), cq[40]);       // termcost
#pragma unroll
                    for (int i = 0; i < QL_NU; ++i) gz[QL_NX + i] = 0.0;       // lands beyond n_nlp in the staging area
                }
                if (gradrow) {
#pragma unroll
                    for (int i = QL_NX / 2; i < QL_NZK / 2; ++i) zk2[i] = make_double2(gz[2 * i], gz[2 * i + 1]);
                }
                lane_term = term;
            }
            if (P.io.f) {
                __syncwarp();                       // the previous pass's terms have been read by every lane
                fbuf[lane] = lane_term;             // read back in the next pass, or after the last one (below)
            }
            if (late_ticket && p == 0) {
                nb = take_get(tkt);
#ifndef QL_NO_L2_PREFETCH
                // (measured: +13 % with the cost/gradient part in the evaluation, -17 % for the short g-only
                // evaluation, where the prefetch is still in flight when the load itself is issued;
                // profiles/r02_kernel_ab.md)
                if (zbulk && nb < P.B && lane == 0) prefetch_l2(zrow_of(nb), 8u * (unsigned)(n_of(nb) + 1));
#endif
            }

            // flush this pass's gradient slice with coalesced stores; the slice is then free for the defects
            double* const slice = zbuf + p * QL_LANES * QL_NZK;
            if (gradrow) {
                __syncwarp();
                const int e0 = p * QL_LANES * QL_NZK;
                const int cnt = min(QL_LANES * QL_NZK, c.n_nlp - e0);
                if ((reinterpret_cast<uintptr_t>(gradrow) & 15) == 0) {      // e0 is even: 16-byte stores
                    const double2* s2 = reinterpret_cast<const double2*>(slice);
                    double2* d2 = reinterpret_cast<double2*>(gradrow + e0);
                    // (one load, one store at a time on purpose: batching the loads ahead of the stores measured 8 % slower,
                    // profiles/r02_kernel_ab.md)
                    for (int i = lane; i < (cnt >> 1); i += QL_LANES) QL_GST(d2 + i, s2[i]);
                    if ((cnt & 1) && lane == 0) QL_GST(gradrow + e0 + cnt - 1, slice[cnt - 1]);
                } else {
                    for (int i = lane; i < cnt; i += QL_LANES) QL_GST(gradrow + e0 + i, slice[i]);
                }
                __syncwarp();
            }

            // ---- 3. constraints (constraints.jl:145-158) and the RK4 Jacobian values
            // the defects of this pass go to g[c_dyn + 15 (k_first - 1) ...]: stage them at the same parity as their
            // destination so that the flush can use 16-byte loads and stores
            double* const ddst = grow ? grow + c.c_dyn + p * QL_LANES * QL_NX : nullptr;
            const int dpar = (int)((reinterpret_cast<uintptr_t>(ddst) >> 3) & 1);
            double jv[WITH_JAC ? QL_NJ_MAX : 1];
            double jtheta = 0.0;
            if (has_u && (WITH_JAC || grow)) {
                double xn[QL_NX];
                if (WITH_JAC) {
                    if (k >= c.k_trans) ql_rk4_jac_mode3(xk, uk, K, xn, jv);
                    else if (c.init_mode == 1) ql_rk4_jac_mode1(xk, uk, K, xn, jv);
                    else ql_rk4_jac_mode2(xk, uk, K, xn, jv);
                } else {
                    if (k >= c.k_trans) ql_rk4_mode3(xk, uk, K, xn);
                    else if (c.init_mode == 1) ql_rk4_mode1(xk, uk, K, xn);
                    else ql_rk4_mode2(xk, uk, K, xn);
                }
                if (jump) {   // jump1_map / jump2_map, planar_quadruped.jl:250-260
                    xn[4] = 0.0; xn[6] = 0.0; xn[10] = 0.0; xn[11] = 0.0; xn[12] = 0.0; xn[13] = 0.0;
                }
                if (grow) {   // dynamics defect, constraints.jl:25-36: 15 consecutive rows per knot, staged in my slice
#pragma unroll
                    for (int i = 0; i < QL_NX; ++i) slice[dpar + lane * QL_NX + i] = __dsub_rn(xn[i], xnx[i]);
                }
            }
            if (act && (WITH_JAC || grow)) {
                double s, co;
                sincos(xk[2], &s, &co);
                // quirk Q4 (constraints.jl:269-273): branch on theta > 0
                jtheta = (xk[2] > 0) ? __dmul_rn(-c.half_lb, co) : __dmul_rn(c.half_lb, co);
                if (grow) {
                    QL_GST(grow + c.c_cfirst + (k - 1), first_is_y1 ? xk[4] : xk[6]);                                   // :58/:60
                    if (k >= c.k_trans) QL_GST(grow + c.c_cother + (k - c.k_trans), first_is_y1 ? xk[6] : xk[4]);      // :84/:86
                    QL_GST(grow + c.c_body + (k - 1), __dsub_rn(xk[1], __dmul_rn(c.half_lb, fabs(s))));                 // :109
                    if (k == c.N - 1) QL_GST(grow + c.c_fctrl, __dadd_rn(__dadd_rn(uk[1], uk[3]), c.mbg));       // :154
                }
            }

            // ---- 4. flush this pass's dynamics defects with coalesced stores
            __syncwarp();
            if (grow) {
                const int k_first = p * QL_LANES + 1;
                const int ndyn = min(QL_LANES, c.N - k_first) * QL_NX;      // knots of this pass with k < N
                // image element j <-> ddst[j - dpar]; the pairs (j, j+1) with j even are 16-byte aligned on both sides
                const int j0 = dpar, j1 = dpar + ndyn;
                const int a = (j0 + 1) & ~1, e = j1 & ~1;
                const double2* s2 = reinterpret_cast<const double2*>(slice);
                double2* d2 = reinterpret_cast<double2*>(ddst - dpar);
                for (int i = (a >> 1) + lane; i < (e >> 1); i += QL_LANES) QL_GST(d2 + i, s2[i]);
                if (lane == 0 && a > j0 && ndyn > 0) QL_GST(ddst, slice[j0]);
                if (lane == 1 && e < j1 && e >= a) QL_GST(ddst + (e - dpar), slice[e]);
                __syncwarp();
            }
            if (p == c.npass - 1) {
                // zbuf is dead: prefetch the next decision vector while the Jacobian values stream out
                if (JM == JM_BLOCK) nb = take();
                if (nb < P.B) stage_z(zrow_of(nb), zaddr, mbar, n_of(nb), lane, zbulk);
            }
            if constexpr (JM == JM_PROD) prod_pass<FASTDIV>(P, c, b, p, lane, k, xk, jv, jtheta, jb);

            // ---- 5'. SPARSE_TRUE: every lane writes its whole run; the pass leaves as two bulk stores of 16 knots
            // (a half-pass staging buffer keeps the shared memory per warp small enough for 8 warps per SM)
            if (JM == JM_TRUE || JM == JM_VALS) {
                auto run_off = [&](int kk) { return JM == JM_TRUE ? ql_true_run_off(c, kk) : ql_vals_run_off(c, kk); };
                for (int half = 0; half < 2; ++half) {
                    const int k_first = p * QL_LANES + 16 * half + 1;
                    if (k_first > c.N) break;
                    const int k_end = min(c.N, k_first + 15) + 1;
                    const int start = run_off(k_first);
                    const int end = (k_end > c.N) ? (JM == JM_TRUE ? c.nnz_true : c.nnz_vals) : run_off(k_end);
                    const int base = start & ~1;
                    if (P.bulk && lane == 0) bulk_wait_read<0>();     // the previous store has read the buffer
                    __syncwarp();
                    if (act && (lane >> 4) == half) {
                        const unsigned raddr = jaddr + 8u * (unsigned)(run_off(k) - base);
                        if (JM == JM_TRUE) ql_true_write_run(c, k, jv, jtheta, raddr);
                        else ql_vals_write_run(c, k, jv, jtheta, raddr);
                    }
                    if (bulk) {
                        fence_proxy_async();
                        __syncwarp();
                        const int a = (start + 1) & ~1, e = end & ~1;
                        if (lane == 0) {
                            if (e > a) bulk_store(jrow + a, jaddr + 8u * (unsigned)(a - base), 8u * (unsigned)(e - a));
                            bulk_commit();
                        }
                        if (lane == 1 && (start & 1)) jrow[start] = jb[start - base];
                        if (lane == 2 && (end & 1)) jrow[end - 1] = jb[end - 1 - base];
                    } else {
                        __syncwarp();
                        for (int i = lane; i < end - start; i += QL_LANES) jrow[start + i] = jb[start - base + i];
                        __syncwarp();
                    }
                }
            }

            // ---- 5. SPARSE_BLOCK: stream this pass's share of the Jacobian values
            if (JM == JM_BLOCK) {
                const int roff = act ? ql_run_off(c, k) : 0;
                const int e4 = ql_e4(c, k), e6 = ql_e6(c, k), fc = ql_fc(c, k);
                const int sb = __ldg(seg_begin + p), se = __ldg(seg_begin + p + 1);
                for (int s = sb; s < se; ++s) {
                    const int4 rec = *reinterpret_cast<const int4*>(plan + s);
                    const int start = rec.x, end = rec.y;
                    const int k0 = (int)(short)(rec.z & 0xffff), nk = (int)(signed char)((rec.z >> 16) & 0xff);
                    const int bi = ql_seg_buffer(segctr++), tm = (int)(short)(rec.w & 0xffff);
                    double* const buf = jb + bi * QL_JBUF;
                    const unsigned baddr = jaddr + (unsigned)bi * (QL_JBUF * 8u);
                    const int base = start & ~1;                 // image[0] <-> stream offset `base`
                    const bool mine = act && k >= k0 && k < k0 + nk;
                    const unsigned raddr = baddr + 8u * (unsigned)(roff - base);
                    unsigned pg[7];                              // run start + extras preceding each column group
                    pg[0] = raddr;
                    pg[1] = raddr + 8u;
                    pg[2] = raddr + 16u;
                    pg[3] = raddr + 8u * (2 + e4);
                    pg[4] = raddr + 8u * (2 + e4 + e6);
                    pg[5] = raddr + 8u * (2 + e4 + e6 + fc);
                    pg[6] = raddr + 8u * (2 + e4 + e6 + 2 * fc);

                    // the bulk store issued two segments ago read this buffer: wait until it is done
                    // (a ragged launch mixes bulk and plain rows: a plain row commits no groups, so it waits for all)
                    if (P.bulk && lane == 0) { if (bulk) bulk_wait_read<1>(); else bulk_wait_read<0>(); }
                    __syncwarp();

                    if ((bi ? tmpl1 : tmpl0) != tm) {            // different constant image: rebuild
                        for (int i = lane; i < QL_JBUF / 2; i += QL_LANES) st_shared_zero16(baddr + 16u * i);
                        __syncwarp();
                        {   // lanes 0-15 write the constants of knot k0, lanes 16-31 those of knot k0+1, one slot each
                            const int kk = k0 + (lane >> 4);
                            if ((lane >> 4) < nk)
                                ql_write_run_constants_slot(c, kk, buf + (ql_run_off(c, kk) - base), lane & 15);
                        }
                        if (mine && has_u) {     // constant entries of the RK4 block, by the knot's owner lane
                            if (k >= c.k_trans) ql_const_mode3(pg, jump);
                            else if (c.init_mode == 1) ql_const_mode1(pg, jump);
                            else ql_const_mode2(pg, jump);
                        }
                        if (bi) tmpl1 = tm; else tmpl0 = tm;
                    }
                    if (mine) {
                        if (has_u) {
                            if (k >= c.k_trans) ql_patch_mode3(jv, pg, jump);
                            else if (c.init_mode == 1) ql_patch_mode1(jv, pg, jump);
                            else ql_patch_mode2(jv, pg, jump);
                        }
                        st_shared_f64(raddr + 8u * (unsigned)ql_theta_pos(c, k), jtheta);   // constraints.jl:269-273
                    }
                    if (bulk) {
                        fence_proxy_async();
                        __syncwarp();
                        const int a = (start + 1) & ~1, e = end & ~1;      // 16 B aligned interior
                        if (lane == 0) {
                            if (e > a) bulk_store(jrow + a, baddr + 8u * (unsigned)(a - base), 8u * (unsigned)(e - a));
                            bulk_commit();
                        }
                        if (lane == 1 && (start & 1)) jrow[start] = buf[start - base];
                        if (lane == 2 && (end & 1)) jrow[end - 1] = buf[end - 1 - base];
                    } else {
                        __syncwarp();
                        for (int i = lane; i < end - start; i += QL_LANES) jrow[start + i] = buf[start - base + i];
                    }
                }
            }
        }

        // ---- 6. cost (accumulated in the reference's order above)
        if (P.io.f) {
            fsum = f_chain(fsum, fbuf);          // the last pass's terms
            if (lane == 0) QL_GST(P.io.f + pi, fsum);
        }
        b = nb;
    }
    if (WITH_JAC && P.bulk && lane == 0) bulk_wait_all();
    // the last CTA to leave re-arms the counters for the next launch on this stream
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(P.ticket + 1, 1u) == gridDim.x - 1) {
            P.ticket[0] = 0u;
            P.ticket[1] = 0u;
        }
    }
