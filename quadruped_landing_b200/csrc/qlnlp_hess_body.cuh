// qlnlp_hess_body.cuh -- the body of the Hessian kernel (qlnlp_hess.cuh), NOT a header: it is included inside
// hess_kernel and hess_prod_kernel, which define FASTDIV, PROD and the launch record P (one text, and the existing
// kernel reads its __grid_constant__ parameter directly, as in qlnlp_eval_body.cuh).
    extern __shared__ __align__(16) double smem[];
    const QlClass& c = P.c;
    const int lane = threadIdx.x;
    double* const zbuf = smem;
    const unsigned mbar = smem_addr(zbuf + zbuf_len(c.N) - 1);
    double* const hb = zbuf + zbuf_len(c.N);
    const unsigned zaddr = smem_addr(zbuf), haddr = smem_addr(hb);
    Consts<FASTDIV> K;
    K.g = c.g; K.mb = c.mb; K.mf = c.mf; K.Ib = c.Ib; K.rmb = P.rmb; K.rmf = P.rmf; K.rIb = P.rIb;
    const bool zbulk = P.zbulk != 0;
    unsigned zphase = 0;
    if (zbulk) {
        if (lane == 0) mbar_init(mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        __syncwarp();
    }
    // evaluations are handed out in index order through the stream's ticket counter, like in eval_kernel: the rows
    // being written at any moment stay within a narrow, advancing window
    auto take_issue = [&]() -> unsigned { return lane == 0 ? atomicAdd(P.ticket, 1u) : 0u; };
    auto take_get = [&](unsigned t) -> long long { return (long long)__shfl_sync(0xffffffffu, t, 0); };
    asm volatile("griddepcontrol.wait;" ::: "memory");      // (a predecessor launched with the dependent-launch attribute)
    long long b = take_get(take_issue());
    if (b < P.B) stage_z(P.Z + b * P.ldz, zaddr, mbar, c.n_nlp, lane, zbulk);
    while (b < P.B) {
        if (zbulk) { mbar_wait(mbar, zphase); zphase ^= 1u; }
        else cp_async_wait_all();
        __syncwarp();
        const unsigned tkt = take_issue();                 // the next ticket: drawn now, read after the first pass
        long long nb = P.B;
        const double sigma = P.sigma ? __ldg(P.sigma + b) : P.sigma0;
        const double* const lrow = P.lam + b * P.ldlam;
        double* const hrow = PROD ? nullptr : P.H + b * P.ldh;
        for (int p = 0; p < c.npass; ++p) {
            const int k = p * QL_LANES + lane + 1;
            const bool act = k <= c.N, has_u = k < c.N;
            const bool jump = has_u && (k == c.k_trans - 1);
            // this pass's share of the stream
            const int k_first = p * QL_LANES + 1, k_end = min(c.N, k_first + QL_LANES - 1) + 1;
            const int start = ql_hess_run_off(c, k_first);
            const int end = (k_end > c.N) ? ql_hess_nnz(c) : ql_hess_run_off(c, k_end);
            const int base = start & ~1;
            if (P.bulk && lane == 0) bulk_wait_read<0>();         // the previous pass's store has read the image
            __syncwarp();
            const double* vk = nullptr;
            if constexpr (PROD) vk = hprod_v<FASTDIV>(P, b) + (long long)QL_NZK * (k - 1);
            if (act) {
                const double* zk = zbuf + (k - 1) * QL_NZK;
                double x[QL_NX], u[QL_NU];
#pragma unroll
                for (int i = 0; i < QL_NX; ++i) x[i] = zk[i];
#pragma unroll
                for (int i = 0; i < QL_NU; ++i) u[i] = has_u ? zk[QL_NX + i] : 0.0;
                const unsigned raddr = haddr + 8u * (unsigned)(ql_hess_run_off(c, k) - base);
                // body-clearance row yb - lb/2 |sin(theta)|: second derivative of the branch constraints.jl:269-273 takes
                const double as = __dmul_rn(c.half_lb, sin(x[2]));
                const double tt = __dmul_rn(__ldg(lrow + c.c_body + (k - 1)), (x[2] > 0) ? as : -as);
                const double* ct = P.cost + (k - 1);
                const int np = P.npad;
                if (has_u) {
                    // (each lane loads its own 15 multipliers: staging the pass's 480 through shared memory with
                    // coalesced loads measured 8 % slower - the wait for them is then exposed at the top of the pass)
                    double lam[QL_NX];
#pragma unroll
                    for (int i = 0; i < QL_NX; ++i) lam[i] = __ldg(lrow + c.c_dyn + QL_NX * (k - 1) + i);
                    if (jump) {    // rows the jump map overwrites with constants (planar_quadruped.jl:250-260)
                        lam[4] = 0.0; lam[6] = 0.0; lam[10] = 0.0; lam[11] = 0.0; lam[12] = 0.0; lam[13] = 0.0;
                    }
                    double hv[QL_NH_MAX];
                    if (k >= c.k_trans) ql_rk4_hess_mode3(x, u, K, lam, hv);
                    else if (c.init_mode == 1) ql_rk4_hess_mode1(x, u, K, lam, hv);
                    else ql_rk4_hess_mode2(x, u, K, lam, hv);
                    // objective: f_k = h * stagecost_k(x, u)   (costs.jl:12, quadratic_cost.jl:44-47)
                    const double h = u[4];
                    double ox[QL_NX], ou[QL_NU - 1], hx[QL_NX], hu[QL_NU - 1];
#pragma unroll
                    for (int i = 0; i < QL_NX; ++i) {
                        const double Qi = __ldg(ct + i * np), qi = __ldg(ct + (15 + i) * np);
                        ox[i] = __dmul_rn(sigma, __dmul_rn(h, Qi));
                        hx[i] = __dmul_rn(sigma, __dadd_rn(__dmul_rn(Qi, x[i]), qi));
                    }
#pragma unroll
                    for (int i = 0; i < QL_NU - 1; ++i) {
                        const double Ri = __ldg(ct + (30 + i) * np), ri = __ldg(ct + (35 + i) * np);
                        ou[i] = __dmul_rn(sigma, __dmul_rn(h, Ri));
                        hu[i] = __dmul_rn(sigma, __dadd_rn(__dmul_rn(Ri, u[i]), ri));
                    }
                    const double R4 = __ldg(ct + 34 * np), r4 = __ldg(ct + 39 * np);
                    const double hh = __dmul_rn(sigma, __dadd_rn(__dmul_rn(2.0, __dadd_rn(__dmul_rn(R4, h), r4)), __dmul_rn(h, R4)));
                    if constexpr (PROD) {
                        double v[QL_NZK], o[QL_NZK];
#pragma unroll
                        for (int i = 0; i < QL_NZK; ++i) v[i] = __ldg(vk + i);
                        if (k >= c.k_trans) ql_hess_prod_mode3(hv, ox, ou, hx, hu, hh, tt, v, o);
                        else if (c.init_mode == 1) ql_hess_prod_mode1(hv, ox, ou, hx, hu, hh, tt, v, o);
                        else ql_hess_prod_mode2(hv, ox, ou, hx, hu, hh, tt, v, o);
                        double2* const hb2 = reinterpret_cast<double2*>(hb + lane * QL_NZK);
#pragma unroll
                        for (int i = 0; i < QL_NZK / 2; ++i) hb2[i] = make_double2(o[2 * i], o[2 * i + 1]);
                    } else {
                        if (k >= c.k_trans) ql_hess_store_mode3(hv, ox, ou, hx, hu, hh, tt, raddr);
                        else if (c.init_mode == 1) ql_hess_store_mode1(hv, ox, ou, hx, hu, hh, tt, raddr);
                        else ql_hess_store_mode2(hv, ox, ou, hx, hu, hh, tt, raddr);
                    }
                } else {
                    // knot N: termcost 0.5 x'Qx + q'x + c (quadratic_cost.jl:49-52) -> sigma * Q_ii on the diagonal
#pragma unroll
                    for (int i = 0; i < QL_NX; ++i) {
                        const double d = __dmul_rn(sigma, __ldg(ct + i * np));
                        const double hd = i == 2 ? __dadd_rn(d, tt) : d;
                        if constexpr (PROD) hb[lane * QL_NZK + i] = __dmul_rn(hd, __ldg(vk + i));
                        else st_shared_f64(raddr + 8u * i, hd);
                    }
                }
            }
            if constexpr (PROD) {
                __syncwarp();
                double* const hvrow = hprod_hv<FASTDIV>(P, b);
                const int e0 = p * QL_LANES * QL_NZK;
                const int cnt = min(QL_LANES * QL_NZK, c.n_nlp - e0);
                if ((reinterpret_cast<uintptr_t>(hvrow) & 15) == 0) {
                    const double2* s2 = reinterpret_cast<const double2*>(hb);
                    double2* d2 = reinterpret_cast<double2*>(hvrow + e0);
                    for (int i = lane; i < (cnt >> 1); i += QL_LANES) gst<true>(d2 + i, s2[i]);
                    if ((cnt & 1) && lane == 0) gst<true>(hvrow + e0 + cnt - 1, hb[cnt - 1]);
                } else {
                    for (int i = lane; i < cnt; i += QL_LANES) gst<true>(hvrow + e0 + i, hb[i]);
                }
                __syncwarp();
            } else if (P.bulk) {
                fence_proxy_async();
                __syncwarp();
                const int a = (start + 1) & ~1, e = end & ~1;
                if (lane == 0) {
                    if (e > a) bulk_store(hrow + a, haddr + 8u * (unsigned)(a - base), 8u * (unsigned)(e - a));
                    bulk_commit();
                }
                if (lane == 1 && (start & 1)) hrow[start] = hb[start - base];
                if (lane == 2 && (end & 1)) hrow[end - 1] = hb[end - 1 - base];
            } else {
                __syncwarp();
                for (int i = lane; i < end - start; i += QL_LANES) hrow[start + i] = hb[start - base + i];
                __syncwarp();
            }
            if (p == 0) {
                nb = take_get(tkt);
                // the next evaluation's decision vector and multipliers: ask L2 for them now
                if (nb < P.B && lane == 0) {
                    if (zbulk) prefetch_l2(P.Z + nb * P.ldz, 8u * (unsigned)(c.n_nlp + 1));
                    const double* ln = P.lam + nb * P.ldlam;
                    if ((reinterpret_cast<uintptr_t>(ln) & 15) == 0) prefetch_l2(ln, (8u * (unsigned)c.m_nlp) & ~15u);
                }
            }
        }
        __syncwarp();
        if (nb < P.B) stage_z(P.Z + nb * P.ldz, zaddr, mbar, c.n_nlp, lane, zbulk);
        b = nb;
    }
    if (P.bulk && lane == 0) bulk_wait_all();
    // the last CTA to leave re-arms the counters for the next launch on this stream
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(P.ticket + 1, 1u) == gridDim.x - 1) {
            P.ticket[0] = 0u;
            P.ticket[1] = 0u;
        }
    }
