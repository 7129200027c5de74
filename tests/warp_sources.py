"""User densities written in the warp calling convention (UserModel(..., warp=True)), shared by the compile test, the
GPU tests and benchmarks/user_model_warp.py.  Hand-written sources define potential_and_grad(q, g, d, data, w);
autodiff sources define log_density(q, d, data, w)."""

# Neal's funnel, v = q[0] ~ N(0, 3), x_i ~ N(0, exp(v / 2)), constants dropped: coordinates split across lanes, every
# lane reuses v
FUNNEL_WARP = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    const S v = q[0];
    const S inv_var = exp(-v);
    S lp = (T)0;
    for (int i = 1 + w.lane; i < d; i += w.size) lp += (T)(-0.5) * square(q[i]) * inv_var - (T)0.5 * v;
    return w.sum(lp) + (T)(-0.5) * square(v) / (T)9;
}
"""

# the same funnel with a hand-written gradient, U = v^2 / 18 + sum 0.5 x^2 e^-v + 0.5 (d - 1) v
FUNNEL_WARP_HAND = r"""
template <typename T>
__device__ T potential_and_grad(const T* q, T* g, int d, const T* data, const Warp& w) {
    const T v = q[0], iv = exp(-v);
    T u = 0, s = 0;
    for (int i = 1 + w.lane; i < d; i += w.size) {
        const T x = q[i];
        u += (T)0.5 * x * x * iv;
        s += x * x;
        g[i] = x * iv;
    }
    u = w.sum(u);
    s = w.sum(s);
    if (w.lane == 0) g[0] = v / (T)9 + (T)0.5 * (T)(d - 1) - (T)0.5 * s * iv;
    return u + v * v / (T)18 + (T)0.5 * (T)(d - 1) * v;
}
"""

# the thread-per-chain counterpart of FUNNEL_WARP_HAND
FUNNEL_THREAD_HAND = r"""
template <typename T>
__device__ T potential_and_grad(const T* q, T* g, int d, const T* data) {
    const T v = q[0], iv = exp(-v);
    T u = 0, s = 0;
    for (int i = 1; i < d; ++i) {
        const T x = q[i];
        u += (T)0.5 * x * x * iv;
        s += x * x;
        g[i] = x * iv;
    }
    g[0] = v / (T)9 + (T)0.5 * (T)(d - 1) - (T)0.5 * s * iv;
    return u + v * v / (T)18 + (T)0.5 * (T)(d - 1) * v;
}
"""

# Bayesian logistic regression, data = [n, X (n x d, row-major), y (n)], standard normal prior: data rows split across
# lanes, so every lane reads every beta
LOGISTIC_WARP = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    const int n = (int)data[0];
    const T* X = data + 1;
    const T* y = X + n * d;
    S lp = (T)0;
    for (int j = w.lane; j < d; j += w.size) lp -= (T)0.5 * square(q[j]);
    for (int i = w.lane; i < n; i += w.size) {
        S s = (T)0;
        for (int j = 0; j < d; ++j) s += q[j] * X[i * d + j];
        lp -= softplus(s) - s * y[i];
    }
    return w.sum(lp);
}
"""

# -1/2 (q - mu)^T A (q - mu), data = [mu (d), A (d x d)]: rows split across lanes, every lane touches every input
QUAD_ROWS = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    const T* mu = data;
    const T* A = data + d;
    S lp = (T)0;
    for (int i = w.lane; i < d; i += w.size) {
        S t = (T)0;
        for (int j = 0; j < d; ++j) t += (q[j] - mu[j]) * A[i * d + j];
        lp -= (T)0.5 * ((q[i] - mu[i]) * t);
    }
    return w.sum(lp);
}
"""

# the same form with the coordinates split across lanes: one collective per row
QUAD_COLS = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    const T* mu = data;
    const T* A = data + d;
    S lp = (T)0;
    for (int i = 0; i < d; ++i) {
        S t = (T)0;
        for (int j = w.lane; j < d; j += w.size) t += (q[j] - mu[j]) * A[i * d + j];
        t = w.sum(t);
        if (i % w.size == w.lane) lp -= (T)0.5 * ((q[i] - mu[i]) * t);
    }
    return w.sum(lp);
}
"""

# x * x on one node: both operands of each product are the same input or the same node
SHARED_WARP = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    S lp = (T)0;
    for (int i = w.lane; i < d; i += w.size) {
        const S y = (T)3 * q[i] + (T)1;
        lp -= q[i] * q[i] + y * y;
    }
    return w.sum(lp);
}
"""

# multivariate Student-t, data = [nu]: the collective is used nonlinearly
STUDENT_T_WARP = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    const T nu = data[0];
    S s = (T)0;
    for (int i = w.lane; i < d; i += w.size) s += square(q[i]);
    return (T)(-0.5) * (nu + (T)d) * log1p(w.sum(s) / nu);
}
"""

# lanes with different operation counts between collectives: the number of terms depends on the chain's q[0] and is
# spread over the lanes, then a branch on each lane's own values
BRANCHY_WARP = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    const int n = (int)(fabs(q[0].v) * (T)4);
    S lp = (T)0;
    if (w.lane == 0) lp = (T)(-0.5) * square(q[0]);
    for (int k = 1 + w.lane; k <= n; k += w.size) {
        const int i = 1 + k % (d - 1);
        lp -= square(q[i] - (T)(0.1 * k)) * (T)(0.5 / k);
    }
    const S a = w.sum(lp);
    S b = (T)0;
    for (int i = w.lane; i < d; i += w.size)
        if (q[i].v > (T)0) b += (T)0.25 * square(q[i]);
    return a - w.sum(b);
}
"""

# independent Gaussians, data = [mu (d), 1 / sigma^2 (d)]
IID_WARP = r"""
template <typename S, typename T>
__device__ S log_density(const S* q, int d, const T* data, const Warp& w) {
    S lp = (T)0;
    for (int i = w.lane; i < d; i += w.size) lp -= (T)0.5 * square(q[i] - data[i]) * data[d + i];
    return w.sum(lp);
}
"""

AUTODIFF = {"funnel": FUNNEL_WARP, "logistic": LOGISTIC_WARP, "quad_rows": QUAD_ROWS, "quad_cols": QUAD_COLS,
            "shared": SHARED_WARP, "student_t": STUDENT_T_WARP, "branchy": BRANCHY_WARP, "iid": IID_WARP}
HAND = {"funnel_hand": FUNNEL_WARP_HAND}
