// vega_b200.hpp — C++ host-side mirror of vega's operator API for the shuffle path, header-only,
// above the C ABI in vega_b200.h.  The reference is compiled Rust and its toolchain is absent from
// this image, so this is the compiled-language host layer: same names, argument meaning and error
// behaviour as the reference for the calls on the path —
//   Context::new / make_rdd / parallelize          src/context.rs:333-345,399-431
//   PairRdd::group_by_key / reduce_by_key / join   src/rdd/pair_rdd.rs:35-52,54-80,104-121
//   PairRdd::cogroup                               src/rdd/pair_rdd.rs:123-155
//   left / right / full outer joins                (absent from the reference; Spark semantics, std::optional sides)
//   Rdd::count_by_value / distinct / collect       src/rdd/rdd.rs:450-459,502-522,420-434
//   Rdd::intersection / subtract                   src/rdd/rdd.rs:838-946
// Rows are Vec<(K,V)> with K in {u64,i64,i32,u32} and V in {u64,i64,f64}; reduce_by_key takes a
// named Op (the reference's serde_closure cannot cross into CUDA).  Errors throw vega::Error
// (the reference returns Result<_> / panics).
#pragma once
#include <cstdint>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "vega_b200.h"

namespace vega {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error("vega_b200 error " + std::to_string(c) + ": " + m), code(c) {}
};

inline void check(int rc)
{
    if (rc != VB_OK) throw Error(rc, vb_last_error());
}

enum class Op { Sum = VB_AGG_SUM, Min = VB_AGG_MIN, Max = VB_AGG_MAX };

namespace detail {
template <typename T> struct dtype;
template <> struct dtype<uint64_t> { static constexpr int code = VB_U64; static constexpr uint32_t width = 8; };
template <> struct dtype<int64_t> { static constexpr int code = VB_I64; static constexpr uint32_t width = 8; };
template <> struct dtype<uint32_t> { static constexpr int code = VB_U64; static constexpr uint32_t width = 4; };
template <> struct dtype<int32_t> { static constexpr int code = VB_I64; static constexpr uint32_t width = 4; };
template <> struct dtype<double> { static constexpr int code = VB_F64; static constexpr uint32_t width = 8; };

template <typename T> inline uint64_t to_bits(T v)
{
    if constexpr (std::is_same<T, double>::value) { uint64_t b; __builtin_memcpy(&b, &v, 8); return b; }
    else if constexpr (std::is_signed<T>::value) return (uint64_t)(int64_t)v;
    else return (uint64_t)v;
}
template <typename T> inline T from_bits(uint64_t b)
{
    if constexpr (std::is_same<T, double>::value) { double d; __builtin_memcpy(&d, &b, 8); return d; }
    else return (T)b;
}

struct ShufDeleter { void operator()(vb_shuf *s) const { vb_shuffle_free(s); } };
using ShufPtr = std::unique_ptr<vb_shuf, ShufDeleter>;
}  // namespace detail

class Context : public std::enable_shared_from_this<Context> {
public:
    // `Context::new()` (src/context.rs:333): here it opens CUDA device `device`.
    static std::shared_ptr<Context> create(int device = 0)
    {
        std::shared_ptr<Context> c(new Context());
        check(vb_ctx_create(device, &c->ctx_));
        return c;
    }
    ~Context() { if (ctx_) vb_ctx_destroy(ctx_); }
    vb_ctx *raw() const { return ctx_; }
    uint64_t new_shuffle_id() { return next_id_++; }

    template <typename K, typename V> class PairRddT;
    template <typename K> class KeyRddT;

    template <typename K, typename V>
    PairRddT<K, V> make_rdd(const std::vector<std::pair<K, V>> &data, size_t num_slices);
    template <typename K, typename V>
    PairRddT<K, V> parallelize(const std::vector<std::pair<K, V>> &data, size_t num_slices) { return make_rdd(data, num_slices); }
    template <typename K> KeyRddT<K> parallelize(const std::vector<K> &data, size_t num_slices);

private:
    Context() = default;
    vb_ctx *ctx_ = nullptr;
    uint64_t next_id_ = 0;
};

namespace detail {
// Run one shuffle: slice like ParallelCollection::slice, one map task per slice, seal.
template <typename K>
inline ShufPtr run_shuffle(Context &sc, const std::vector<uint64_t> &keys, const std::vector<uint64_t> *vals, size_t num_slices,
                           size_t num_splits, int vcode, int agg)
{
    if (num_slices < 1) throw Error(VB_ERR_INVALID, "Number of slices should be greater than or equal to 1");
    const uint64_t n = keys.size();
    std::vector<uint64_t> starts(std::min<uint64_t>(n, num_slices) + 2);
    const uint64_t n_map = vb_slice(n, num_slices, starts.data());
    vb_shuf *raw = nullptr;
    check(vb_shuffle_create(sc.raw(), sc.new_shuffle_id(), (uint32_t)n_map, (uint32_t)num_splits, dtype<K>::code, vcode, agg,
                            VB_PART_HASH_METRO64, &raw));
    ShufPtr s(raw);
    if (dtype<K>::width == 4) check(vb_shuffle_set_key_width(raw, 4));
    for (uint64_t m = 0; m < n_map; ++m) {
        const uint64_t lo = starts[m], cnt = starts[m + 1] - lo;
        check(vb_shuffle_map_soa(raw, (uint32_t)m, cnt ? keys.data() + lo : nullptr, (vals && cnt) ? vals->data() + lo : nullptr, cnt, VB_HOST));
    }
    check(vb_shuffle_seal(raw));
    return s;
}
}  // namespace detail

template <typename K, typename V>
class Context::PairRddT {
public:
    PairRddT(std::shared_ptr<Context> sc, const std::vector<std::pair<K, V>> &data, size_t num_slices)
        : sc_(std::move(sc)), num_slices_(num_slices)
    {
        keys_.reserve(data.size());
        vals_.reserve(data.size());
        for (auto &kv : data) { keys_.push_back(detail::to_bits<K>(kv.first)); vals_.push_back(detail::to_bits<V>(kv.second)); }
    }
    size_t number_of_splits() const { return num_slices_; }

    // group_by_key(num_splits).collect()  →  Vec<(K, Vec<V>)>, values in input order
    std::vector<std::pair<K, std::vector<V>>> group_by_key(size_t num_splits) const
    {
        auto s = detail::run_shuffle<K>(*sc_, keys_, &vals_, num_slices_, num_splits, detail::dtype<V>::code, VB_AGG_GROUP);
        std::vector<std::pair<K, std::vector<V>>> out;
        for (uint32_t r = 0; r < num_splits; ++r) {
            uint64_t nk = 0, nv = 0;
            check(vb_shuffle_reduce_size(s.get(), r, &nk, &nv));
            std::vector<uint64_t> k(nk), o(nk + 1), v(nv);
            check(vb_shuffle_reduce(s.get(), r, k.data(), nullptr, o.data(), v.data(), VB_HOST));
            for (uint64_t i = 0; i < nk; ++i) {
                std::vector<V> vs;
                for (uint64_t j = o[i]; j < o[i + 1]; ++j) vs.push_back(detail::from_bits<V>(v[j]));
                out.emplace_back(detail::from_bits<K>(k[i]), std::move(vs));
            }
        }
        return out;
    }

    // reduce_by_key(op, num_splits).collect()  →  Vec<(K, V)>
    std::vector<std::pair<K, V>> reduce_by_key(Op op, size_t num_splits) const
    {
        auto s = detail::run_shuffle<K>(*sc_, keys_, &vals_, num_slices_, num_splits, detail::dtype<V>::code, (int)op);
        std::vector<std::pair<K, V>> out;
        for (uint32_t r = 0; r < num_splits; ++r) {
            uint64_t nk = 0, nv = 0;
            check(vb_shuffle_reduce_size(s.get(), r, &nk, &nv));
            std::vector<uint64_t> k(nk), c(nk);
            check(vb_shuffle_reduce(s.get(), r, k.data(), c.data(), nullptr, nullptr, VB_HOST));
            for (uint64_t i = 0; i < nk; ++i) out.emplace_back(detail::from_bits<K>(k[i]), detail::from_bits<V>(c[i]));
        }
        return out;
    }

    // self.join(other, num_splits).collect()  →  Vec<(K, (V, W))>, inner join
    template <typename W>
    std::vector<std::pair<K, std::pair<V, W>>> join(const PairRddT<K, W> &other, size_t num_splits) const
    {
        auto a = detail::run_shuffle<K>(*sc_, keys_, &vals_, num_slices_, num_splits, detail::dtype<V>::code, VB_AGG_COGROUP);
        auto b = detail::run_shuffle<K>(*sc_, other.keys_, &other.vals_, other.num_slices_, num_splits, detail::dtype<W>::code, VB_AGG_COGROUP);
        std::vector<std::pair<K, std::pair<V, W>>> out;
        for (uint32_t r = 0; r < num_splits; ++r) {
            uint64_t n = 0;
            check(vb_join_size(a.get(), b.get(), r, &n));
            std::vector<uint64_t> k(n), v(n), w(n);
            check(vb_join(a.get(), b.get(), r, k.data(), v.data(), w.data(), VB_HOST));
            for (uint64_t i = 0; i < n; ++i)
                out.emplace_back(detail::from_bits<K>(k[i]), std::make_pair(detail::from_bits<V>(v[i]), detail::from_bits<W>(w[i])));
        }
        return out;
    }

    // self.cogroup(other, num_splits).collect()  →  Vec<(K, (Vec<V>, Vec<W>))>; per partition the keys of self in its
    // order, then the keys only `other` has; an empty Vec on the side that lacks a key
    template <typename W>
    std::vector<std::pair<K, std::pair<std::vector<V>, std::vector<W>>>> cogroup(const PairRddT<K, W> &other, size_t num_splits) const
    {
        auto a = detail::run_shuffle<K>(*sc_, keys_, &vals_, num_slices_, num_splits, detail::dtype<V>::code, VB_AGG_COGROUP);
        auto b = detail::run_shuffle<K>(*sc_, other.keys_, &other.vals_, other.num_slices_, num_splits, detail::dtype<W>::code, VB_AGG_COGROUP);
        std::vector<std::pair<K, std::pair<std::vector<V>, std::vector<W>>>> out;
        for (uint32_t r = 0; r < num_splits; ++r) {
            uint64_t nk = 0, nv = 0, nw = 0;
            check(vb_cogroup_size(a.get(), b.get(), r, &nk, &nv, &nw));
            std::vector<uint64_t> k(nk), ov(nk + 1), v(nv), ow(nk + 1), w(nw);
            check(vb_cogroup(a.get(), b.get(), r, k.data(), ov.data(), v.data(), ow.data(), w.data(), VB_HOST));
            for (uint64_t i = 0; i < nk; ++i) {
                std::vector<V> vs;
                std::vector<W> ws;
                for (uint64_t j = ov[i]; j < ov[i + 1]; ++j) vs.push_back(detail::from_bits<V>(v[j]));
                for (uint64_t j = ow[i]; j < ow[i + 1]; ++j) ws.push_back(detail::from_bits<W>(w[j]));
                out.emplace_back(detail::from_bits<K>(k[i]), std::make_pair(std::move(vs), std::move(ws)));
            }
        }
        return out;
    }

    // Spark's outer joins (absent from the reference): Vec<(K, (Option<V>, Option<W>))>, rows of a key contiguous
    template <typename W>
    std::vector<std::pair<K, std::pair<std::optional<V>, std::optional<W>>>> left_outer_join(const PairRddT<K, W> &other, size_t num_splits) const
    {
        return outer_join(other, num_splits, VB_JOIN_LEFT_OUTER);
    }
    template <typename W>
    std::vector<std::pair<K, std::pair<std::optional<V>, std::optional<W>>>> right_outer_join(const PairRddT<K, W> &other, size_t num_splits) const
    {
        return outer_join(other, num_splits, VB_JOIN_RIGHT_OUTER);
    }
    template <typename W>
    std::vector<std::pair<K, std::pair<std::optional<V>, std::optional<W>>>> full_outer_join(const PairRddT<K, W> &other, size_t num_splits) const
    {
        return outer_join(other, num_splits, VB_JOIN_FULL_OUTER);
    }

    std::shared_ptr<Context> sc_;
    size_t num_slices_;
    std::vector<uint64_t> keys_, vals_;

private:
    template <typename W>
    std::vector<std::pair<K, std::pair<std::optional<V>, std::optional<W>>>> outer_join(const PairRddT<K, W> &other, size_t num_splits, int kind) const
    {
        auto a = detail::run_shuffle<K>(*sc_, keys_, &vals_, num_slices_, num_splits, detail::dtype<V>::code, VB_AGG_COGROUP);
        auto b = detail::run_shuffle<K>(*sc_, other.keys_, &other.vals_, other.num_slices_, num_splits, detail::dtype<W>::code, VB_AGG_COGROUP);
        std::vector<std::pair<K, std::pair<std::optional<V>, std::optional<W>>>> out;
        for (uint32_t r = 0; r < num_splits; ++r) {
            uint64_t n = 0;
            check(vb_join_outer_size(a.get(), b.get(), r, kind, &n));
            std::vector<uint64_t> k(n), v(n), w(n);
            std::vector<uint8_t> valid(n);
            check(vb_join_outer(a.get(), b.get(), r, kind, k.data(), v.data(), w.data(), valid.data(), VB_HOST));
            for (uint64_t i = 0; i < n; ++i) {
                std::optional<V> ov;
                std::optional<W> ow;
                if (valid[i] & VB_JOIN_HAS_V) ov = detail::from_bits<V>(v[i]);
                if (valid[i] & VB_JOIN_HAS_W) ow = detail::from_bits<W>(w[i]);
                out.emplace_back(detail::from_bits<K>(k[i]), std::make_pair(ov, ow));
            }
        }
        return out;
    }
};

template <typename K>
class Context::KeyRddT {
public:
    KeyRddT(std::shared_ptr<Context> sc, const std::vector<K> &data, size_t num_slices) : sc_(std::move(sc)), num_slices_(num_slices)
    {
        for (auto &k : data) keys_.push_back(detail::to_bits<K>(k));
    }
    // count_by_value().collect() → Vec<(K, u64)>   (src/rdd/rdd.rs:450-459)
    std::vector<std::pair<K, uint64_t>> count_by_value() const
    {
        std::vector<uint64_t> starts(std::min<uint64_t>(keys_.size(), num_slices_) + 2);
        const size_t n_splits = vb_slice(keys_.size(), num_slices_, starts.data());
        auto s = detail::run_shuffle<K>(*sc_, keys_, nullptr, num_slices_, n_splits, VB_U64, VB_AGG_COUNT);
        std::vector<std::pair<K, uint64_t>> out;
        for (uint32_t r = 0; r < n_splits; ++r) {
            uint64_t nk = 0, nv = 0;
            check(vb_shuffle_reduce_size(s.get(), r, &nk, &nv));
            std::vector<uint64_t> k(nk), c(nk);
            check(vb_shuffle_reduce(s.get(), r, k.data(), c.data(), nullptr, nullptr, VB_HOST));
            for (uint64_t i = 0; i < nk; ++i) out.emplace_back(detail::from_bits<K>(k[i]), c[i]);
        }
        return out;
    }
    // intersection(other[, num_splits]).collect() / subtract(other).collect()   (src/rdd/rdd.rs:838-946): the reference
    // cogroups (x, None) of both sides and reads the two Vec lengths; here ONE tagged SUM shuffle — side A rows carry 1,
    // side B rows 2^32 — so a key's sum says on which sides it occurred.  Each key once, like the reference.
    std::vector<K> intersection(const KeyRddT<K> &other, size_t num_splits = 0) const { return set_op(other, num_splits, true); }
    std::vector<K> subtract(const KeyRddT<K> &other, size_t num_splits = 0) const { return set_op(other, num_splits, false); }

    // distinct().collect()   (src/rdd/rdd.rs:502-522)
    std::vector<K> distinct() const
    {
        std::vector<K> out;
        for (auto &kv : count_by_value()) out.push_back(kv.first);
        return out;
    }

private:
    std::vector<K> set_op(const KeyRddT<K> &other, size_t num_splits, bool both) const
    {
        std::vector<uint64_t> sa(std::min<uint64_t>(keys_.size(), num_slices_) + 2), sb(std::min<uint64_t>(other.keys_.size(), other.num_slices_) + 2);
        const uint64_t na = vb_slice(keys_.size(), num_slices_, sa.data()), nb = vb_slice(other.keys_.size(), other.num_slices_, sb.data());
        if (num_splits == 0) num_splits = (size_t)na;                       // self.number_of_splits()
        vb_shuf *raw = nullptr;
        check(vb_shuffle_create(sc_->raw(), sc_->new_shuffle_id(), (uint32_t)(na + nb), (uint32_t)num_splits, detail::dtype<K>::code, VB_U64,
                                VB_AGG_SUM, VB_PART_HASH_METRO64, &raw));
        detail::ShufPtr s(raw);
        if (detail::dtype<K>::width == 4) check(vb_shuffle_set_key_width(raw, 4));
        const std::vector<uint64_t> ta(keys_.size(), 1ull), tb(other.keys_.size(), 1ull << 32);
        for (uint64_t m = 0; m < na; ++m)
            check(vb_shuffle_map_soa(raw, (uint32_t)m, keys_.data() + sa[m], ta.data() + sa[m], sa[m + 1] - sa[m], VB_HOST));
        for (uint64_t m = 0; m < nb; ++m)
            check(vb_shuffle_map_soa(raw, (uint32_t)(na + m), other.keys_.data() + sb[m], tb.data() + sb[m], sb[m + 1] - sb[m], VB_HOST));
        check(vb_shuffle_seal(raw));
        std::vector<K> out;
        for (uint32_t r = 0; r < num_splits; ++r) {
            uint64_t nk = 0, nv = 0;
            check(vb_shuffle_reduce_size(raw, r, &nk, &nv));
            std::vector<uint64_t> k(nk), c(nk);
            check(vb_shuffle_reduce(raw, r, k.data(), c.data(), nullptr, nullptr, VB_HOST));
            for (uint64_t i = 0; i < nk; ++i) {
                const bool in_a = (c[i] & 0xFFFFFFFFull) != 0, in_b = (c[i] >> 32) != 0;
                if (both ? (in_a && in_b) : (in_a && !in_b)) out.push_back(detail::from_bits<K>(k[i]));
            }
        }
        return out;
    }

    std::shared_ptr<Context> sc_;
    size_t num_slices_;
    std::vector<uint64_t> keys_;
};

template <typename K, typename V>
Context::PairRddT<K, V> Context::make_rdd(const std::vector<std::pair<K, V>> &data, size_t num_slices)
{
    return PairRddT<K, V>(shared_from_this(), data, num_slices);
}
template <typename K>
Context::KeyRddT<K> Context::parallelize(const std::vector<K> &data, size_t num_slices)
{
    return KeyRddT<K>(shared_from_this(), data, num_slices);
}

}  // namespace vega
