// openfhe_json.cpp -- import / export of OpenFHE 1.0.x binfhe objects in cereal JSON form (SURVEY.md 8 row f-3).
//
// The reference has no serialization calls of its own (no Serial:: in src/); what a maintainer would exchange are the files OpenFHE's
// own examples write with  Serial::SerializeToFile(path, obj, SerType::JSON)  (boolean-serial-json.cpp): the secret key
// (LWEPrivateKey), the refresh key (cc.GetRefreshKey(): RingGSWACCKey / "BSkey"), the switching key (cc.GetSwitchKey(): LWESwitchingKey /
// "KSkey") and ciphertexts (LWECiphertext).  Layout as recalled from openfhe-development v1.0.x (the library is NOT available in this
// environment, so the layout is unverified -- see INTEGRATION.md "Closing the parity gap"):
//
//   root                    {"value0": <object>}
//   shared_ptr<T>           {"ptr_wrapper": {"id": <u32>, "data": <T>}}            unique_ptr<T>  {"ptr_wrapper": {"valid": 1, "data": <T>}}
//   versioned class         first member "cereal_class_version": <u32>
//   NativeInteger           a JSON number (some versions: a decimal string, or {"v": n})
//   NativeVector            {"v": [ints...], "m": modulus}
//   NativePoly              {"v": unique_ptr<NativeVector>, "f": 0 (EVALUATION) | 1 (COEFFICIENT), "p": shared_ptr<ILParams>}
//   LWEPrivateKeyImpl       {"s": NativeVector}                                     (ternary key stored modulo the vector's modulus)
//   LWECiphertextImpl       {"a": NativeVector, "b": NativeInteger}
//   LWESwitchingKeyImpl     {"k": [N][baseKS][dKS] of LWECiphertextImpl}            (later 1.0.x: {"a": [..][..][..] vectors, "b": [..][..][..] ints})
//   RingGSWEvalKeyImpl      {"elements": [2 dG][2] of NativePoly}                   (EVALUATION format, psi = smallest primitive 2N-th root, CT order)
//   RingGSWACCKeyImpl       {"k": [d0][d1][d2] of shared_ptr<RingGSWEvalKeyImpl>}   GINX: [1][2][n] (+1 keys, then -1 keys); AP: [n][baseR][dR], j = 0 unused
//
// Because that layout cannot be checked here, the reader is STRUCTURAL rather than positional: it unwraps ptr_wrapper / value0 / single-
// member wrappers wherever they occur, accepts integers as numbers, strings or {"v": n}, and finds polynomials (objects with "v" and "f")
// and ciphertexts (objects with "a" and "b") in document order, checking only the counts and moduli.  The writer emits exactly the layout
// above.  Polynomials in EVALUATION format are converted with the engine's host NTT, which uses OpenFHE's convention (SURVEY C.6).
#include "../csrc/engine.hpp"
#include <cctype>
#include <cstdio>
#include <cstring>
#include <memory>

using namespace bfhe;

namespace {

// ---- minimal JSON DOM ----
struct JVal {
  enum Kind { NUL, NUM, STR, ARR, OBJ } kind = NUL;
  u64 num = 0;
  bool neg = false;
  std::string str;
  std::vector<JVal> arr;
  std::vector<u64> nums; // an array of plain non-negative integers is kept packed (a STD128_OPT refresh key holds 16.4 M of them)
  std::vector<std::pair<std::string, JVal>> obj;
  const JVal *get(const char *key) const {
    if (kind != OBJ) return nullptr;
    for (auto &kv : obj)
      if (kv.first == key) return &kv.second;
    return nullptr;
  }
};
struct JParser {
  const char *p, *end;
  std::string err;
  void ws() { while (p < end && std::isspace((unsigned char)*p)) p++; }
  bool fail(const char *m) { if (err.empty()) err = std::string(m) + " at offset " + std::to_string((size_t)(p - start)); return false; }
  const char *start;
  bool value(JVal &v, int depth = 0) {
    if (depth > 64) return fail("JSON nested too deeply");
    ws();
    if (p >= end) return fail("unexpected end of JSON");
    if (*p == '{') {
      v.kind = JVal::OBJ; p++; ws();
      if (p < end && *p == '}') { p++; return true; }
      for (;;) {
        ws();
        JVal k;
        if (p >= end || *p != '"' || !string(k.str)) return fail("expected a member name");
        ws();
        if (p >= end || *p != ':') return fail("expected ':'");
        p++;
        v.obj.emplace_back(std::move(k.str), JVal());
        if (!value(v.obj.back().second, depth + 1)) return false;
        ws();
        if (p < end && *p == ',') { p++; continue; }
        if (p < end && *p == '}') { p++; return true; }
        return fail("expected ',' or '}'");
      }
    }
    if (*p == '[') {
      v.kind = JVal::ARR; p++; ws();
      if (p < end && *p == ']') { p++; return true; }
      for (;;) {
        ws();
        if (v.arr.empty() && p < end && std::isdigit((unsigned char)*p)) { // packed fast path
          u64 x = 0;
          while (p < end && std::isdigit((unsigned char)*p)) x = x * 10 + (u64)(*p++ - '0');
          if (p < end && (*p == '.' || *p == 'e' || *p == 'E')) return fail("non-integer number");
          v.nums.push_back(x);
        } else {
          if (!v.nums.empty()) { // mixed array: fall back to the general form
            for (u64 x : v.nums) { v.arr.emplace_back(); v.arr.back().kind = JVal::NUM; v.arr.back().num = x; }
            v.nums.clear();
          }
          v.arr.emplace_back();
          if (!value(v.arr.back(), depth + 1)) return false;
        }
        ws();
        if (p < end && *p == ',') { p++; continue; }
        if (p < end && *p == ']') { p++; return true; }
        return fail("expected ',' or ']'");
      }
    }
    if (*p == '"') { v.kind = JVal::STR; return string(v.str); }
    if (*p == '-' || std::isdigit((unsigned char)*p)) {
      v.kind = JVal::NUM;
      if (*p == '-') { v.neg = true; p++; }
      u64 x = 0;
      if (p >= end || !std::isdigit((unsigned char)*p)) return fail("bad number");
      while (p < end && std::isdigit((unsigned char)*p)) x = x * 10 + (u64)(*p++ - '0');
      if (p < end && (*p == '.' || *p == 'e' || *p == 'E')) return fail("non-integer number");
      v.num = x;
      return true;
    }
    for (const char *lit : {"true", "false", "null"}) {
      const size_t n = std::strlen(lit);
      if ((size_t)(end - p) >= n && !std::strncmp(p, lit, n)) { p += n; v.kind = JVal::NUL; v.num = lit[0] == 't'; return true; }
    }
    return fail("unexpected character");
  }
  bool string(std::string &out) {
    p++; // opening quote
    while (p < end && *p != '"') {
      if (*p == '\\' && p + 1 < end) { out.push_back(p[1]); p += 2; }
      else out.push_back(*p++);
    }
    if (p >= end) return fail("unterminated string");
    p++;
    return true;
  }
};

// strip cereal's wrappers: {"value0": x}, {"ptr_wrapper": {.., "data": x}}, and any object whose only non-version member is an object / array
const JVal *unwrap(const JVal *v) {
  for (int guard = 0; v && v->kind == JVal::OBJ && guard < 16; guard++) {
    if (const JVal *w = v->get("ptr_wrapper")) { const JVal *d = w->get("data"); if (!d) return nullptr; v = d; continue; }
    if (const JVal *w = v->get("value0")) { if (v->obj.size() <= 2) { v = w; continue; } }
    break;
  }
  return v;
}
bool scalar(const JVal *v, u64 &out) { // number | "decimal string" | {"v": scalar} | {"value0": scalar}
  v = unwrap(v);
  if (!v) return false;
  if (v->kind == JVal::NUM) { if (v->neg) return false; out = v->num; return true; }
  if (v->kind == JVal::STR) {
    if (v->str.empty()) return false;
    u64 x = 0;
    for (char ch : v->str) { if (!std::isdigit((unsigned char)ch)) return false; x = x * 10 + (u64)(ch - '0'); }
    out = x;
    return true;
  }
  if (v->kind == JVal::OBJ) {
    if (const JVal *w = v->get("v")) return scalar(w, out);
    if (const JVal *w = v->get("m_value")) return scalar(w, out);
  }
  return false;
}
// NativeVector: {"v": [...], "m": modulus} (possibly through wrappers), or a bare array
bool vector_of(const JVal *v, std::vector<u64> &out, u64 *modulus) {
  v = unwrap(v);
  if (!v) return false;
  const JVal *a = v;
  if (v->kind == JVal::OBJ) {
    a = unwrap(v->get("v"));
    if (a && a->kind == JVal::OBJ) return vector_of(a, out, modulus); // unique_ptr<NativeVector> inside a polynomial
    if (modulus) { u64 m = 0; if (const JVal *mv = v->get("m")) { if (scalar(mv, m)) *modulus = m; } }
  }
  if (!a || a->kind != JVal::ARR) return false;
  if (!a->nums.empty()) { out = a->nums; return true; }
  out.resize(a->arr.size());
  for (size_t i = 0; i < a->arr.size(); i++)
    if (!scalar(&a->arr[i], out[i])) return false;
  return true;
}
bool is_poly(const JVal *v) { return v && v->kind == JVal::OBJ && v->get("v") && v->get("f"); }
bool is_ct(const JVal *v) { return v && v->kind == JVal::OBJ && v->get("a") && v->get("b"); }
template <class Pred> void collect(const JVal *v, Pred pred, std::vector<const JVal *> &out) { // document order
  if (!v) return;
  if (pred(v)) { out.push_back(v); return; }
  if (v->kind == JVal::ARR) for (auto &e : v->arr) collect(&e, pred, out);
  if (v->kind == JVal::OBJ) for (auto &kv : v->obj) collect(&kv.second, pred, out);
}

bool flatten_ints(const JVal *v, std::vector<u64> &out) { // nested arrays of integers, document order
  v = unwrap(v);
  if (!v) return false;
  if (v->kind == JVal::ARR) {
    out.insert(out.end(), v->nums.begin(), v->nums.end());
    for (auto &e : v->arr) if (!flatten_ints(&e, out)) return false;
    return true;
  }
  u64 t;
  if (!scalar(v, t)) return false;
  out.push_back(t);
  return true;
}

int read_file(const char *path, std::string &buf) {
  FILE *f = std::fopen(path, "rb");
  if (!f) { set_error(std::string("cannot open ") + path); return BFHE_ERR_IO; }
  std::fseek(f, 0, SEEK_END);
  const long sz = std::ftell(f);
  std::fseek(f, 0, SEEK_SET);
  buf.resize((size_t)std::max(0L, sz));
  const size_t r = std::fread(&buf[0], 1, buf.size(), f);
  std::fclose(f);
  if (r != buf.size()) { set_error("short read"); return BFHE_ERR_IO; }
  return BFHE_OK;
}
int parse_file(const char *path, std::unique_ptr<JVal> &root) {
  std::string buf;
  if (int rc = read_file(path, buf)) return rc;
  root.reset(new JVal());
  JParser jp{buf.data(), buf.data() + buf.size(), "", buf.data()};
  if (!jp.value(*root)) { set_error("OpenFHE JSON: " + jp.err); return BFHE_ERR_FORMAT; }
  return BFHE_OK;
}
int fmt_err(const std::string &m) { set_error("OpenFHE JSON: " + m); return BFHE_ERR_FORMAT; }

// ---- writer helpers ----
struct Out {
  FILE *f;
  void s(const char *t) { std::fputs(t, f); }
  void n(u64 v) { std::fprintf(f, "%llu", (unsigned long long)v); }
  void vec(const u64 *v, size_t cnt, u64 mod) {
    s("{\"cereal_class_version\":1,\"v\":[");
    for (size_t i = 0; i < cnt; i++) { if (i) s(","); n(v[i]); }
    s("],\"m\":"); n(mod); s("}");
  }
};
u32 g_ptr_id = 0x80000001u; // cereal numbers first occurrences of shared pointers 1, 2, ... with the top bit set

} // namespace

extern "C" int bfhe_import_openfhe_json(bfhe_ctx *c, int what, const char *path) {
  if (!c || !path) return BFHE_ERR_ARG;
  std::unique_ptr<JVal> root;
  if (int rc = parse_file(path, root)) return rc;
  const bfhe_params &p = c->p;
  if (what == BFHE_OFHE_SECRET_KEY) {
    const JVal *o = unwrap(root.get());
    const JVal *sv = o && o->kind == JVal::OBJ ? o->get("s") : nullptr;
    std::vector<u64> s;
    u64 mod = 0;
    if (!sv || !vector_of(sv, s, &mod)) return fmt_err("LWEPrivateKey: member \"s\" (NativeVector) not found");
    if (s.size() != p.n) return fmt_err("LWEPrivateKey: dimension " + std::to_string(s.size()) + ", this context has n = " + std::to_string(p.n));
    if (mod == 0) mod = p.qKS;
    c->sk.resize(p.n);
    for (u32 i = 0; i < p.n; i++) {
      if (s[i] == 0) c->sk[i] = 0;
      else if (s[i] == 1) c->sk[i] = 1;
      else if (s[i] == mod - 1) c->sk[i] = -1;
      else return fmt_err("LWEPrivateKey: coefficient " + std::to_string(i) + " is not ternary");
    }
    c->has_sk = true;
    return BFHE_OK;
  }
  if (what == BFHE_OFHE_REFRESH_KEY) {
    std::vector<const JVal *> polys;
    collect(root.get(), is_poly, polys);
    const u32 N = p.N, rows = 2 * p.dG;
    const size_t per_key = (size_t)rows * 2;
    if (polys.empty() || polys.size() % per_key) return fmt_err("refresh key: " + std::to_string(polys.size()) + " polynomials, not a multiple of 2 dG x 2");
    const size_t nkeys = polys.size() / per_key;
    const size_t want = p.method == BFHE_GINX ? (size_t)2 * p.n : (size_t)p.n * (p.baseR - 1) * p.dR;
    if (nkeys != want) return fmt_err("refresh key: " + std::to_string(nkeys) + " RGSW ciphertexts, expected " + std::to_string(want));
    forget_mask_seed(c);
    c->bk_coef.assign(c->bk_words, 0);
    std::vector<u64> v;
    std::vector<u32> tmp(N);
    for (size_t kk = 0; kk < nkeys; kk++) {
      // document order -> internal order.  GINX: file [0][sign][i], internal [i][sign].  AP: file [i][j = 1..baseR-1][k] (the unused j = 0
      // slot is a null pointer and contributes no polynomial), internal [i][j - 1][k]: the same order.
      size_t dst = kk;
      if (p.method == BFHE_GINX) { const size_t sign = kk / p.n, i = kk % p.n; dst = i * 2 + sign; }
      for (size_t e = 0; e < per_key; e++) {
        const JVal *po = polys[kk * per_key + e];
        u64 mod = 0, fmt = 0;
        if (!vector_of(po, v, &mod) || v.size() != N) return fmt_err("refresh key: polynomial " + std::to_string(kk * per_key + e) + " is not a vector of N values");
        if (mod && mod != p.Q) return fmt_err("refresh key: ring modulus " + std::to_string(mod) + " in the file, this context uses Q = " + std::to_string(p.Q) +
                                              " (the kernels need 32 Q < 2^32 and are built for that prime; see DESIGN.md section 3)");
        scalar(po->get("f"), fmt);
        for (u32 j = 0; j < N; j++) { if (v[j] >= p.Q) return fmt_err("refresh key: coefficient out of range"); tmp[j] = (u32)v[j]; }
        if (fmt == 0) c->hntt.inv(tmp.data()); // EVALUATION -> coefficients (CT bit-reversed order, smallest psi: HostNtt's convention)
        std::memcpy(c->bk_coef.data() + (dst * per_key + e) * N, tmp.data(), (size_t)N * 4);
      }
    }
    c->ofhe_have_bk = true;
  } else if (what == BFHE_OFHE_SWITCH_KEY) {
    std::vector<const JVal *> cts;
    collect(root.get(), is_ct, cts);
    const size_t want = (size_t)p.N * p.baseKS * p.dKS;
    forget_mask_seed(c);
    c->ksk.assign(c->ksk_elems * c->ksk_elem_bytes, 0);
    auto put = [&](size_t idx, u64 val) {
      if (c->ksk_elem_bytes == 2) reinterpret_cast<u16 *>(c->ksk.data())[idx] = (u16)val;
      else reinterpret_cast<u32 *>(c->ksk.data())[idx] = (u32)val;
    };
    std::vector<u64> a;
    if (cts.size() == want) { // [N][baseKS][dKS] of LWECiphertextImpl: the internal order
      for (size_t e = 0; e < want; e++) {
        u64 mod = 0, b = 0;
        if (!vector_of(cts[e]->get("a"), a, &mod) || a.size() != p.n || !scalar(cts[e]->get("b"), b)) return fmt_err("switching key: entry " + std::to_string(e) + " is not an LWE ciphertext of dimension n");
        if (mod && mod != p.qKS) return fmt_err("switching key: modulus " + std::to_string(mod) + ", expected qKS = " + std::to_string(p.qKS));
        for (u32 t = 0; t < p.n; t++) put(e * (p.n + 1) + t, a[t]);
        put(e * (p.n + 1) + p.n, b);
      }
    } else if (cts.size() == 1) { // later 1.0.x: {"a": [N][baseKS][dKS] vectors, "b": [N][baseKS][dKS] integers}
      std::vector<const JVal *> vecs;
      std::vector<u64> ints;
      collect(cts[0]->get("a"), [](const JVal *v) { const JVal *u = unwrap(v); return u && u->kind == JVal::OBJ && u->get("v") != nullptr; }, vecs);
      if (!flatten_ints(cts[0]->get("b"), ints)) return fmt_err("switching key: member \"b\" is not an array of integers");
      if (vecs.size() != want || ints.size() != want) return fmt_err("switching key: " + std::to_string(vecs.size()) + " vectors / " + std::to_string(ints.size()) + " integers, expected " + std::to_string(want));
      for (size_t e = 0; e < want; e++) {
        const u64 b = ints[e];
        if (!vector_of(vecs[e], a, nullptr) || a.size() != p.n) return fmt_err("switching key: bad entry " + std::to_string(e));
        for (u32 t = 0; t < p.n; t++) put(e * (p.n + 1) + t, a[t]);
        put(e * (p.n + 1) + p.n, b);
      }
    } else {
      return fmt_err("switching key: " + std::to_string(cts.size()) + " LWE ciphertexts, expected N x baseKS x dKS = " + std::to_string(want));
    }
    c->ofhe_have_ksk = true;
  } else {
    return BFHE_ERR_ARG;
  }
  if (c->ofhe_have_bk && c->ofhe_have_ksk) { // both halves of the bootstrapping key are in: same state as after bfhe_btkeygen
    c->has_bt = true;
    c->dev_keys = false;
    c->form_cost_measured = false;
    if (c->device >= 0) return ensure_device_keys(c);
  }
  return BFHE_OK;
}

extern "C" int bfhe_export_openfhe_json(const bfhe_ctx *c, int what, const char *path) {
  if (!c || !path) return BFHE_ERR_ARG;
  const bfhe_params &p = c->p;
  if (what == BFHE_OFHE_SECRET_KEY ? !c->has_sk : !c->has_bt) { set_error("no such key in this context"); return BFHE_ERR_STATE; }
  FILE *f = std::fopen(path, "w");
  if (!f) { set_error(std::string("cannot open ") + path); return BFHE_ERR_IO; }
  Out o{f};
  o.s("{\"value0\":{\"ptr_wrapper\":{\"id\":"); o.n(g_ptr_id); o.s(",\"data\":{\"cereal_class_version\":1,");
  std::vector<u64> v;
  if (what == BFHE_OFHE_SECRET_KEY) {
    v.resize(p.n);
    for (u32 i = 0; i < p.n; i++) v[i] = c->sk[i] < 0 ? p.qKS - 1 : (u64)c->sk[i];
    o.s("\"s\":"); o.vec(v.data(), v.size(), p.qKS);
  } else if (what == BFHE_OFHE_REFRESH_KEY) {
    const u32 N = p.N, rows = 2 * p.dG;
    const size_t per_key = (size_t)rows * 2;
    std::vector<u32> tmp(N), bk(c->bk_words);
    host_full_bk(c, bk.data());
    v.resize(N);
    u32 id = 2;
    auto rgsw = [&](size_t src) { // shared_ptr<RingGSWEvalKeyImpl>
      o.s("{\"ptr_wrapper\":{\"id\":"); o.n(0x80000000u | id++); o.s(",\"data\":{\"cereal_class_version\":1,\"elements\":[");
      for (u32 r = 0; r < rows; r++) {
        o.s(r ? ",[" : "[");
        for (u32 cc = 0; cc < 2; cc++) {
          std::memcpy(tmp.data(), bk.data() + (src * per_key + (size_t)r * 2 + cc) * N, (size_t)N * 4);
          c->hntt.fwd(tmp.data()); // EVALUATION format, as BTKeyGen leaves it
          for (u32 j = 0; j < N; j++) v[j] = tmp[j];
          if (cc) o.s(",");
          o.s("{\"cereal_class_version\":1,\"v\":{\"ptr_wrapper\":{\"valid\":1,\"data\":"); o.vec(v.data(), N, p.Q);
          o.s("}},\"f\":0,\"p\":{\"ptr_wrapper\":{\"id\":1}}}"); // ILParams: first occurrence carries the ring parameters, later ones only the id
        }
        o.s("]");
      }
      o.s("]}}}");
    };
    o.s("\"k\":[");
    if (p.method == BFHE_GINX) {
      o.s("[");
      for (u32 sign = 0; sign < 2; sign++) {
        o.s(sign ? ",[" : "[");
        for (u32 i = 0; i < p.n; i++) { if (i) o.s(","); rgsw((size_t)i * 2 + sign); }
        o.s("]");
      }
      o.s("]");
    } else {
      for (u32 i = 0; i < p.n; i++) {
        o.s(i ? ",[" : "[");
        for (u32 j = 0; j < p.baseR; j++) {
          o.s(j ? ",[" : "[");
          for (u32 k = 0; k < p.dR; k++) {
            if (k) o.s(",");
            if (j == 0) o.s("{\"ptr_wrapper\":{\"id\":0}}"); // unused slot: null pointer
            else rgsw(((size_t)i * (p.baseR - 1) + (j - 1)) * p.dR + k);
          }
          o.s("]");
        }
        o.s("]");
      }
    }
    o.s("]");
  } else if (what == BFHE_OFHE_SWITCH_KEY) {
    std::vector<u8> ksk(c->ksk_elems * c->ksk_elem_bytes);
    host_full_ksk(c, ksk.data());
    auto get = [&](size_t idx) -> u64 {
      return c->ksk_elem_bytes == 2 ? reinterpret_cast<const u16 *>(ksk.data())[idx] : reinterpret_cast<const u32 *>(ksk.data())[idx];
    };
    v.resize(p.n);
    o.s("\"k\":[");
    for (u32 i = 0; i < p.N; i++) {
      o.s(i ? ",[" : "[");
      for (u32 j = 0; j < p.baseKS; j++) {
        o.s(j ? ",[" : "[");
        for (u32 k = 0; k < p.dKS; k++) {
          const size_t e = ((size_t)i * p.baseKS + j) * p.dKS + k;
          for (u32 t = 0; t < p.n; t++) v[t] = get(e * (p.n + 1) + t);
          if (k) o.s(",");
          o.s("{\"cereal_class_version\":1,\"a\":"); o.vec(v.data(), p.n, p.qKS); o.s(",\"b\":"); o.n(get(e * (p.n + 1) + p.n)); o.s("}");
        }
        o.s("]");
      }
      o.s("]");
    }
    o.s("]");
  } else {
    std::fclose(f);
    return BFHE_ERR_ARG;
  }
  o.s("}}}}\n");
  const bool bad = std::ferror(f) != 0;
  std::fclose(f);
  if (bad) { set_error("write error"); return BFHE_ERR_IO; }
  return BFHE_OK;
}

extern "C" int bfhe_import_openfhe_ct_json(const bfhe_ctx *c, const char *path, uint32_t *ct_row) {
  if (!c || !path || !ct_row) return BFHE_ERR_ARG;
  std::unique_ptr<JVal> root;
  if (int rc = parse_file(path, root)) return rc;
  std::vector<const JVal *> cts;
  collect(root.get(), is_ct, cts);
  if (cts.size() != 1) return fmt_err("expected one LWECiphertext, found " + std::to_string(cts.size()));
  std::vector<u64> a;
  u64 mod = 0, b = 0;
  if (!vector_of(cts[0]->get("a"), a, &mod) || a.size() != c->p.n || !scalar(cts[0]->get("b"), b)) return fmt_err("LWECiphertext: need \"a\" of dimension n and \"b\"");
  if (mod && mod != c->p.q) return fmt_err("LWECiphertext: modulus " + std::to_string(mod) + ", this context has q = " + std::to_string(c->p.q));
  for (u32 i = 0; i < c->p.n; i++) { if (a[i] >= c->p.q) return fmt_err("LWECiphertext: coefficient out of range"); ct_row[i] = (u32)a[i]; }
  if (b >= c->p.q) return fmt_err("LWECiphertext: b out of range");
  ct_row[c->p.n] = (u32)b;
  for (u32 i = c->p.n + 1; i < c->p.ct_stride; i++) ct_row[i] = 0;
  return BFHE_OK;
}
extern "C" int bfhe_export_openfhe_ct_json(const bfhe_ctx *c, const uint32_t *ct_row, const char *path) {
  if (!c || !path || !ct_row) return BFHE_ERR_ARG;
  FILE *f = std::fopen(path, "w");
  if (!f) { set_error(std::string("cannot open ") + path); return BFHE_ERR_IO; }
  Out o{f};
  std::vector<u64> v(c->p.n);
  for (u32 i = 0; i < c->p.n; i++) v[i] = ct_row[i];
  o.s("{\"value0\":{\"ptr_wrapper\":{\"id\":"); o.n(g_ptr_id); o.s(",\"data\":{\"cereal_class_version\":1,\"a\":");
  o.vec(v.data(), v.size(), c->p.q);
  o.s(",\"b\":"); o.n(ct_row[c->p.n]); o.s("}}}}\n");
  std::fclose(f);
  return BFHE_OK;
}
